#include "textio.h"

#include <cinttypes>
#include <cmath>
#include <cstring>

namespace ibdhost {

bool ends_with_gz(const std::string &fn) {
    return fn.size() >= 3 && fn.compare(fn.size() - 3, 3, ".gz") == 0;
}

std::string tract_header(bool summary, bool posterior) {
    std::string h = summary ? "Summary\t" : "";
    h += "Tract\tInferred_State\tFirst_Segment\tLast_Segment\tSTART\tEND\tN_Segments\tNUM_SITES\tLOD10";
    h += posterior ? "\tP_Mean\tP_Min\n" : "\n";
    return h;
}

// LOD10: log10 of the likelihood ratio of the called state against the better of the other two over the tract; it
// is negative where the penalties, not the likelihoods, decided the call
std::string tract_row(const hiddengem_tract &r, int64_t k, uint64_t start, uint64_t end, int64_t n_sites, bool posterior) {
    const int s = r.state;
    const double lod = (r.loglik[s] - std::fmax(r.loglik[(s + 1) % 3], r.loglik[(s + 2) % 3])) / std::log(10.0);
    char row[320];
    int n = snprintf(row, sizeof row, "%" PRId64 "\t%d\t%" PRId64 "\t%" PRId64 "\t%" PRIu64 "\t%" PRIu64 "\t%" PRId64 "\t%" PRId64 "\t%.4f", k + 1, s,
                     r.first_bin + 1, r.first_bin + r.n_bins, start, end, r.n_bins, n_sites, lod);
    if (posterior) n += snprintf(row + n, sizeof row - (size_t)n, "\t%.6f\t%.6f", r.post_mean, r.post_min);
    row[n++] = '\n';
    return std::string(row, (size_t)n);
}

bool LineReader::open(const std::string &path) {
    close();
    path_ = path;
    if (!ends_with_gz(path)) {
        // same diagnostics as fileOpen() for a plain file that cannot be opened
        FILE *f = fopen(path.c_str(), "r");
        if (!f) {
            fprintf(stderr, "Failed to open %s.\n", path.c_str());
            perror("Error");
            return false;
        }
        fclose(f);
    }
    gz_ = gzopen(path.c_str(), "r");
    if (!gz_) return false;
    gzbuffer(gz_, 1 << 20);
    buf_.resize(1 << 22);
    beg_ = end_ = 0;
    eof_ = false;
    return true;
}

void LineReader::close() {
    if (gz_) gzclose(gz_);
    gz_ = nullptr;
}

bool LineReader::fill() {
    if (eof_) return false;
    if (beg_ > 0) {
        memmove(buf_.data(), buf_.data() + beg_, end_ - beg_);
        end_ -= beg_;
        beg_ = 0;
    }
    if (end_ == buf_.size()) buf_.resize(buf_.size() * 2);
    const int n = gzread(gz_, buf_.data() + end_, (unsigned)std::min<size_t>(buf_.size() - end_, 1u << 30));
    if (n <= 0) {
        eof_ = true;
        return false;
    }
    end_ += (size_t)n;
    return true;
}

bool LineReader::next(const char **line, size_t *len) {
    size_t scan = beg_;
    for (;;) {
        const char *nl = (const char *)memchr(buf_.data() + scan, '\n', end_ - scan);
        if (nl) {
            *line = buf_.data() + beg_;
            *len = (size_t)(nl - (buf_.data() + beg_)) + 1;
            beg_ += *len;
            return true;
        }
        scan = end_ - beg_;  // offset relative to beg_, which fill() moves to 0
        if (!fill()) {
            if (end_ > beg_) {  // last line without a newline
                *line = buf_.data() + beg_;
                *len = end_ - beg_;
                beg_ = end_;
                return true;
            }
            return false;
        }
        scan += beg_;
    }
}

// sqrt of a variance; one a rounding below 0 is 0, NaN stays NaN
static double sd_of(double v) { return v > 0 ? std::sqrt(v) : (v == v ? 0.0 : v); }

std::string share_sd_lines(const double *expected, const double *cov, double n) {
    std::string out;
    char row[160];
    for (int k = 0; k < 3; k++) {
        const double sd = sd_of(cov[k * 4]);
        out.append(row, (size_t)snprintf(row, sizeof row, "#%% posterior IBD%d sd (n = %.2f): %.2f\n", k, sd, (sd / n) * 100));
    }
    const double phi = (expected[1] / 4 + expected[2] / 2) / n;
    const double var = (cov[4] / 16 + cov[8] / 4 + cov[5] / 4) / (n * n);
    out.append(row, (size_t)snprintf(row, sizeof row, "#%% posterior kinship (sd = %.4f): %.4f\n", sd_of(var), phi));
    return out;
}

}  // namespace ibdhost
