// textio.h — line reader for plain and gzip text (replaces File_Src / get_line_FS,
// src/file-io.c:20-75 of the reference).  Unlike the reference there is no 30,720-byte line cap
// (src/file-io.h:10), so panels with more than 7,679 individuals are read whole.
#pragma once

#include <zlib.h>

#include <cstdio>
#include <string>
#include <vector>

#include "../../../include/ibdgem_b200.h"

namespace ibdhost {

class LineReader {
public:
    LineReader() = default;
    ~LineReader() { close(); }
    LineReader(const LineReader &) = delete;
    LineReader &operator=(const LineReader &) = delete;

    // On failure prints the reference's message for plain files ("Failed to open %s." + perror,
    // src/file-io.c:98-108) and returns false.
    bool open(const std::string &path);
    void close();
    // Next line including its '\n' (if any) in [*line, *line + *len); false at end of file.
    // The pointer stays valid until the next call.
    bool next(const char **line, size_t *len);
    const std::string &path() const { return path_; }

private:
    bool fill();
    std::string path_;
    gzFile gz_ = nullptr;  // gzopen reads plain files transparently as well
    std::vector<char> buf_;
    size_t beg_ = 0, end_ = 0;
    bool eof_ = false;
};

// true iff the name ends in ".gz" (src/file-io.c:10-18)
bool ends_with_gz(const std::string &fn);

// --tracts tables (hiddengem --tracts, ibdgem --hiddengem --tracts): the header line (with the leading Summary column
// or without it), and one tract's columns from Tract on (k = 0-based index within its table; start / end: START of its
// first bin and END of its last; n_sites: NUM_SITES summed over its bins), each ending in '\n'.
std::string tract_header(bool summary, bool posterior);
std::string tract_row(const hiddengem_tract &r, int64_t k, uint64_t start, uint64_t end, int64_t n_sites, bool posterior);

// --share-sd lines (hiddengem, ibdgem --hiddengem): from the posterior mean (expected[3]) and covariance (cov[3][3]) of
// the bins per state of n bins, "#% posterior IBDk sd (n = <sd of N_k>): <sd of the share in %>" for k = 0, 1, 2 and
// "#% posterior kinship (sd = <sd>): <phi>" with phi = (N_1 / 4 + N_2 / 2) / n, each ending in '\n'.
std::string share_sd_lines(const double *expected, const double *cov, double n);

}  // namespace ibdhost
