"""End-to-end drop-in tests of the native command lines on a GPU box: bin/ibdgem and bin/hiddengem
are run with the reference's own arguments and their output FILES are compared with the reference's
(the 18 shipped golden files and the reference runs under tests/golden/ref_runs)."""
import json
import os
import subprocess

import pytest

import hostlib

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _built():
    hostlib.build()


def _run(binary, args, cwd=None):
    r = subprocess.run([os.path.join(hostlib.BIN, binary)] + args, capture_output=True, text=True, cwd=cwd, timeout=300)
    assert r.returncode == 0, r.stderr
    return r


def _body(path):
    with open(path) as fh:
        return fh.read().split("\n", 1)[1]  # line 1 records the invoked command


def _same_summary(got, want, exact):
    g, w = got.splitlines(), want.splitlines()
    assert len(g) == len(w) and g[0] == w[0]
    for a, b in zip(g[1:], w[1:]):
        fa, fb = a.split("\t"), b.split("\t")
        assert fa[:3] == fb[:3] and fa[6] == fb[6]  # segment, start, end, number of sites: bit-exact
        for x, y in zip(fa[3:6], fb[3:6]):
            if exact:
                assert x == y
            elif "nan" in y:
                assert x == y
            else:  # the reference's 7 printed digits of a LINEAR product vs exp() of a log-sum
                assert float(x) == pytest.approx(float(y), rel=2e-6, abs=1e-300)


@pytest.mark.parametrize("k", [1, 2, 3])
def test_fixture_commands_reproduce_the_golden_files(fixture_dir, tmp_path, k):
    inp, gold = os.path.join(fixture_dir, "input"), os.path.join(fixture_dir, "output")
    r = _run("ibdgem", ["-H", os.path.join(inp, "test.hap"), "-L", os.path.join(inp, "test.legend"), "-I",
                        os.path.join(inp, "test.indv"), "-P", os.path.join(inp, f"test{k}.pileup"), "-N", f"sample{k}", "-O",
                        str(tmp_path)])
    assert f"Running sample{k}-vs-sample1 comparison..." in r.stderr and "Run time:" in r.stderr
    for t in (1, 2, 3):
        for kind in ("tab", "summary"):
            name = f"sample{k}.sample{t}.{kind}.txt"
            got, want = open(tmp_path / name).read(), open(os.path.join(gold, name)).read()
            if kind == "tab":
                assert got.split("\n", 1)[1] == want.split("\n", 1)[1]
                assert got.startswith("# Entered command: ")
            else:
                assert got == want  # including the reference's own underflow-to-zero row


IMPUTE_RUNS = ["nonld_w10", "ld_w10", "ld_w10_self", "ld_w25_bg", "ld_v_w10", "nonld_v_w7", "ld_D1_w10", "nonld_D05_v",
               "filters", "af_pos", "ld_w100_underflow"]
VCF_RUNS = ["vcf_nonld_w10", "vcf_ld_w10", "vcf_q30_v"]


@pytest.mark.parametrize("run", IMPUTE_RUNS + VCF_RUNS)
@pytest.mark.parametrize("extra", [[], ["--batch", "2"]])
def test_reference_runs(golden_dir, tmp_path, run, extra):
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    meta = json.load(open(os.path.join(ca, run, "ARGS.json")))
    src = ["-V", "panel.vcf"] if "vcf" in meta else ["-H", "panel.hap", "-L", "panel.legend", "-I", "panel.indv"]
    _run("ibdgem", src + ["-P", "unk.pileup", "-O", str(tmp_path)] + meta["args"] + extra, cwd=ca)
    want_files = sorted(f for f in os.listdir(os.path.join(ca, run)) if f.endswith(".txt"))
    assert sorted(os.listdir(tmp_path)) == want_files
    ld = "--LD" in meta["args"]
    for f in want_files:
        got, want = open(tmp_path / f).read(), open(os.path.join(ca, run, f)).read()
        if f.endswith(".tab.txt"):
            assert got.split("\n", 1)[1] == want.split("\n", 1)[1]  # every per-site row and counter byte-exact
        else:
            # non-LD rows are printed from the reference's own linear products (ibdgem_scores.w_lik_linear): identical
            # bytes, underflow rows included.  --LD means over the background are log-sum-exps of thousands of terms
            # in another order: compared numerically (their LIBD2 column is exact again, checked below).
            _same_summary(got, want, exact=not ld)
            if ld and "_v_" not in run and "_D" not in run:
                for a, b in zip(got.splitlines()[1:], want.splitlines()[1:]):
                    assert a.split("\t")[5] == b.split("\t")[5]


def test_no_tab_writes_only_summaries(golden_dir, tmp_path):
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    _run("ibdgem", ["-H", "panel.hap", "-L", "panel.legend", "-I", "panel.indv", "-P", "unk.pileup", "-O", str(tmp_path),
                    "--LD", "-w", "10", "--no-tab", "-s", "ind2,ind3"], cwd=ca)
    assert sorted(os.listdir(tmp_path)) == ["UNKWN.ind2.summary.txt", "UNKWN.ind3.summary.txt"]
    _same_summary(open(tmp_path / "UNKWN.ind2.summary.txt").read(),
                  open(os.path.join(ca, "ld_w10", "UNKWN.ind2.summary.txt")).read(), exact=False)


_LOOSE = ["--p01", "0.2", "--p02", "0.05", "--p12", "0.3"]
HG = [("nonld_w10", "ind2", "default", []), ("nonld_w10", "ind3", "default", []), ("nonld_w10", "ind5", "default", []),
      ("nonld_w10", "ind2", "loose", _LOOSE), ("nonld_w10", "ind3", "loose", _LOOSE), ("nonld_w10", "ind5", "loose", _LOOSE),
      ("ld_w100_underflow", "ind3", "ld_underflow", [])]


@pytest.mark.parametrize("run,ind,tag,args", HG)
def test_hiddengem_matches_reference_stdout(golden_dir, run, ind, tag, args):
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    r = _run("hiddengem", ["-s", os.path.join(ca, run, f"UNKWN.{ind}.summary.txt")] + args)
    want = open(os.path.join(ca, "hiddengem", f"{ind}.{tag}.txt")).read()
    g, w = r.stdout.splitlines(), want.splitlines()
    assert len(g) == len(w) and g[0] == w[0]
    exact = 0
    for a, b in zip(g[1:], w[1:]):
        if b.startswith("#"):
            assert a == b  # "#% IBDk (n = …): …" — integer state counts
            continue
        fa, fb = a.split("\t"), b.split("\t")
        assert fa[0] == fb[0] and fa[4] == fb[4]  # segment and Inferred_State: bit-exact
        for x, y in zip(fa[1:4], fb[1:4]):
            assert float(x) == pytest.approx(float(y), rel=2e-5)
        exact += a == b
    assert exact >= 0.9 * (len(w) - 4)  # the printed 6 digits agree except at rounding ties


def test_targets_sharded_over_two_devices(golden_dir, tmp_path):
    """--gpus 2: one host thread and one engine per device, contiguous shards of the target list."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    _run("ibdgem", ["-H", "panel.hap", "-L", "panel.legend", "-I", "panel.indv", "-P", "unk.pileup", "-O", str(tmp_path),
                    "--LD", "-w", "10", "--gpus", "2"], cwd=ca)
    want_files = sorted(f for f in os.listdir(os.path.join(ca, "ld_w10")) if f.endswith(".txt"))
    assert sorted(os.listdir(tmp_path)) == want_files
    for f in want_files:
        got, want = open(tmp_path / f).read(), open(os.path.join(ca, "ld_w10", f)).read()
        if f.endswith(".tab.txt"):
            assert got.split("\n", 1)[1] == want.split("\n", 1)[1]
        else:
            _same_summary(got, want, exact=False)


def test_panel_cache_runs_reproduce_the_golden_files(fixture_dir, tmp_path):
    """--panel-cache: the run that writes the cache and the run that loads it (another pileup) both
    reproduce the shipped golden files byte for byte."""
    inp, gold = os.path.join(fixture_dir, "input"), os.path.join(fixture_dir, "output")
    cache = str(tmp_path / "panel.cache")
    for k, what in ((1, "written"), (2, "loaded")):
        out = tmp_path / f"out{k}"
        out.mkdir()
        r = _run("ibdgem", ["-H", os.path.join(inp, "test.hap"), "-L", os.path.join(inp, "test.legend"), "-I",
                            os.path.join(inp, "test.indv"), "-P", os.path.join(inp, f"test{k}.pileup"), "-N", f"sample{k}",
                            "-O", str(out), "--panel-cache", cache])
        assert f"panel cache {cache}: {what}" in r.stderr
        for t in (1, 2, 3):
            for kind in ("tab", "summary"):
                name = f"sample{k}.sample{t}.{kind}.txt"
                assert _body(out / name) == _body(os.path.join(gold, name))


def test_hiddengem_several_tables_in_one_call(golden_dir):
    """-s given several times (additive): tables are read and formatted by several threads, scored in
    one batch, and printed in command-line order — the same text as one call per table."""
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    files = [os.path.join(ca, "nonld_w10", f"UNKWN.{ind}.summary.txt") for ind in ("ind2", "ind3", "ind5", "ind3", "ind2")]
    single = [_run("hiddengem", ["-s", f]).stdout for f in files[:3]]
    args = []
    for f in files:
        args += ["-s", f]
    together = _run("hiddengem", args).stdout
    assert together == single[0] + single[1] + single[2] + single[1] + single[0]


def _write_summary(path, l):
    with open(path, "w") as fh:
        fh.write("# SEGMENT\tSTART\tEND\tLIBD0\tLIBD1\tLIBD2\tNUM_SITES\n")
        for i, (a, b, c) in enumerate(l):
            fh.write("%d\t%d\t%d\t%e\t%e\t%e\t100\n" % (i + 1, 1000 + 6000 * i, 6940 + 6000 * i, a, b, c))


def _states(text):
    rows = [ln.split("\t") for ln in text.splitlines()[1:] if not ln.startswith("#")]
    return [r[4] for r in rows], [ln for ln in text.splitlines() if ln.startswith("#")]


# Expected hiddengem output of the tables below, stored under tests/golden/hiddengem_tables (see
# tests/golden/make_hiddengem_golden.py): per table the Inferred_State column as one string of digits and the
# three "#% IBDk" lines; for the long table also every 10th row of the printed scores.
HG_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hiddengem_tables")
TIE_PENALTIES = {"half": ["--p01", "0.5", "--p02", "0.25", "--p12", "0.5"], "one": ["--p01", "1", "--p02", "1", "--p12", "1"],
                 "default": []}


def _tie_tables():
    """Likelihoods from a small dyadic set: with power-of-two penalties the long double products are exact."""
    import numpy as np
    rng = np.random.default_rng(17)
    vals = np.array([2.0 ** -k for k in range(4, 12)] + [3 * 2.0 ** -9, 5 * 2.0 ** -10])
    tables = []
    for k, n in enumerate((40, 300, 2500)):
        l = vals[rng.integers(0, len(vals), (n, 3))]
        if k == 1:
            l[7] = l[8] = [2.0 ** -6] * 3  # identical columns: every candidate ties
        tables.append(l)
    return tables


def _long_table():
    """12,000 nearly flat bins with planted 100-bin segments."""
    import numpy as np
    rng = np.random.default_rng(23)
    n = 12000
    l = 1e-3 * (1.0 + 0.01 * rng.random((n, 3)))
    seg = np.repeat(rng.integers(0, 3, n // 100 + 1), 100)[:n]
    l[np.arange(n), seg] *= 1.05
    return l


def _golden_states(name):
    """(states, count lines) of a stored expected output, in the form _states() returns."""
    with open(os.path.join(HG_GOLDEN, name + ".states.txt")) as fh:
        lines = fh.read().splitlines()
    return list(lines[0]), lines[1:]


@pytest.mark.parametrize("pen", list(TIE_PENALTIES.values()))
def test_hiddengem_adversarial_ties_against_the_reference_binary(tmp_path, pen):
    """Likelihoods from a small dyadic set and power-of-two penalties: the reference's long double products are
    exact, so its arg-max sees many EXACT ties (lowest index wins), where sums of fp64 logarithms differ in the
    last bits.  The near-tie guard must hand such tables to the long double recurrence: Inferred_State and the
    state counts are compared with the reference's recurrence (stored golden output)."""
    tag = next(t for t, p in TIE_PENALTIES.items() if p == pen)
    for k, l in enumerate(_tie_tables()):
        p = str(tmp_path / f"tie{k}.summary.txt")
        _write_summary(p, l)
        got = _run("hiddengem", ["-s", p] + pen).stdout
        ws, wc = _golden_states(f"tie{k}.{tag}")
        gs, gc = _states(got)
        assert gs == ws and gc == wc


def test_hiddengem_long_table_past_the_long_double_range(tmp_path):
    """12,000 nearly flat bins: the reference's running products pass below LDBL_MIN around bin 10,300, lose bits and
    end at 0.00000e+00 with every later tie resolved to state 0.  Tables whose scores leave the normal long double
    range are re-evaluated with the reference's own recurrence, so states and counts still agree."""
    p = str(tmp_path / "long.summary.txt")
    _write_summary(p, _long_table())
    got = _run("hiddengem", ["-s", p]).stdout
    ws, wc = _golden_states("long")
    gs, gc = _states(got)
    assert gs == ws and gc == wc
    with open(os.path.join(HG_GOLDEN, "long.rows.txt")) as fh:
        want_rows = fh.read().splitlines()
    assert any("0.00000e+00" in r for r in want_rows)  # the reference's recurrence did underflow
    got_rows = {r.split("\t", 1)[0]: r for r in got.splitlines()[1:] if not r.startswith("#")}
    exact = sum(got_rows.get(r.split("\t", 1)[0]) == r for r in want_rows)
    assert exact >= 0.9 * len(want_rows)


def test_ibdgem_hiddengem_chaining_matches_the_two_step_run(golden_dir, tmp_path):
    """--hiddengem (additive): the window scores go into the batched Viterbi as natural logs inside the same run.
    The states must be those the reference's hiddengem infers from the summary files (golden stdout)."""
    ca = os.path.join(golden_dir, "ref_runs", "caseA")
    meta = json.load(open(os.path.join(ca, "nonld_w10", "ARGS.json")))
    _run("ibdgem", ["-H", "panel.hap", "-L", "panel.legend", "-I", "panel.indv", "-P", "unk.pileup", "-O", str(tmp_path)] +
         meta["args"] + ["--hiddengem", "--no-tab"], cwd=ca)
    for ind in ("ind2", "ind3", "ind5"):
        got = open(tmp_path / f"UNKWN.{ind}.hiddengem.txt").read()
        want = open(os.path.join(ca, "hiddengem", f"{ind}.default.txt")).read()
        gs, gc = _states(got)
        ws, wc = _states(want)
        assert gs == ws and gc == wc
        assert got.splitlines()[0] == want.splitlines()[0]
