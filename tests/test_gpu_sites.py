"""Site report: the Poisson strand tests of listed SNVs in every tumour, called or not, through every layer -- site_test_kernel
and as_site_tests_host* (against the oracle, the caller's call sets and the compiled reference's stored grid) and the sites=
argument of AmpliSolveVariantCalling (Site_Report.txt against the program's own VCFs and summary, in every program form)."""
import signal
import subprocess
from pathlib import Path

import numpy as np
import pytest

from amplisolve_b200 import api
from oracle import pyoracle
from tests import golden_util as gu
from tests import test_gpu_bam_programs as bp
from tests.test_gpu_parity import P_ABS_QUANTA, P_REL_TOL
from tests.test_gpu_sweep import BIN, C_VALUES, FORMATS, _irregular, ee, encode, run, stage, sweep_data, vc, vc_outputs

pytestmark = pytest.mark.gpu
P_STAR = np.frombuffer(np.uint64(0x3FD43D136248490E).tobytes(), np.float64)[0]


# ---- 1. the entry point against the oracle and the caller ------------------------------------------------------------
@pytest.fixture(scope="module")
def site_data(ctx):
    normals, tumours, ref, nxt, head = sweep_data()
    ref = ref.copy()
    ref[::29] = 4                                   # N reference bases: never tested
    views = ctx.estimate_thresholds_sweep(normals, C_VALUES, 100, nxt, head)["thr_view"]
    return tumours, ref, views


def expected(tumours, ref, view, slot, alt, cut=100):
    """counts and status of every (tumour, site) from the tensor; p from the oracle where the device must evaluate it"""
    fw, bw = tumours[:, 0][:, slot], tumours[:, 1][:, slot]          # [T][H][4]
    absent = fw[..., 0] >= 0x80000000
    dfw, dbw = fw.sum(-1, dtype=np.uint32), bw.sum(-1, dtype=np.uint32)
    kfw, kbw = np.take_along_axis(fw, alt[None, :, None], -1)[..., 0], np.take_along_axis(bw, alt[None, :, None], -1)[..., 0]
    testable = (ref[slot] <= 3) & (alt != ref[slot])
    status = np.where(absent, api.SITE_NO_DATA, np.where(~testable[None], api.SITE_NOT_TESTABLE,
                      np.where((dfw < cut) | (dbw < cut), api.SITE_LOW_COVERAGE, 0)))
    e = view[slot, alt]                                               # [H][2]
    return absent, dfw, dbw, kfw, kbw, status, e


def p_ok(got, want):
    well = want >= 1e-4
    return np.all(np.where(well, np.abs(got - want) <= P_REL_TOL * want, np.abs(got - want) <= P_ABS_QUANTA + P_REL_TOL * np.abs(want)))


@pytest.mark.parametrize("tile", [0, 256])
@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("n_c", [1, 2, 5, 8])
def test_site_tests_against_oracle_and_caller(ctx, site_data, n_c, fmt, tile):
    tumours, ref, views = site_data
    T, _, P, _ = tumours.shape
    slot = np.repeat(np.arange(P, dtype=np.int32), 4)                 # every (slot, alt) of the panel, alt = ref included
    alt = np.tile(np.arange(4, dtype=np.int32), P)
    counts, wide = encode(tumours, fmt)
    got = ctx.site_tests(counts, ref, views[:n_c], 100, slot, alt, wide_records=wide)
    assert got.shape == (n_c, T, 4 * P)
    ctx.set_host_tile_slots(tile)
    try:
        calls = ctx.call_variants_sweep(counts, ref, views[:n_c], 100, wide_records=wide)
    finally:
        ctx.set_host_tile_slots(0)
    seen = set()
    for c in range(n_c):
        g = got[c]
        absent, dfw, dbw, kfw, kbw, status, e = expected(tumours, ref, views[c], slot, alt)
        present = ~absent
        assert np.array_equal(g["depth_fw"][present], dfw[present]) and np.array_equal(g["depth_bw"][present], dbw[present])
        assert np.array_equal(g["alt_fw"][present], kfw[present]) and np.array_equal(g["alt_bw"][present], kbw[present])
        assert np.all(g["depth_fw"][absent] == 0) and np.all(np.isnan(g["p_fw"][absent]))
        fixed = status != 0
        assert np.array_equal(g["status"][fixed], status[fixed])
        assert np.all(np.isin(g["status"][~fixed], [api.SITE_CALLED, api.SITE_NOT_CALLED]))
        tested = present & (status != api.SITE_NOT_TESTABLE)
        assert np.all(np.isnan(g["p_fw"][~tested]))
        t_i, h_i = np.nonzero(tested)
        pick = np.random.default_rng(c).choice(len(t_i), size=min(len(t_i), 3000), replace=False)   # the oracle is slow
        t_i, h_i = t_i[pick], h_i[pick]
        for strand, d, k in ((0, dfw, kfw), (1, dbw, kbw)):
            want = np.array([pyoracle.poisson_p(int(k[t, h]), int(d[t, h]), float(e[h, strand])) for t, h in zip(t_i, h_i)])
            assert p_ok(g["p_fw" if strand == 0 else "p_bw"][t_i, h_i], want), (c, strand)
        # CALLED is the caller's decision: the same set, the same p bit for bit
        called = g["status"] == api.SITE_CALLED
        t_c, h_c = np.nonzero(called)
        mine = sorted(zip(t_c.tolist(), slot[h_c].tolist(), alt[h_c].tolist()))
        theirs = calls[c]
        assert mine == sorted(zip(theirs["sample"].tolist(), theirs["slot"].tolist(), theirs["alt"].tolist())), c
        order = np.lexsort((alt[h_c], slot[h_c], t_c))
        assert np.array_equal(g["p_fw"][t_c, h_c][order].view(np.uint64), theirs["p_fw"].view(np.uint64))
        assert np.array_equal(g["p_bw"][t_c, h_c][order].view(np.uint64), theirs["p_bw"].view(np.uint64))
        assert np.all((g["p_fw"][called] <= P_STAR) & (g["p_bw"][called] <= P_STAR))
        seen |= set(np.unique(g["status"]).tolist())
    assert seen == {1, 2, 3, 4, 5}


def test_site_tests_argument_checks(ctx, site_data):
    tumours, ref, views = site_data
    T, _, P, _ = tumours.shape
    tv = np.ascontiguousarray(views)
    out = np.zeros(8 * T * 4, api.SITE_TEST_DTYPE)

    def call(n_c, slot, alt, t=T):
        slot, alt = np.asarray(slot, np.int32), np.asarray(alt, np.int32)
        return api.lib().as_site_tests_host(ctx._h, api._hp(tumours), t, P, api._hp(ref), api._hp(tv), n_c, api._hp(slot), api._hp(alt),
                                            len(slot), 100, api._hp(out))
    assert call(1, [0, P - 1], [1, 3]) == 0
    for n_c in (0, 9):
        assert call(n_c, [0], [1]) == -1, n_c
    for slot, alt in (([P], [0]), ([-1], [0]), ([0], [4]), ([0], [-1])):
        assert call(1, slot, alt) == -1, (slot, alt)
    out[:] = np.zeros(1, api.SITE_TEST_DTYPE)
    assert call(2, [], []) == 0 and call(2, [3], [1], t=0) == 0        # nothing to do, nothing written
    assert np.all(out["status"] == 0)
    assert ctx.site_tests(tumours[:0], ref, views[:2], 100, [3], [1]).shape == (2, 0, 1)


# ---- 2. against the compiled reference's stored grid -----------------------------------------------------------------
def one_sample_tensor(k, depth, ref_base=0, alt=1):
    """one tumour, one slot per grid point: `alt` carries k reads of `depth` on both strands"""
    n = len(k)
    c = np.zeros((1, 2, n, 4), np.uint32)
    c[0, :, :, alt] = k
    c[0, :, :, ref_base] = depth - k
    return c


def test_site_tests_against_the_reference_grid(ctx):
    g = np.load(gu.GOLDEN / "vc_function_grid.npz")
    keep = g["q_err"] != -1.0                       # a caller view never holds -1 ("-1_-1" reads as 0.01)
    assert (~keep).sum() == 594
    k, rd, err = g["q_k"][keep], g["q_rd"][keep], g["q_err"][keep]
    assert np.all(k <= rd)
    n = len(k)
    counts = one_sample_tensor(k.astype(np.uint32), rd.astype(np.uint32))
    view = np.zeros((n, 4, 2), np.float32)
    view[:, 1, 0] = view[:, 1, 1] = err
    got = ctx.site_tests(counts, np.zeros(n, np.uint8), view, 1, np.arange(n), np.ones(n))[0, 0]
    q = np.array([pyoracle.q_from_p(p) for p in got["p_fw"]])
    want = g["q"][keep]
    # the p contract (DESIGN 3.6): device exp / log against glibc's, so Q agrees to 1e-9 as in test_gpu_parity; the
    # saturated (p < 1e-10) and zero (k = 0) points exactly
    assert np.allclose(q, want, rtol=1e-9, atol=1e-9)
    assert np.array_equal(q == 100, want == 100) and np.array_equal(q == 0, want == 0)
    assert (want == 100).sum() > 100 and (want == 0).sum() > 100
    assert np.array_equal(got["p_fw"].view(np.uint64), got["p_bw"].view(np.uint64))
    # decisions of VC:898 on the d_* points
    keep = (g["d_efw"] != -1.0) & (g["d_ebw"] != -1.0)
    n = int(keep.sum())
    counts = np.zeros((1, 2, n, 4), np.uint32)
    for strand, kk, dd in ((0, "d_kfw", "d_fw"), (1, "d_kbw", "d_bw")):
        counts[0, strand, :, 1] = g[kk][keep]
        counts[0, strand, :, 0] = g[dd][keep] - g[kk][keep]
    view = np.zeros((n, 4, 2), np.float32)
    view[:, 1, 0], view[:, 1, 1] = g["d_efw"][keep], g["d_ebw"][keep]
    got = ctx.site_tests(counts, np.zeros(n, np.uint8), view, int(g["d_cut"]), np.arange(n), np.ones(n))[0, 0]
    assert np.array_equal(got["status"] == api.SITE_CALLED, g["d_call"][keep].astype(bool))


# ---- 3. the program ------------------------------------------------------------------------------------------------------
def panel_rows(case):
    """(chrom, pos, ref letter) of every slot, in panel order"""
    return [(c, p, case["ref_letters"][i]) for i, (c, p) in enumerate(case["slots"])]


def site_file(case, td, extra_lines=()):
    """every called (chrom, pos, alt) of the golden summary, its other alts, every tenth panel position with all its alts
    (A,C,G,T as one multi-ALT record), an indel, a chromosome and a position not in the panel, a REF mismatch"""
    rows = panel_rows(case)
    lines = ["##fileformat=VCF-like", "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO"]
    for line in case["summary"].splitlines()[1:]:
        f = line.split("\t")
        ref, alt = f[3].split("->")
        lines.append(f"{f[1]}\t{f[2]}\t.\t{ref}\t{alt}\t.\tPASS\t.")
    for c, p, r in rows[::10]:
        if r in "ACGT":
            lines.append(f"{c}\t{p}\tid\t{r}\tA,C,G,T")
    c, p, r = rows[3]
    wrong = "ACGT"[("ACGT".index(r) + 1) % 4] if r in "ACGT" else "A"
    lines += [f"{c}\t{p}\t.\t{r}\t{r}T", f"{c}\t{p}\t.\t{r}T\t{r}", "chrUn\t5\t.\tA\tC", f"{c}\t999999999\t.\tA\tC",
              f"{c}\t{p}\t.\t{wrong}\tA", *extra_lines]
    (td / "sites.vcf").write_text("\n".join(lines) + "\n")
    n = sum(len(l.split("\t")[4].split(",")) for l in lines if not l.startswith("#") and len(l.split("\t")[3]) == 1
            and all(len(a) == 1 for a in l.split("\t")[4].split(",")))
    return n


def report(path):
    lines = Path(path).read_text().splitlines()
    assert lines[0].split("\t") == ["Filename", "Chrom", "Position", "Ref", "Alt", "RD_fw", "RD_bw", "Reads_fw", "Reads_bw", "AF",
                                    "Noise_fw", "Noise_bw", "Qscore_fw", "Qscore_bw", "Status"]
    return [l.split("\t") for l in lines[1:]]


def vcf_keys(path):
    return {(f[0], f[1], f[4]) for f in (l.split("\t") for l in Path(path).read_text().splitlines() if not l.startswith("#"))}


def vc_sites(case, error_file, out, cwd, sites="sites.vcf", env=None, tumours="T"):
    return run("AmpliSolveVariantCalling", [f"errorFile={error_file}", f"tumour_dir={tumours}", f"output_dir={out}",
                                            f"coverage_cutoff={int(case['cutoff'])}", "p_value=0.05", f"sites={sites}"], cwd, env)


def check_report(case, out, n_sites, names):
    rows = report(out / "Site_Report.txt")
    assert len(rows) == n_sites * len(names)
    assert [r[0] for r in rows[::n_sites]] == names                   # tumours in the summary's order
    summary = {}
    for l in (out / "Summary_Variant_Info.txt").read_text().splitlines()[1:]:
        f = l.split("\t")
        summary[(f[0], f[1], f[2], f[3].split("->")[1])] = (f[14], f[15])
    for nm in names:
        keys = vcf_keys(out / f"{nm}.vcf")
        for r in (r for r in rows if r[0] == nm):
            if r[-1] == "CALLED":
                assert (r[1], r[2], r[4]) in keys, r
                assert (r[12], r[13]) == summary[(nm, r[1], r[2], r[4])], r
            else:
                assert (r[1], r[2], r[4]) not in keys or r[-1] in ("NOT_IN_PANEL", "REF_MISMATCH"), r
            if r[-1] in ("NO_DATA", "NOT_IN_PANEL", "REF_MISMATCH"):
                assert r[5:14] == ["-"] * 9, r
    return rows


@pytest.mark.parametrize("name", gu.CASES)
def test_site_report_on_golden_cases(name, tmp_path):
    case = gu.load(name)
    stage(case, tmp_path)
    n = site_file(case, tmp_path)
    (tmp_path / "table.txt").write_text(case["noise_table"])
    vc(case, "table.txt", "plain", tmp_path)
    out = vc_sites(case, "table.txt", "rep", tmp_path)
    assert out.count("record skipped") == 2 and "sites.vcf line" in out
    got = vc_outputs(tmp_path / "rep")
    assert "Site_Report.txt" in got
    del got["Site_Report.txt"]
    assert got == vc_outputs(tmp_path / "plain")                     # every other output byte for byte
    names = [r.split("\t")[0] for r in (tmp_path / "rep" / "Site_Report.txt").read_text().splitlines()[1::n]]
    rows = check_report(case, tmp_path / "rep", n, names)
    status = {r[-1] for r in rows}
    assert {"CALLED", "NOT_CALLED", "LOW_COVERAGE", "NOT_TESTABLE", "NOT_IN_PANEL", "REF_MISMATCH"} <= status, status
    if name == "toy_slice":
        assert {r[-1] for r in rows if r[0] == "T3"} <= {"NO_DATA", "NOT_IN_PANEL", "REF_MISMATCH"}
        assert "NO_DATA" in status
    # a malformed line and a missing file: the error, and nothing written
    for bad, msg in (("chr1\t12\t.\tA", "fewer than five"), ("chr1\tx12\t.\tA\tC", "is not an integer")):
        (tmp_path / "bad.vcf").write_text("#h\n" + bad + "\n")
        out = vc_sites(case, "table.txt", "bad", tmp_path, sites="bad.vcf")
        assert msg in out and "bad.vcf line 2" in out
        assert not (tmp_path / "bad").exists()
    out = vc_sites(case, "table.txt", "none", tmp_path, sites="missing.vcf")
    assert "Cannot open missing.vcf" in out and not (tmp_path / "none").exists()
    # usage text for a sixth argument that is not sites=, and for eight arguments
    for args in (["x=1"], ["sites=sites.vcf", "y"]):
        r = subprocess.run([str(BIN / "AmpliSolveVariantCalling"), "errorFile=table.txt", "tumour_dir=T", "output_dir=u",
                            "coverage_cutoff=100", "p_value=0.05", *args], cwd=tmp_path, capture_output=True, text=True)
        assert "not correct" in r.stdout and "sites=" in r.stdout and not (tmp_path / "u").exists()


def test_site_report_on_irregular_rows(tmp_path):
    """RD-column rows are tested with the caller's forward depth; rows beyond a position's slots are not reported"""
    mod = _irregular()
    case = gu.load("synth_small")
    stage(case, tmp_path)
    mod.apply_patches(tmp_path, case, ee_rd=False)
    n = site_file(case, tmp_path)
    (tmp_path / "table.txt").write_text(case["noise_table"])
    vc(case, "table.txt", "plain", tmp_path, {"AS_GROUP_SAMPLES": "2"})
    vc_sites(case, "table.txt", "rep", tmp_path, env={"AS_GROUP_SAMPLES": "2"})
    got = vc_outputs(tmp_path / "rep")
    del got["Site_Report.txt"]
    assert got == vc_outputs(tmp_path / "plain")
    rows = report(tmp_path / "rep" / "Site_Report.txt")
    assert len(rows) == n * len(case["tumour_names"])
    summary = {}
    for l in (tmp_path / "rep" / "Summary_Variant_Info.txt").read_text().splitlines()[1:]:
        f = l.split("\t")
        summary.setdefault((f[0], f[1], f[2], f[3].split("->")[1]), []).append((f[14], f[15], f[4]))
    rep = {(r[0], r[1], r[2], r[4]): r for r in rows}
    # CALLED <=> the caller called (tumour, first slot of the position, alt): a repeated row's calls come out twice in the
    # summary with the same cells, the row with an RD column 9 above its counts is tested with forward depth RD - reverse
    assert {k for k, r in rep.items() if r[-1] == "CALLED"} == {k for k in summary if k in rep}
    for k, r in rep.items():
        if r[-1] == "CALLED":
            assert (r[12], r[13], str(int(r[5]) + int(r[6]))) in summary[k], r
    assert any(len(v) == 2 for k, v in summary.items() if k in rep)          # the repeated called row


# ---- 4. program forms --------------------------------------------------------------------------------------------------
def test_site_report_in_every_program_form(tmp_path, socket_path):
    import torch
    case = gu.load("synth_small")
    stage(case, tmp_path)
    site_file(case, tmp_path)
    ten = ["0.001", "0.0015", "0.002", "0.0025", "0.003", "0.0035", "0.004", "0.0045", "0.005", "0.0075"]
    ee(case, ",".join(ten), "sw", tmp_path)
    tables = sorted((tmp_path / "sw").glob("positionSpecificNoise_*.txt"))
    assert len(tables) == 10
    vc_sites(case, "sw", "vsw", tmp_path)                            # ten tables: two passes
    for t in tables:
        vc_sites(case, f"sw/{t.name}", f"one_{t.stem}", tmp_path)
        assert (tmp_path / "vsw" / t.stem / "Site_Report.txt").read_text() == (tmp_path / f"one_{t.stem}" / "Site_Report.txt").read_text()
    want = (tmp_path / f"one_{tables[0].stem}" / "Site_Report.txt").read_text()
    vc_sites(case, f"sw/{tables[0].name}", "g1", tmp_path, env={"AS_GROUP_SAMPLES": "1"})
    assert (tmp_path / "g1" / "Site_Report.txt").read_text() == want
    if torch.cuda.device_count() >= 2:
        vc_sites(case, f"sw/{tables[0].name}", "two", tmp_path, env={"AS_DEVICES": "0,1", "AS_GROUP_SAMPLES": "2"})
        assert (tmp_path / "two" / "Site_Report.txt").read_text() == want
    srv = subprocess.Popen([str(BIN / "amplisolve_b200_serve"), f"socket={socket_path}"], cwd="/", stderr=subprocess.PIPE, text=True)
    try:
        assert "ready" in srv.stderr.readline()
        for rnd in range(2):
            vc_sites(case, f"sw/{tables[0].name}", f"srv{rnd}", tmp_path, env={"AS_SERVER": socket_path})
            assert (tmp_path / f"srv{rnd}" / "Site_Report.txt").read_text() == want
    finally:
        srv.send_signal(signal.SIGTERM)
        srv.wait(timeout=20)


def test_site_report_on_bam_directories(tmp_path):
    bp.make_case(tmp_path, n_normals=4, n_tumours=3)
    bp.run("AmpliSolveErrorEstimation", bp.ee_args("ee"), tmp_path)
    table = next((tmp_path / "ee").glob("positionSpecificNoise_*.txt"))
    rows = [l.split("\t") for l in table.read_text().splitlines()[1:]]
    lines = [f"{r[0]}\t{r[1]}\t.\t{r[2]}\tA,C,G,T" for r in rows if r[2] in ("A", "C", "G", "T")]
    (tmp_path / "sites.vcf").write_text("\n".join(lines) + "\n")
    bp.run("AmpliSolveVariantCalling", bp.vc_args(f"ee/{table.name}", "vb") + ["sites=sites.vcf"], tmp_path, {"AS_GROUP_SAMPLES": "2"})
    rep = report(tmp_path / "vb" / "Site_Report.txt")
    assert len(rep) == 4 * len(lines) * len(list((tmp_path / "T").glob("*.bam")))
    # the same tumours as ASEQ files (computeCounts' output, read as ASEQ input): the same report
    dummy = (tmp_path / "vb" / "AmpliSolveVariantCalling_interm_files" / "dummyVCF_1.vcf").read_text().splitlines()
    bp.two_step(tmp_path, [tuple(l.split("\t")[:2]) for l in dummy], "T")
    bp.run("AmpliSolveVariantCalling", bp.vc_args(f"ee/{table.name}", "va") + ["sites=sites.vcf"], tmp_path)
    assert (tmp_path / "vb" / "Site_Report.txt").read_text() == (tmp_path / "va" / "Site_Report.txt").read_text()
    assert any(r[-1] == "CALLED" for r in rep)
