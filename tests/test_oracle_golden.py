"""CPU tests: the oracle (oracle/liboracle.so) against the golden vectors generated from the real reference
(tests/golden/make_golden.py), and, where oracle/_ref exists (dev container), against the reference live."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from oracle import pyoracle
from tests import golden_util as gu

ROOT = Path(__file__).resolve().parent.parent
P_STAR = np.frombuffer(np.uint64(0x3FD43D136248490E).tobytes(), dtype=np.float64)[0]


@pytest.fixture(scope="module")
def grid():
    return np.load(gu.GOLDEN / "vc_function_grid.npz")


def test_kf_gammaq_bitwise(grid):
    got = np.array([pyoracle.kf_gammaq(s, z) for s, z in zip(grid["gq_s"], grid["gq_z"])])
    assert np.array_equal(got.view(np.uint64), grid["gq"].view(np.uint64))


def test_q_score_bitwise(grid):
    got = np.array([pyoracle.poisson_q(k, rd, e) for k, rd, e in zip(grid["q_k"], grid["q_rd"], grid["q_err"])])
    assert np.array_equal(got.view(np.uint64), grid["q"].view(np.uint64))
    assert (grid["q"] == -888).sum() > 100 and (grid["q"] == 100).sum() > 100 and (grid["q"] == 0).sum() > 100


def test_call_decisions_and_the_p_star_threshold(grid):
    """VC:898 as a predicate on the double p: Q >= 5 <=> p <= P_STAR (what the device evaluates)."""
    g = grid
    want = g["d_call"].astype(bool)
    dec = np.empty(len(want), bool)
    for i in range(len(want)):
        pf = pyoracle.poisson_p(g["d_kfw"][i], g["d_fw"][i], g["d_efw"][i])
        pb = pyoracle.poisson_p(g["d_kbw"][i], g["d_bw"][i], g["d_ebw"][i])
        dec[i] = (g["d_fw"][i] >= 100 and g["d_bw"][i] >= 100 and pf <= P_STAR and pb <= P_STAR)
    assert np.array_equal(dec, want)
    # the threshold itself: P_STAR is the largest double whose x87 long double Q is >= 5
    assert pyoracle.q_at_least(P_STAR, 5) and not pyoracle.q_at_least(np.nextafter(P_STAR, 1.0), 5)
    # plain fp64 log10 would accept one more double: the reason the device compares p, not Q
    assert -10 * np.log10(np.nextafter(P_STAR, 1.0)) >= 5


def test_fisher_standin(grid):
    got = np.array([pyoracle.fisher(a, b, c, d) for a, b, c, d in zip(grid["f_a"], grid["f_b"], grid["f_c"], grid["f_d"])])
    assert np.allclose(got, grid["f_p"], rtol=1e-12, atol=0)


def test_fisher_pinned_against_boost_math():
    """The Fisher column against a REAL Boost.Math hypergeometric pdf (scipy's compiled-in Boost, evaluated by
    tests/golden/make_fisher_boost.py over the reference's loop, VC:3797-3814) on all 1,202 call rows of the golden
    cases, 1,500 seeded tables up to depth ~250,000 and 2,194 SYMMETRIC tables (r = N - r or n = N - n: exhaustive for
    N <= 28, seeded beyond), where terms tie with the cutoff and a whole term of p hangs on the last bit of the pdf:
      * N <= 170 (Boost's factorial-table branch, restated in hyper_pdf_factorial): p is BIT-IDENTICAL to Boost's;
      * elsewhere the oracle's and the product's p agree with Boost's to 2e-9 relative -- on every table of Boost's
        prime-factorisation branch (N <= 104,723: any depth up to ~50,000x per strand), ties included, and on every
        non-symmetric table beyond; 16 of the 69 symmetric tables beyond N = 104,723 (Boost's Lanczos branch, whose mirror
        terms are not bitwise equal) differ by one tied term: the one unpinned corner (DESIGN.md);
      * same YES/NO strand-bias flag at the float p_value (VC:903) and the same FisherPvalue text at both precisions the
        reference prints (6 digits on the first row, 4 after) wherever p is a normal double."""
    from amplisolve_b200 import fisher_test
    g = np.load(gu.GOLDEN / "fisher_boost.npz")
    tables = list(zip(g["fw"].tolist(), g["bw"].tolist(), g["alt_fw"].tolist(), g["alt_bw"].tolist()))
    want = g["p_boost"]
    n_ties0 = int(g["n_before_ties"])
    assert n_ties0 == 2702 and int(g["n_from_fixtures"]) == 1202 and len(tables) == 4896
    N = g["fw"] + g["bw"] + g["alt_fw"] + g["alt_bw"]
    lanczos_tie = (np.arange(len(tables)) >= n_ties0) & (N > 104723)
    for name, fn in (("oracle", pyoracle.fisher), ("product", fisher_test)):
        got = np.array([fn(*t) for t in tables])
        assert np.array_equal(got[N <= 170], want[N <= 170]), name                       # bit-identical to Boost
        normal = (want > 1e-300) & ~lanczos_tie
        assert np.all(np.abs(got - want)[normal] <= 2e-9 * want[normal]), name
        assert np.all(got[want <= 1e-300] < 1e-300), name
        assert int((np.abs(got - want)[lanczos_tie] > 2e-9 * want[lanczos_tie]).sum()) <= 16, name
        for p_value in (np.float32(0.05), np.float32(0.01), np.float32(0.001)):
            assert np.array_equal((got <= p_value)[~lanczos_tie], (want <= p_value)[~lanczos_tie]), name
        for digits in (6, 4):
            assert [gu.fmt_g(x, digits) for x in got[normal]] == [gu.fmt_g(x, digits) for x in want[normal]], name
    # the strings the compiled reference (with the stand-in header) printed for the fixture calls are Boost's strings
    nf = int(g["n_from_fixtures"])
    for txt, p in zip(g["printed_by_standin"][:nf], want[:nf]):
        assert str(txt) in (gu.fmt_g(p, 6), gu.fmt_g(p, 4))


def test_product_fisher_equals_oracle_bitwise(grid):
    from amplisolve_b200 import fisher_test
    for a, b, c, d in zip(grid["f_a"], grid["f_b"], grid["f_c"], grid["f_d"]):
        assert fisher_test(a, b, c, d) == pyoracle.fisher(a, b, c, d)
    assert fisher_test(-1, 5, 1, 1) == -1.0


def oracle_on_case(case):
    from tests import synth
    normals = case["normals"][case["normal_order"]]
    rows, off = pyoracle.dense_to_rows(synth.to_oracle_layout(normals), case["pos_id"])
    nz = pyoracle.noise_estimate(rows, off, case["U"], np.float32(case["c_value"]), int(case["cutoff"]))
    return nz


@pytest.mark.parametrize("name", gu.CASES)
def test_noise_table_text_identical(name):
    case = gu.load(name)
    nz = oracle_on_case(case)
    pid = case["pos_id"]
    lines = gu.noise_table_lines(case, nz["thr"][pid], nz["germ_val"][pid], nz["germ_present"][pid])
    want = case["noise_table"].splitlines()
    assert len(lines) == len(want)
    bad = [i for i, (a, b) in enumerate(zip(lines, want)) if a != b]
    assert not bad, (bad[:5], lines[bad[0]], want[bad[0]])


@pytest.mark.parametrize("name", gu.CASES)
def test_call_rows_identical(name):
    from tests import synth
    case = gu.load(name)
    order = case["tumour_order"]
    tumours = case["tumours"][order]
    thr_slots = gu.parse_noise_thresholds(case)
    thr_u = np.zeros((case["U"], 4, 2), np.float32)
    thr_u[case["pos_id"]] = thr_slots
    ref_u = np.full(case["U"], 255, np.uint8)
    ref_u[case["pos_id"]] = case["ref_code"]
    rows, off = pyoracle.dense_to_rows(synth.to_oracle_layout(tumours), case["pos_id"])
    calls = pyoracle.call_variants(rows, off, case["U"], ref_u, thr_u, int(case["cutoff"]))
    want = gu.golden_call_rows(case)
    assert len(calls) == len(want)
    present = tumours[:, 0, :, 0] != 0xFFFFFFFF
    rows_slot = [np.nonzero(present[s])[0] for s in range(len(order))]
    first = True
    for c, w in zip(calls, want):
        slot = rows_slot[c["sample"]][c["row"]]
        chrom, pos = case["slots"][slot]
        got = (case["tumour_names"][order[c["sample"]]], chrom, pos, "ACGT"[c["ref"]], "ACGT"[c["alt"]],
               int(c["FW"] + c["BW"]), int(c["FW"]), int(c["BW"]), int(c["k_fw"]), int(c["k_bw"]),
               gu.fmt_g(c["q_fw"]), gu.fmt_g(c["q_bw"]), gu.fmt_g(c["fisher_p"], 6 if first else 4))
        assert got == w
        first = False


def test_hash_iteration_order_matches_observed_toy_order():
    """SURVEY.md A.5/B.5: with germline_dir=N the reference visits N5,N3,N2,N4,N1; with tumour_dir=T: T3,T2,T1."""
    n = [f"N/N{i}.PILEUP.ASEQ" for i in range(1, 6)]
    assert [n[i][2:4] for i in pyoracle.hash_iteration_order(n)] == ["N5", "N3", "N2", "N4", "N1"]
    t = [f"T/T{i}.PILEUP.ASEQ" for i in range(1, 4)]
    assert [t[i][2:4] for i in pyoracle.hash_iteration_order(t)] == ["T3", "T2", "T1"]


needs_ref = pytest.mark.skipif(not (ROOT / "oracle" / "_ref" / "libvc_ref_funcs.so").exists(),
                               reason="oracle/_ref is only built where /root/reference exists")


@needs_ref
def test_live_reference_grids():
    """Larger random grids against the compiled reference itself (dev container only)."""
    L = C.CDLL(str(ROOT / "oracle" / "_ref" / "libvc_ref_funcs.so"))
    rng = np.random.default_rng(99)
    n = 200000
    s = rng.integers(1, 30000, n).astype(np.float64)
    z = s * np.exp(rng.normal(scale=0.5, size=n))
    want = np.empty(n)
    L.ref_kf_gammaq_vec(s.ctypes.data_as(C.c_void_p), z.ctypes.data_as(C.c_void_p), want.ctypes.data_as(C.c_void_p), C.c_long(n))
    kf = pyoracle.lib().aso_kf_gammaq
    got = np.array([kf(a, b) for a, b in zip(s[:40000], z[:40000])])
    assert np.array_equal(got.view(np.uint64), want[:40000].view(np.uint64))


def _reference_lib():
    """The compiled reference (oracle/_ref), or None: it is built only where the original sources are at hand."""
    path = ROOT / "oracle" / "_ref" / "libvc_ref_funcs.so"
    return C.CDLL(str(path)) if path.exists() else None


def test_screen_continued_fraction_branch_never_calls(grid):
    """SURVEY.md B.6(3), the screen both caller kernels rely on: whenever kf_gammaq takes the continued-fraction
    branch (m >= k and m > 1, VC:3728) the reference's Q stays below 5 -- including where the 99-step cap leaves
    the fraction unconverged.  Checked on a dense grid with the oracle's kf_gammaq, which equals the reference's bit for bit
    on the continued-fraction points of the stored reference grid (tests/golden/vc_function_grid.npz) and, where the
    compiled reference is present, on the whole dense grid."""
    rng = np.random.default_rng(7)
    ks = np.unique(np.concatenate([np.arange(1, 400), np.geomspace(400, 2_000_000, 1500).astype(np.int64),
                                   rng.integers(1, 200000, 3000)]))
    ratios = np.concatenate([[1.0, 1.0 + 1e-12, 1.0 + 1e-9, 1.0 + 1e-7, 1.00001, 1.0001, 1.001, 1.003, 1.01, 1.02, 1.05,
                              1.1, 1.2, 1.5, 2.0, 3.0, 10.0, 100.0], 1.0 + np.geomspace(1e-6, 1.0, 40)])
    s = np.repeat(ks.astype(np.float64), len(ratios))
    z = s * np.tile(ratios, len(ks))
    keep = (z >= s) & (z > 1.0)
    s, z = s[keep], z[keep]
    kf = pyoracle.lib().aso_kf_gammaq
    out = np.array([kf(a, b) for a, b in zip(s, z)])
    cf = (grid["gq_z"] >= grid["gq_s"]) & (grid["gq_z"] > 1.0)
    stored = np.array([kf(a, b) for a, b in zip(grid["gq_s"][cf], grid["gq_z"][cf])])
    assert cf.sum() > 900 and np.array_equal(stored.view(np.uint64), grid["gq"][cf].view(np.uint64))
    L = _reference_lib()
    if L is not None:
        want = np.empty(len(s))
        L.ref_kf_gammaq_vec(s.ctypes.data_as(C.c_void_p), z.ctypes.data_as(C.c_void_p), want.ctypes.data_as(C.c_void_p),
                            C.c_long(len(s)))
        assert np.array_equal(out.view(np.uint64), want.view(np.uint64))
    p = 1.0 - out
    assert len(s) > 250000
    assert np.all(p > P_STAR), (s[p <= P_STAR][:5], z[p <= P_STAR][:5])
    assert p.min() > 0.49


def test_toy_data_end_to_end_against_reference():
    """BASELINE.json configs[0]: the whole of Toy_data through the oracle, against the noise table the compiled reference
    wrote for it (tests/golden/toy_full.npz)."""
    case = gu.load("toy_full")
    assert np.float32(case["c_value"]) == np.float32(0.002) and int(case["cutoff"]) == 100
    nz = oracle_on_case(case)
    pid = case["pos_id"]
    lines = gu.noise_table_lines(case, nz["thr"][pid], nz["germ_val"][pid], nz["germ_present"][pid])
    want = case["noise_table"].splitlines()
    assert lines == want
    assert len(want) == 41487


def test_screen_critical_mean_never_calls(grid):
    """The second exact screen of the caller (AS_MCRIT, scripts/critical_means.py): for k = 1..64 and every mean from the
    table value m*(k)(1 + 1e-9) up to 3k, the reference's Q stays below 5 -- on the series branch (m < k), at
    m <= 1 (k = 1) and on the continued-fraction branch alike; a hair below m*(k) it reaches 5.  e = 2^-20 makes
    m = depth * e exact.  Checked with the oracle's Q, which equals the reference's bit for bit on the stored reference grid's
    points with k = 1..64 (tests/golden/vc_function_grid.npz) and, where the compiled reference is present, on this grid."""
    import sys
    sys.path.insert(0, str(ROOT / "scripts"))
    from critical_means import critical_means
    mc = np.array(critical_means())
    ks, depths = [], []
    for k in range(1, 65):
        lo = int(np.ceil(mc[k - 1] * 2 ** 20))
        grid_k = np.unique(np.concatenate([lo + np.arange(0, 200), np.geomspace(lo, 3 * k * 2 ** 20 + lo, 400).astype(np.int64)]))
        ks.append(np.full(len(grid_k), k))
        depths.append(grid_k)
    k = np.concatenate(ks).astype(np.int32)
    rd = np.concatenate(depths).astype(np.int32)
    err = np.full(len(k), 2.0 ** -20, np.float32)
    kb = np.arange(1, 65, dtype=np.int32)
    rb = np.floor(mc / (1 + 1e-9) * (1 - 3e-6) * 2 ** 20).astype(np.int32)
    eb = np.full(64, 2.0 ** -20, np.float32)
    q = np.array([pyoracle.poisson_q(a, b, c) for a, b, c in zip(k, rd, err)])
    qb = np.array([pyoracle.poisson_q(a, b, c) for a, b, c in zip(kb, rb, eb)])
    small = (grid["q_k"] >= 1) & (grid["q_k"] <= 64)
    stored = np.array([pyoracle.poisson_q(a, b, c) for a, b, c in zip(grid["q_k"][small], grid["q_rd"][small], grid["q_err"][small])])
    assert small.sum() > 2000 and np.array_equal(stored.view(np.uint64), grid["q"][small].view(np.uint64))
    L = _reference_lib()
    if L is not None:
        for kk, rr, ee, got in ((k, rd, err, q), (kb, rb, eb, qb)):
            want = np.empty(len(kk), np.float64)
            L.ref_poisson_q_vec(kk.ctypes.data_as(C.c_void_p), rr.ctypes.data_as(C.c_void_p), ee.ctypes.data_as(C.c_void_p),
                                want.ctypes.data_as(C.c_void_p), C.c_long(len(kk)))
            assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    assert len(k) > 30000 and (q < 5).all(), (k[q >= 5][:5], rd[q >= 5][:5])
    # just below the critical mean the strand test passes: the table is tight, not merely safe
    assert (qb >= 5).all()
