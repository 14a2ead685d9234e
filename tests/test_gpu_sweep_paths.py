"""Every launch path of the two sweep kernels, against the straightforward caller (call kernel 0, no screens) and the oracle.

Deferred caller (as_call_deferred.cu: scan -> resolve -> series): several pieces per range, the four scan ring geometries,
overflow of the candidate list, of the survivor lists and of both, n_c = 1 ... 8, the scan's pre-screen bound taken over
tables that disagree, short sample axes and ranges that do not start on a tile.  Noise model (as_noise_pattern.cu and the
single-value kernels): the 32-bit alt-read folds past 4096 normals, and the re-election of a slot's keep pattern.

Each test also shows that the path it targets ran: kernel-launch counts for pieces, the child process of each scan
geometry, a host model of the scan for the list overflows, a model of the pattern state machine for re-election, and
alt-read sums beyond 32 bits for the folds.  Call lists are compared byte for byte after sorting by (sample, slot, alt),
thresholds as float bit patterns.
"""
import functools
import os
import subprocess
import sys
import textwrap
from pathlib import Path

import numpy as np
import pytest

from tests.test_gpu_parity import check_calls, check_noise, oracle_calls, oracle_noise

ROOT = Path(__file__).resolve().parent.parent
pytestmark = pytest.mark.gpu

TILE = 128
PIECE_TILES = 148 * 7 * 2          # as_deferred_chunks: a piece holds at least two waves of scan CTAs
CUT = 100
ORDER = ["sample", "slot", "alt"]
ABSENT = 0xFFFFFFFF


# ---- host model of the deferred caller's scan and resolve screens ---------------------------------------------------
@functools.lru_cache(maxsize=1)
def mcrit():
    sys.path.insert(0, str(ROOT / "scripts"))
    from critical_means import critical_means
    return np.array(critical_means())


def _eff(e):
    e = np.asarray(e, np.float32)
    return np.where(e == 0, np.float32(0.0010008), e)


def scan_bounds(ref, views):
    """R = floor(e_min * 2^32) per (slot, strand): e_min over every table and every alt base but the reference; -1 puts no
    bound, e outside (0, 1) switches the pre-screen off (R = 0).  [P][2] uint64."""
    e = _eff(views)                                                      # [n_c][P][4][2]
    R = np.where((e > 0) & (e < 1), np.floor(e.astype(np.float64) * 2.0 ** 32), 0).astype(np.uint64)
    R = np.where(np.asarray(views) == -1, np.uint64(0xFFFFFFFF), R)
    is_ref = np.arange(4)[None, :] == np.asarray(ref)[:, None]           # [P][4]
    R = np.where(is_ref[None, :, :, None], np.uint64(0xFFFFFFFF), R)
    return R.min(axis=(0, 2))


def prescreen_k(depth, R):
    """as_call.cuh prescreen_k, __umulhi as (d16 * R) >> 32."""
    depth = depth.astype(np.uint64)
    d16 = np.where(depth > 0x0FFFFFFF, np.uint64(0xFFFFFFFF), depth << np.uint64(4))
    m16 = (d16 * R) >> np.uint64(32)
    lo = m16 >> np.uint64(4)
    hi = lo + (((m16 & np.uint64(15)) + np.uint64(9)) >> np.uint64(4))
    return np.where(hi <= 64, hi, lo)


def _strands(counts):
    fw = counts[:, 0].astype(np.uint64)
    bw = counts[:, 1].astype(np.uint64)
    FW = fw.sum(-1) & np.uint64(0xFFFFFFFF)
    BW = bw.sum(-1) & np.uint64(0xFFFFFFFF)
    return fw, bw, FW, BW


def scan_candidates(counts, ref, views, cut=CUT, block=1 << 18):
    """The scan's integer tests: present record, min(FW, BW) >= cut, alt != ref, ref <= 3, k > prescreen_k on both strands.
    Returns the candidate mask [T][P][4] (bool)."""
    T, _, P, _ = counts.shape
    ref = np.asarray(ref)
    out = np.zeros((T, P, 4), bool)
    for b in range(0, P, block):
        e = min(P, b + block)
        fw, bw, FW, BW = _strands(counts[:, :, b:e])
        R = scan_bounds(ref[b:e], views[:, b:e])
        mf, mb = prescreen_k(FW, R[None, :, 0]), prescreen_k(BW, R[None, :, 1])
        m = (fw > mf[..., None]) & (bw > mb[..., None])
        ok = (counts[:, 0, b:e, 0] < 0x80000000) & (np.minimum(FW, BW) >= cut)
        notref = (ref[b:e, None] <= 3) & (np.arange(4)[None, :] != ref[b:e, None])
        out[:, b:e] = m & ok[..., None] & notref[None]
    return out


def _can_pass(k, depth, err):
    k = k.astype(np.int64)
    m = depth.astype(np.float64) * _eff(err).astype(np.float64)
    mc = mcrit()[np.clip(k - 1, 0, 63)]
    return (np.asarray(err) != -1) & ~((m >= k) & (m > 1)) & ~((k >= 1) & (k <= 64) & (m >= mc))


def survivors(counts, views, cands, block=1 << 18):
    """strand_can_pass on both strands, per table, for the candidates: [n_c][T][P][4] (bool)."""
    n_c = views.shape[0]
    T, _, P, _ = counts.shape
    out = np.zeros((n_c, T, P, 4), bool)
    for b in range(0, P, block):
        e = min(P, b + block)
        fw, bw, FW, BW = _strands(counts[:, :, b:e])
        for ci in range(n_c):
            v = views[ci, b:e]                                               # [p][4][2]
            out[ci, :, b:e] = (cands[:, b:e] & _can_pass(fw, FW[..., None], v[None, :, :, 0])
                               & _can_pass(bw, BW[..., None], v[None, :, :, 1]))
    return out


def assert_calls_modelled(calls, cands, surv_ci):
    """Every call is a modelled candidate and a modelled survivor of its table."""
    s, p, a = calls["sample"], calls["slot"], calls["alt"]
    assert cands[s, p, a].all() and surv_ci[s, p, a].all()


# ---- device helpers ---------------------------------------------------------------------------------------------------
def _sweep_dev(ctx, d_t, d_ref, d_views, cap, slot_range=None):
    import torch
    from amplisolve_b200 import CALL_DTYPE
    n_c = d_views.shape[0]
    calls = torch.empty(n_c * cap * CALL_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    n = torch.zeros(n_c, dtype=torch.int64, device="cuda")
    ctx.call_variants_sweep_dev(d_t, d_ref, d_views, CUT, calls, n, slot_range=slot_range)
    torch.cuda.synchronize()
    n = n.cpu().numpy()
    assert (n <= cap).all()
    rows = calls.view(n_c, cap * CALL_DTYPE.itemsize)
    return [np.sort(rows[i, :n[i] * CALL_DTYPE.itemsize].cpu().numpy().view(CALL_DTYPE), order=ORDER) for i in range(n_c)]


def _single_dev(ctx, d_t, d_ref, d_view, cap, slot_range=None):
    import torch
    from amplisolve_b200 import CALL_DTYPE
    calls = torch.empty(cap * CALL_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    n = torch.zeros(1, dtype=torch.int64, device="cuda")
    ctx.call_variants_dev(d_t, d_ref, d_view, CUT, calls, n, slot_range=slot_range)
    torch.cuda.synchronize()
    k = int(n.item())
    assert k <= cap
    return np.sort(calls[:k * CALL_DTYPE.itemsize].cpu().numpy().view(CALL_DTYPE), order=ORDER)


def _kernel0(ctx, d_t, d_ref, d_views, cap, slot_range=None):
    ctx.set_call_kernel(0)
    try:
        return [_single_dev(ctx, d_t, d_ref, d_views[i], cap, slot_range) for i in range(d_views.shape[0])]
    finally:
        ctx.set_call_kernel(-1)


def _pieces(n_slots, want):
    tiles = (n_slots + TILE - 1) // TILE
    return max(1, min(want, 8, tiles // PIECE_TILES))


def _piece_bounds(b, e, want):
    tiles = (e - b + TILE - 1) // TILE
    n = _pieces(e - b, want)
    return [min(e, b + (tiles * ch // n) * TILE) for ch in range(n + 1)]


def _options(ctx, **kw):
    for k, v in kw.items():
        ctx.set_option(k, v)


def _reset(ctx):
    _options(ctx, deferred_chunks=1, deferred_capacity=0, call_kernel=-1, noise_kernel=-1, host_tile_slots=0)


# ---- B1: pieces ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big_panel(ctx):
    """16,577 tiles less a ragged tail (2,121,805 slots, twins every 5th position), 6 tumours, thresholds of a 5-value
    noise-floor sweep over 8 synthetic normals."""
    import torch
    P = 16577 * TILE - 51
    gen = dict(seed=424242, mean_depth=2000.0, twin_period=5, absent_rate=0.01)
    normals, ref = ctx.synth_counts_dev(8, P, **gen)
    tumours, _ = ctx.synth_counts_dev(6, P, somatic_rate=5e-4, sample_offset=1 << 20, want_ref=False, **gen)
    nxt, head = ctx.synth_twin_links_dev(P, seed=424242, twin_period=5)
    c_values = [0.001, 0.002, 0.003, 0.004, 0.005]
    thr = torch.empty((5, P, 4, 2), dtype=torch.float32, device="cuda")
    ctx.estimate_thresholds_sweep_dev(normals, c_values, CUT, thr, ctx.alloc_noise_outputs(P), nxt, head)
    views = ctx.thresholds_caller_view_dev(thr)
    torch.cuda.synchronize()
    del normals
    h_t = tumours.cpu().numpy().view(np.uint32)
    h_ref, h_views, h_head = ref.cpu().numpy(), views.cpu().numpy(), head.cpu().numpy()
    cands = scan_candidates(h_t, h_ref, h_views)
    surv = survivors(h_t, h_views, cands)
    want = _kernel0(ctx, tumours, ref, views, 1 << 19)
    yield dict(P=P, d_t=tumours, d_ref=ref, d_views=views, h_t=h_t, h_ref=h_ref, h_views=h_views, h_head=h_head,
               cands=cands, surv=surv, want=want)
    _reset(ctx)


def _in_range(calls, b, e):
    return calls[(calls["slot"] >= b) & (calls["slot"] < e)]


def _oracle_near(bp, got, bounds, ci, slot_range=None, span=2 * TILE):
    """The oracle on every slot within +-2 tiles of each boundary, widened to whole twin groups, inside the slot range
    that was called."""
    P, head = bp["P"], bp["h_head"]
    lo, hi = slot_range if slot_range is not None else (0, P)
    sel = np.zeros(P, bool)
    for q in bounds:
        sel[max(0, q - span):min(P, q + span)] = True
    sel[head[sel]] = True                                 # the whole group: its head and every member of that head
    sel |= sel[head]
    sel[:lo] = False
    sel[hi:] = False
    slots = np.nonzero(sel)[0]
    sub = np.ascontiguousarray(bp["h_t"][:, :, slots])
    pos = np.arange(len(slots), dtype=np.int32)
    want, _, _ = oracle_calls(sub, pos, len(slots), bp["h_ref"][slots], bp["h_views"][ci][slots], CUT)
    g = got[np.isin(got["slot"], slots)].copy()
    g["slot"] = np.searchsorted(slots, g["slot"])
    present = sub[:, 0, :, 0] != ABSENT
    check_calls(g, want, [np.nonzero(present[s])[0] for s in range(sub.shape[0])])
    return len(g)


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6, 7, 8])
def test_deferred_pieces(ctx, big_panel, k):
    """Item 1: the multi-piece path of as_launch_call_deferred -- per-piece list shares cap / n_chunks, the scan of piece
    i+1 beside the resolve / series of piece i on the side stream, the event join.  deferred_chunks = k cuts the
    2,121,805-slot range into min(k, tiles // 2072) pieces (the kernel-launch count shows it: 3 per piece); every table
    equals call kernel 0 and, around every piece boundary, the oracle."""
    bp = big_panel
    P = bp["P"]
    pieces = min(k, ((P + TILE - 1) // TILE) // PIECE_TILES)
    assert pieces == k
    try:
        ctx.set_option("deferred_chunks", k)
        n0 = ctx.kernel_launches
        got = _sweep_dev(ctx, bp["d_t"], bp["d_ref"], bp["d_views"], 1 << 19)
        assert ctx.kernel_launches - n0 == 3 * pieces
        ctx.set_call_kernel(20)
        n0 = ctx.kernel_launches
        one = _single_dev(ctx, bp["d_t"], bp["d_ref"], bp["d_views"][0], 1 << 19)
        assert ctx.kernel_launches - n0 == 3 * pieces
    finally:
        _reset(ctx)
    assert one.tobytes() == bp["want"][0].tobytes()
    for ci, w in enumerate(bp["want"]):
        assert len(w) > 100 and got[ci].tobytes() == w.tobytes(), ci
        assert_calls_modelled(got[ci], bp["cands"], bp["surv"][ci])
    if k in (1, 3, 8):
        for ci in (0, 4):
            assert _oracle_near(bp, got[ci], _piece_bounds(0, P, k), ci) > 0


def test_deferred_pieces_unaligned_range(ctx, big_panel):
    """Items 1 and 6: a slot range (77, P - 13) that starts inside a tile, cut into 8 pieces (the tail of the range is a
    ragged tile) -- equal to call kernel 0 on the same range."""
    bp = big_panel
    P = bp["P"]
    b, e = 77, P - 13
    assert _pieces(e - b, 8) == 8
    try:
        ctx.set_option("deferred_chunks", 8)
        n0 = ctx.kernel_launches
        got = _sweep_dev(ctx, bp["d_t"], bp["d_ref"], bp["d_views"], 1 << 19, slot_range=(b, e))
        assert ctx.kernel_launches - n0 == 3 * 8
    finally:
        _reset(ctx)
    for ci, w in enumerate(bp["want"]):
        assert got[ci].tobytes() == _in_range(w, b, e).tobytes(), ci
    assert _oracle_near(bp, got[0], _piece_bounds(b, e, 8), 0, slot_range=(b, e)) > 0


@pytest.fixture(scope="module")
def strong_panel(ctx, big_panel):
    """The big panel's tumours with an alt at 10 % on both strands of every record of every 8th slot: most candidates are
    then survivors, so that a survivor list can be shown to overflow even when the candidate list left some out."""
    import torch
    bp = big_panel
    h = bp["h_t"].copy()
    slots = np.arange(0, bp["P"], 8)
    alt = (bp["h_ref"][slots].astype(np.int64) + 1) % 4
    for st in (0, 1):
        rec = h[:, st, slots]                                            # [T][n][4]
        present = rec[..., 0] != ABSENT
        k = np.where(present, rec.astype(np.int64).sum(-1) // 10, 0).astype(np.uint32)
        rec[:, np.arange(len(slots)), alt] += k
        h[:, st, slots] = rec
    d_t = torch.from_numpy(h.view(np.int32)).cuda()
    cands = scan_candidates(h, bp["h_ref"], bp["h_views"])
    surv = survivors(h, bp["h_views"], cands)
    want = _kernel0(ctx, d_t, bp["d_ref"], bp["d_views"], 1 << 21)
    return dict(d_t=d_t, cands=cands, surv=surv, want=want)


@pytest.mark.parametrize("k", [2, 8])
def test_deferred_pieces_every_share_overflows(ctx, big_panel, strong_panel, k):
    """Items 1 and 3: a deferred_capacity whose per-piece share is exceeded, per the scan model, by the candidates of every
    piece, and whose survivor share (a quarter, divided among the pieces) is exceeded by the survivors of some table even
    if every candidate left out of the list were one -- both overflow paths (inline resolve in the scan and in the resolve
    kernel) run in every piece.  The call sets do not change."""
    bp, sp = big_panel, strong_panel
    bounds = _piece_bounds(0, bp["P"], k)
    n_cand = [int(sp["cands"][:, q0:q1].sum()) for q0, q1 in zip(bounds, bounds[1:])]
    n_surv = [int(sp["surv"][:, :, q0:q1].sum(axis=(1, 2, 3)).max()) for q0, q1 in zip(bounds, bounds[1:])]
    x = min(n_cand) - 1                                   # candidate share: one fewer than the smallest piece needs
    cap = k * x
    share_s = max(1, cap // 4) // k
    for c, s in zip(n_cand, n_surv):
        assert c > x and s - (c - x) > share_s, (c, s, x, share_s)
    try:
        _options(ctx, deferred_chunks=k, deferred_capacity=cap)
        got = _sweep_dev(ctx, sp["d_t"], bp["d_ref"], bp["d_views"], 1 << 21)
    finally:
        _reset(ctx)
    for ci, w in enumerate(sp["want"]):
        assert len(w) > 100_000 and got[ci].tobytes() == w.tobytes(), ci
        assert_calls_modelled(got[ci], sp["cands"], sp["surv"][ci])


def test_deferred_capacity_beyond_the_automatic_one(ctx, big_panel):
    """A deferred_capacity above the automatic capacity (1 Mi candidates here) sizes the scratch for itself: the lists
    must not run past it.  Same call sets."""
    bp = big_panel
    try:
        _options(ctx, deferred_chunks=2, deferred_capacity=3 << 20)
        got = _sweep_dev(ctx, bp["d_t"], bp["d_ref"], bp["d_views"], 1 << 19)
    finally:
        _reset(ctx)
    for ci, w in enumerate(bp["want"]):
        assert got[ci].tobytes() == w.tobytes(), ci


def test_deferred_pieces_inside_host_tiles(ctx, big_panel):
    """Item 1 through the host entry point: upload tiles of 1,060,864 slots (8,288 tiles: 4 pieces each at
    deferred_chunks = 8) plus a 77-slot tail; calls equal call kernel 0, and the oracle around every piece and tile
    boundary."""
    bp = big_panel
    P = bp["P"]
    TP = 1_060_864
    try:
        _options(ctx, deferred_chunks=8, host_tile_slots=TP)
        got = ctx.call_variants_sweep(bp["h_t"], bp["h_ref"], bp["h_views"], CUT)
    finally:
        _reset(ctx)
    assert _pieces(TP, 8) == 4
    for ci, w in enumerate(bp["want"]):
        assert got[ci].tobytes() == w.tobytes(), ci
    bounds = sorted({q for t0 in range(0, P, TP) for q in _piece_bounds(t0, min(P, t0 + TP), 8)})
    assert _oracle_near(bp, got[0], bounds, 0) > 0


# ---- B2: scan geometries -----------------------------------------------------------------------------------------------
CHILD = textwrap.dedent("""
    import sys
    import numpy as np
    import torch
    sys.path.insert(0, sys.argv[1])
    from amplisolve_b200 import Context
    from tests.test_gpu_sweep_paths import _sweep_dev
    d = np.load(sys.argv[2])
    ref, views = d["ref"], d["views"]
    P, out = len(ref), {}
    with Context(0) as ctx:
        ctx.set_call_kernel(20)
        d_ref, d_views = torch.from_numpy(ref).cuda(), torch.from_numpy(views).cuda()
        for T in d["Ts"]:
            counts = d[f"counts_{T}"]
            for ci, g in enumerate(ctx.call_variants_sweep(counts, ref, views, 100)):
                out[f"host_{T}_{ci}"] = g
            d_t = torch.from_numpy(counts.view(np.int32)).cuda()
            for ci, g in enumerate(_sweep_dev(ctx, d_t, d_ref, d_views, 1 << 16, slot_range=(77, P - 13))):
                out[f"range_{T}_{ci}"] = g
            ctx.set_option("deferred_capacity", 3)
            for ci, g in enumerate(_sweep_dev(ctx, d_t, d_ref, d_views, 1 << 16)):
                out[f"tiny_{T}_{ci}"] = g
            ctx.set_option("deferred_capacity", 0)
    np.savez(sys.argv[3], **out)
""")


@pytest.fixture(scope="module")
def geom_inputs(ctx, tmp_path_factory):
    """T in {1, 2, 4, 7, 17, 50} tumours (T = 50: gridDim.y = 4 with 16-sample chunks) on a 3,001-slot panel, 3 tables."""
    P, Ts = 3001, [1, 2, 4, 7, 17, 50]
    gen = dict(seed=9090, mean_depth=1800.0, twin_period=4, absent_rate=0.02)
    normals, ref = ctx.synth_counts_dev(10, P, **gen)
    nxt, head = ctx.synth_twin_links_dev(P, seed=9090, twin_period=4)
    import torch
    thr = torch.empty((3, P, 4, 2), dtype=torch.float32, device="cuda")
    ctx.estimate_thresholds_sweep_dev(normals, [0.001, 0.0025, 0.004], CUT, thr, ctx.alloc_noise_outputs(P), nxt, head)
    views = ctx.thresholds_caller_view_dev(thr).cpu().numpy()
    tum, _ = ctx.synth_counts_dev(max(Ts), P, somatic_rate=0.01, sample_offset=1 << 20, want_ref=False, **gen)
    tum = tum.cpu().numpy().view(np.uint32)
    h_ref = ref.cpu().numpy()
    counts = {T: np.ascontiguousarray(tum[:T]) for T in Ts}
    path = tmp_path_factory.mktemp("geom") / "in.npz"
    np.savez(path, ref=h_ref, views=views, Ts=np.array(Ts), **{f"counts_{T}": c for T, c in counts.items()})
    want = {}
    ctx.set_call_kernel(0)
    try:
        for T in Ts:
            want[T] = [ctx.call_variants(counts[T], h_ref, views[ci], CUT) for ci in range(3)]
    finally:
        ctx.set_call_kernel(-1)
    return dict(P=P, Ts=Ts, path=path, want=want)


@pytest.mark.parametrize("geom", [0, 1, 2, 3])
def test_scan_geometries(geom_inputs, geom, tmp_path):
    """Item 2 (and 6): AS_SCAN_GEOM is read once per process, so each ring geometry -- 0 = (3, 2), 1 = (4, 2), 2 = (3, 3),
    3 = (2, 3) samples per stage and stages -- runs in a child process: the host sweep, the device sweep on the unaligned
    range (77, P - 13) and with lists of 3 candidates, for 1 ... 50 tumours (T = 1, 2 are below a stage's K).  Every
    result equals call kernel 0 computed here."""
    gi = geom_inputs
    out = tmp_path / "out.npz"
    env = dict(os.environ, AS_SCAN_GEOM=str(geom))
    r = subprocess.run([sys.executable, "-c", CHILD, str(ROOT), str(gi["path"]), str(out)], env=env, cwd=str(ROOT),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    got = np.load(out)
    P = gi["P"]
    for T in gi["Ts"]:
        for ci, w in enumerate(gi["want"][T]):
            assert len(w) > 0 or T < 4
            assert got[f"host_{T}_{ci}"].tobytes() == w.tobytes(), (T, ci)
            assert got[f"range_{T}_{ci}"].tobytes() == _in_range(w, 77, P - 13).tobytes(), (T, ci)
            assert got[f"tiny_{T}_{ci}"].tobytes() == w.tobytes(), (T, ci)
    assert sum(len(w) for w in gi["want"][50]) > 100


# ---- B3: list capacities, n_c = 1 ... 8 ---------------------------------------------------------------------------------
def _strong_tumours(T, P, seed):
    """Tumours whose candidates are mostly real calls (4 % of records carry an alt at 5-20 % on both strands), so that a
    table's survivors can outnumber a quarter of the candidates; the rest carry 0-2 noise reads per base."""
    rng = np.random.default_rng(seed)
    ref = rng.integers(0, 4, P).astype(np.uint8)
    c = rng.integers(0, 3, (T, 2, P, 4)).astype(np.uint32)
    depth = rng.integers(800, 4000, (T, 2, P)).astype(np.uint32)
    hit = rng.random((T, P)) < 0.04
    alt = (ref[None, :] + rng.integers(1, 4, (T, P))) % 4
    vaf = rng.uniform(0.05, 0.2, (T, P))
    for st in (0, 1):
        k = np.rint(depth[:, st] * vaf).astype(np.uint32)
        t_i, p_i = np.nonzero(hit)
        c[t_i, st, p_i, alt[t_i, p_i]] = k[t_i, p_i]
        c[:, st, np.arange(P), ref] = 0
        c[:, st, np.arange(P), ref] = depth[:, st] - c[:, st].sum(-1)
    c[:, :, ::211] = ABSENT
    return c, ref


@pytest.mark.parametrize("n_c", [1, 2, 3, 4, 5, 6, 7, 8])
def test_deferred_capacities(ctx, n_c):
    """Items 3 and 4: for every n_c (6 and 7 take the rank_hi packing of the resolve kernel), capacities chosen with the
    scan model so that (i) nothing overflows, (ii) only the survivor lists do, (iii) the candidate list overflows by
    exactly one entry, (iv) both lists hold one entry.  Every table equals call kernel 0, and every call is a modelled
    survivor of its table."""
    import torch
    T, P = 12, 2500
    tum, ref = _strong_tumours(T, P, seed=300 + n_c)
    rng = np.random.default_rng(n_c)
    base = rng.choice(np.array([0.001, 0.002, 0.003, 0.0, 0.005], np.float32), (P, 4, 2))
    views = np.stack([base * np.float32(1 + 0.4 * ci) for ci in range(n_c)]).astype(np.float32)
    cands = scan_candidates(tum, ref, views)
    surv = survivors(tum, views, cands)
    N = int(cands.sum())
    S = surv.sum(axis=(1, 2, 3))
    assert N > 200 and 4 * S.max() > N + 8, (N, S)
    cases = {"none": max(N, 4 * int(S.max())) + 8, "survivors": N, "candidates": N - 1, "one": 1}
    assert N <= cases["none"] and S.max() <= cases["none"] // 4
    assert N <= cases["survivors"] and S.max() > cases["survivors"] // 4
    assert N == cases["candidates"] + 1
    assert N > 1 and S.max() > 1
    d_t, d_ref, d_views = (torch.from_numpy(tum.view(np.int32)).cuda(), torch.from_numpy(ref).cuda(),
                           torch.from_numpy(views).cuda())
    want = _kernel0(ctx, d_t, d_ref, d_views, 1 << 16)
    try:
        ctx.set_call_kernel(20)
        for name, cap in cases.items():
            ctx.set_option("deferred_capacity", cap)
            got = _sweep_dev(ctx, d_t, d_ref, d_views, 1 << 16)
            for ci in range(n_c):
                assert got[ci].tobytes() == want[ci].tobytes(), (name, ci)
                assert_calls_modelled(got[ci], cands, surv[ci])
    finally:
        _reset(ctx)
    assert all(len(w) > 50 for w in want)


# ---- B4: screens across tables ------------------------------------------------------------------------------------------
BOUNDARY_ES = np.array([2.0 ** -9, 2.0 ** -7, 0.002, 0.0, 1e-6, -1.0, 0.999, 2.0 ** -20, 0.01, 3e-4], np.float32)


def _prescreen_case(seed, n_c=8):
    """test_integer_prescreen_boundaries with 8 tables: each table takes its own values from the boundary set, so the
    scan's bound (the smallest over tables and alts) differs from most tables' own."""
    rng = np.random.default_rng(seed)
    P, T = 640, 40
    ref = rng.integers(0, 4, P).astype(np.uint8)
    views = BOUNDARY_ES[rng.integers(0, len(BOUNDARY_ES), (n_c, P, 4, 2))]
    same = rng.random(P) < 0.3                      # one value for all bases / strands of a table
    views[:, same] = BOUNDARY_ES[rng.integers(0, len(BOUNDARY_ES), (n_c, same.sum()))][:, :, None, None]
    views[0] = np.where(rng.random((P, 4, 2)) < 0.6, np.float32(0.05), views[0])   # table 0 mostly above the others
    tumours = np.zeros((T, 2, P, 4), np.uint32)
    depth = (rng.choice([512, 1024, 2048, 3000, 5000, 65536, 100000, 1 << 20], (T, 2, P)) * rng.integers(1, 4, (T, 2, P))).astype(np.int64)
    for st in (0, 1):
        for b in range(4):
            e = _eff(views[rng.integers(0, n_c, P), np.arange(P), b, st]).astype(np.float64)   # a random table's boundary
            m = depth[:, st] * np.maximum(e, 0)[None, :]
            k = np.floor(m).astype(np.int64) + rng.integers(-2, 4, (T, P))
            k = np.where(rng.random((T, P)) < 0.15, rng.integers(0, 4, (T, P)), k)
            tumours[:, st, :, b] = np.clip(k, 0, depth[:, st] // 8)
    for st in (0, 1):
        rest = depth[:, st] - tumours[:, st].sum(-1) + tumours[:, st, np.arange(P), ref]
        tumours[:, st, np.arange(P), ref] = np.maximum(rest, 0)
    return tumours, ref, views


def _critical_mean_case(n_c=8):
    """test_critical_mean_screen with 8 tables: table ci scales e = 2^-20 by 2^(ci - 3), so a record straddles the critical
    mean of one table and lies far from it in the others; the scan's bound comes from table 0's 2^-23."""
    mc = mcrit() / (1 + 1e-9)
    offs = np.array([-1e-1, -1e-2, -1e-4, 1e-4, 1e-2, 1e-1])
    ks = np.arange(1, 65)
    P = 64 * n_c
    T = len(offs)
    views = np.empty((n_c, P, 4, 2), np.float32)
    ref = np.zeros(P, np.uint8)
    tumours = np.zeros((T, 2, P, 4), np.uint32)
    for tab in range(n_c):                          # slot block tab: records at table tab's critical mean
        slots = (ks - 1) + 64 * tab
        for ci in range(n_c):
            views[ci, slots] = np.float32(2.0 ** (-20 + ci - 3))
        e_tab = 2.0 ** (-20 + tab - 3)
        for si, off in enumerate(offs):
            depth = np.rint(mc * (1 + off) / e_tab).astype(np.int64)
            for st in (0, 1):
                tumours[si, st, slots, 1] = ks
                tumours[si, st, slots, 0] = depth - ks
    return tumours, ref, views


@pytest.mark.parametrize("case", ["prescreen-1", "prescreen-2", "critical-mean"])
def test_screens_across_tables(ctx, case):
    """Item 5: the scan pre-screens against the smallest threshold over all tables and alts, the resolve kernel screens
    each table on its own.  With 8 tables that disagree per slot, every table equals call kernel 0 on that table and the
    oracle, and the model shows slots where the scan's bound is below the table's own bound."""
    import torch
    if case == "critical-mean":
        tumours, ref, views = _critical_mean_case()
    else:
        tumours, ref, views = _prescreen_case(seed=77 + int(case[-1]))
    n_c, P, T = views.shape[0], views.shape[1], tumours.shape[0]
    bound = scan_bounds(ref, views)
    own = np.stack([scan_bounds(ref, views[ci:ci + 1]) for ci in range(n_c)])
    assert (own > bound[None]).any(axis=(1, 2)).sum() >= n_c - 1
    cands = scan_candidates(tumours, ref, views)
    surv = survivors(tumours, views, cands)
    d_t, d_ref, d_views = (torch.from_numpy(tumours.view(np.int32)).cuda(), torch.from_numpy(ref).cuda(),
                           torch.from_numpy(views).cuda())
    want = _kernel0(ctx, d_t, d_ref, d_views, 1 << 17)
    try:
        ctx.set_call_kernel(20)
        got = _sweep_dev(ctx, d_t, d_ref, d_views, 1 << 17)
        ctx.set_option("deferred_capacity", 5)
        tiny = _sweep_dev(ctx, d_t, d_ref, d_views, 1 << 17)
    finally:
        _reset(ctx)
    pos = np.arange(P, dtype=np.int32)
    for ci in range(n_c):
        assert got[ci].tobytes() == want[ci].tobytes() and tiny[ci].tobytes() == want[ci].tobytes(), ci
        assert_calls_modelled(got[ci], cands, surv[ci])
        w, _, _ = oracle_calls(tumours, pos, P, ref, views[ci], CUT)
        check_calls(got[ci], w, [pos for _ in range(T)])
    assert sum(len(w) for w in want) > 200 and len({len(w) for w in want}) > 2


# ---- C1: 32-bit alt-read folds --------------------------------------------------------------------------------------------
def af_limit(d):
    return (26843545 * int(d)) >> 29


FOLD_C = [0.001, 0.0015, 0.002, 0.003, 0.004, 0.005, 0.0075, 0.01]


def _fold_normals(S):
    """P = 384 (3 tiles).  Every record: FW = 2^24 - 101, BW = 100, each alt base at af_limit(FW) on the forward strand
    (kept: a base's kept alt reads grow by ~838,855 per record), RD = 2^24 - 1 < 2^24 (the fast path).  Slots 100..131: one
    record late in the sample order has RD >= 2^24 (the redo path after the folds).  Twins: slots 140/141 (a pair inside
    a tile), 255/256 (a pair cut by a tile edge: pair kernel), 300/301/302 (a triple: general kernel)."""
    P = 384
    FW = (1 << 24) - 101
    L = af_limit(FW)
    c = np.zeros((S, 2, P, 4), np.uint32)
    c[:, 0, :, 1:] = L
    c[:, 0, :, 0] = FW - 3 * L
    x = np.arange(P) % 5                                 # 0..4 reverse-strand alt reads: kept (af_limit(100) = 4)
    c[:, 1, :, 1] = x
    c[:, 1, :, 0] = 100 - x
    for p in range(100, 132):
        c[S - 1 - (p % 7), 0, p, 0] += 300             # RD = 2^24 + 299
    pos_id = np.arange(P, dtype=np.int64)
    for group in ((140, 141), (255, 256), (300, 301, 302)):
        pos_id[list(group)] = pos_id[group[0]]
    _, dense = np.unique(pos_id, return_inverse=True)
    return c, dense.astype(np.int32), L


@pytest.fixture(scope="module", params=[4095, 4096, 4097, 6000])
def fold_case(request):
    S = request.param
    counts, pos_id, L = _fold_normals(S)
    U = int(pos_id.max()) + 1
    cache = {}

    def want(cv):
        if cv not in cache:
            cache[cv] = oracle_noise(counts, pos_id, U, np.float32(cv), CUT)
        return cache[cv]
    return dict(S=S, counts=counts, pos_id=pos_id, L=L, want=want)


def _dev_noise(out):
    g = {k: v.cpu().numpy() for k, v in out.items()}
    g["count"], g["nrec"] = g["count"].view(np.uint32), g["nrec"].view(np.uint32)
    return g


def _run_noise_everywhere(ctx, counts, pos_id, want, c_values, single_kernels, sweep_kernels, sweep_ncs, tiles):
    """estimate_thresholds_dev under each single-value kernel, estimate_thresholds_sweep_dev for each n_c under each sweep
    kernel, and the host entry points at each upload tile size; every table against the oracle."""
    import torch
    from amplisolve_b200 import twin_links
    nxt, head = twin_links(pos_id)
    P = counts.shape[2]
    d_n = torch.from_numpy(counts.view(np.int32)).cuda()
    d_nxt, d_head = torch.from_numpy(nxt).cuda(), torch.from_numpy(head).cuda()
    try:
        for v in single_kernels:
            ctx.set_noise_kernel(v)
            out = ctx.alloc_noise_outputs(P)
            ctx.estimate_thresholds_dev(d_n, c_values[2], CUT, out, d_nxt, d_head)
            torch.cuda.synchronize()
            check_noise(_dev_noise(out), want(c_values[2]), pos_id)
        for v in sweep_kernels:
            ctx.set_noise_kernel(v)
            for n_c in sweep_ncs:
                cv = c_values[:n_c]
                thr = torch.full((n_c, P, 4, 2), -7.0, dtype=torch.float32, device="cuda")
                out = ctx.alloc_noise_outputs(P)
                ctx.estimate_thresholds_sweep_dev(d_n, cv, CUT, thr, out, d_nxt, d_head)
                torch.cuda.synchronize()
                g = _dev_noise(out)
                for ci, c in enumerate(cv):
                    g["thr"] = thr[ci].cpu().numpy()
                    check_noise(g, want(c), pos_id)
        ctx.set_noise_kernel(-1)
        for tile in tiles:
            ctx.set_host_tile_slots(tile)
            check_noise(ctx.estimate_thresholds(counts, c_values[2], CUT, nxt, head), want(c_values[2]), pos_id)
            sw = ctx.estimate_thresholds_sweep(counts, c_values[:5], CUT, nxt, head)
            for ci, c in enumerate(c_values[:5]):
                check_noise(dict(sw, thr=sw["thr"][ci]), want(c), pos_id)
    finally:
        ctx.set_noise_kernel(-1)
        ctx.set_host_tile_slots(0)


def test_noise_alt_read_folds(ctx, fold_case):
    """Item 7: AS_FOLD_EVERY = 4096 bounds the 32-bit alt-read sums of the pattern kernel (pat_fold), the staged kernel,
    noise_main_kernel and the pair kernel (two records per sample).  With 4095, 4096, 4097 and 6000 normals whose kept alt
    reads sit at the 5 % limit of a depth just under 2^24, a base's sum over all normals passes 2^32 at 6000 (it would wrap
    a uint32 after ~5,120 records and an int32 after ~2,560 without the folds).  Every noise kernel 0 ... 8, the sweep
    with n_c 1, 2, 3, 5, 8 under the default and the non-interleaved kernel, and the host entry points: the oracle's
    tables bit for bit."""
    fc = fold_case
    S, L = fc["S"], fc["L"]
    assert L == 838855
    if S == 6000:
        assert S * L > 1 << 32 and 2 * 2048 * L < 1 << 32
    want = fc["want"](0.002)
    assert (want["count"][fc["pos_id"][:100], 1:] == S).all()                 # every record kept: the sums are the big ones
    _run_noise_everywhere(ctx, fc["counts"], fc["pos_id"], fc["want"], FOLD_C, range(9), [-1, 8], [1, 2, 3, 5, 8], [0, 128])


# ---- C2: pattern re-election -----------------------------------------------------------------------------------------------
PAT_K = 4   # records per stage of every noise_pattern_kernel form


def _rec(kind, rng):
    """One record (fw[4], bw[4]) of a slot whose reference base is A.  R: the reference pattern (C, G, T kept; G sometimes
    exactly at the 5 % limit), G: a germline carrier at 50 % (G, T kept), B: G one read above the 5 % limit (C, T kept),
    U: uncovered (FW below the cutoff), X: absent."""
    if kind == "X":
        return np.full(4, ABSENT, np.uint32), np.full(4, ABSENT, np.uint32)
    out = []
    for st in (0, 1):
        D = int(rng.integers(1500, 2600)) if kind != "U" or st == 1 else 60
        L = af_limit(D)
        v = np.zeros(4, np.int64)
        if kind in ("R", "U"):
            v[1:] = rng.integers(0, 4, 3)
            if st == 0 and rng.random() < 0.5:
                v[2] = L
        elif kind == "G":
            v[1] = D // 2
            v[2:] = rng.integers(0, 3, 2)
        elif kind == "B":
            v[1], v[3] = rng.integers(0, 3, 2)
            v[2] = L + 1 if st == 0 else rng.integers(0, 3)
        v[0] = D - v[1:].sum()
        out.append(v.astype(np.uint32))
    return out[0], out[1]


MASK = {"R": 0b1110, "G": 0b1100, "B": 0b1010, "U": 0, "X": 0}


def pattern_branches(seq):
    """pat_accumulate / pat_irregular of as_noise_pattern.cu over one slot's records, stage by stage: counts of the three
    branches of pat_irregular (regular after all, takeover, spill)."""
    pat, cnt0, irr = None, 0, 0
    n = {"regular": 0, "takeover": 0, "spill": 0}
    for t in range(0, len(seq), PAT_K):
        irregular = []
        for kind in seq[t:t + PAT_K]:
            m = MASK[kind]
            if pat is None and m:
                pat = m
            if m and m == pat:
                cnt0 += 1
            elif m:
                irregular.append(m)
        for m in irregular:
            if m == pat:
                n["regular"] += 1
                cnt0 += 1
            elif cnt0 <= irr:
                n["takeover"] += 1
                pat, cnt0, irr = m, 1, 0
            else:
                n["spill"] += 1
                irr += 1
    return n


def _sequences(S, rng):
    fixed = ["G" + "R" * (S - 1), "GGRR" + "R" * (S - 4), "XU" + "G" + "R" * (S - 3), "UUXG" + "R" * (S - 4),
             ("RGB" * S)[:S], ("GBR" * S)[:S], ("GGGRRRRRRBBBBBBBBBBBBB" * 2)[:S].ljust(S, "B"),
             ("BGGRRRR" * 3)[:S].ljust(S, "R"), "R" * S, "G" * S, ("XR" * S)[:S], "B" + "G" * (S - 1)]
    rand = ["".join(rng.choice(list("RRRRGGBUX"), S)) for _ in range(60)]
    return fixed + rand


def _pattern_normals(S, seed):
    """Singleton slots from the sequences, then in-tile twin pairs whose two slots elect different patterns (R vs G, G vs
    B, a takeover vs none)."""
    rng = np.random.default_rng(seed)
    seqs = _sequences(S, rng)
    pairs = [("R" * S, "G" * S), ("G" + "R" * (S - 1), "B" * S), ("GGRR" + "R" * (S - 4), ("RGB" * S)[:S]),
             ("B" + "G" * (S - 1), "R" * S)]
    slot_seqs = list(seqs)
    pos = list(range(len(seqs)))
    for a, b in pairs:
        pos += [len(pos), len(pos)]                     # consecutive slots of one position: a pair inside the tile
        slot_seqs += [a, b]
    P = len(slot_seqs)
    assert P <= TILE
    c = np.zeros((S, 2, P, 4), np.uint32)
    for p, seq in enumerate(slot_seqs):
        for s, kind in enumerate(seq):
            c[s, 0, p], c[s, 1, p] = _rec(kind, rng)
    _, dense = np.unique(np.array(pos), return_inverse=True)
    return c, dense.astype(np.int32), slot_seqs


@pytest.mark.parametrize("S", [13, 14, 15, 16])
def test_pattern_reelection(ctx, S):
    """Item 8 (and 9): record orders that drive pat_irregular through each branch -- the takeover inside the first stage
    followed by "regular after all" (G R R R), the tie cnt0 == irr (G G R R), uncovered and absent records first, three
    patterns alternating, repeated takeovers, S mod 4 = 1, 2, 3, 0 -- and in-tile twin pairs whose two slots elect
    different patterns (PairBaseXfer merge).  A restatement of the pat / cnt0 / irr state machine shows every branch is
    taken.  Every NC form runs: noise kernels 7 and 8 (NC = 1, interleaved / not), the sweep with n_c 1 ... 8 under the
    default and kernel 8 (NC = 3, 5 interleaved and not, 8); every table equals the oracle's."""
    counts, pos_id, seqs = _pattern_normals(S, seed=500 + S)
    tot = {"regular": 0, "takeover": 0, "spill": 0}
    for q in seqs:
        for k, v in pattern_branches(q).items():
            tot[k] += v
    assert min(tot.values()) >= 3, tot
    assert pattern_branches("G" + "R" * (S - 1)) == {"regular": 1, "takeover": 1, "spill": 1}
    U = int(pos_id.max()) + 1
    cache = {}

    def want(cv):
        if cv not in cache:
            cache[cv] = oracle_noise(counts, pos_id, U, np.float32(cv), CUT)
        return cache[cv]
    _run_noise_everywhere(ctx, counts, pos_id, want, FOLD_C, [7, 8], [-1, 8], range(1, 9), [])
