"""The forward-first caller (call_forward_kernel, call kernel 13 and the default) against the straightforward caller (call
kernel 0, no screens) and the both-strand staged caller it replaced (call kernel 15): call lists byte for byte, sorted by
(sample, slot, alt).

call_forward_kernel streams the forward strand only and fetches a record's reverse-strand word asynchronously when the
forward strand can still make a call; the reverse strand then decides.  Each test shows that the path it targets ran,
with a host model of the forward screen (the records whose reverse word the kernel fetches).
"""
import numpy as np
import pytest

from tests.test_gpu_sweep_paths import _eff, mcrit, prescreen_k

pytestmark = pytest.mark.gpu

CUT = 100
ABSENT = 0xFFFFFFFF
STAGE_SAMPLES = 6      # samples per ring stage of call_forward_kernel<6, 2, 2>
RING = 32              # AS_FWD_PENDING: pending entries per warp


def forward_fetches(tumours, ref, thr, cut=CUT):
    """[T][P] bool: present, FW >= cut and, for some callable base (alt != ref, no -1 threshold on either strand),
    k > prescreen_k(FW, floor(e_b * 2^32)) on the forward strand."""
    fw = tumours[:, 0].astype(np.uint64)
    FW = fw.sum(-1) & np.uint64(0xFFFFFFFF)
    e = _eff(thr[..., 0]).astype(np.float64)
    R = np.where((e > 0) & (e < 1), np.floor(e * 2.0 ** 32), 0).astype(np.uint64)                # [P][4]
    ref = np.asarray(ref)
    callable_ = (np.arange(4)[None, :] != ref[:, None]) & (ref[:, None] <= 3) & (thr[..., 0] != -1) & (thr[..., 1] != -1)
    per = (fw > prescreen_k(FW[..., None], R[None])) & callable_[None]
    return (tumours[:, 0, :, 0] < 0x80000000) & (FW >= cut) & per.any(-1)


def host_calls(ctx, variant, tumours, ref, thr, tile_slots=0, pending_cap=0):
    ctx.set_call_kernel(variant)
    ctx.set_host_tile_slots(tile_slots)
    ctx.set_option("forward_pending_cap", pending_cap)
    try:
        return ctx.call_variants(tumours, ref, thr, CUT)
    finally:
        ctx.set_call_kernel(-1)
        ctx.set_host_tile_slots(0)
        ctx.set_option("forward_pending_cap", 0)


def dev_calls(ctx, variant, d_tum, d_ref, view, slot_ranges=None):
    import torch
    from amplisolve_b200 import CALL_DTYPE, calls_from_device
    T, _, P, _ = d_tum.shape
    calls = torch.empty(max(1 << 16, T * P // 50) * CALL_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    n = torch.zeros(1, dtype=torch.int64, device="cuda")
    ctx.set_call_kernel(variant)
    try:
        for r in slot_ranges or [None]:
            ctx.call_variants_dev(d_tum, d_ref, view, CUT, calls, n, slot_range=r)
        return calls_from_device(calls, n)
    finally:
        ctx.set_call_kernel(-1)


def assert_same(lists):
    first = lists[0]
    for other in lists[1:]:
        assert len(other) == len(first)
        assert other.tobytes() == first.tobytes()
    return first


def _generated(ctx, P, S, T, depth, seed, somatic_rate, vaf):
    gen = dict(seed=seed, mean_depth=depth, twin_period=6)
    normals, ref = ctx.synth_counts_dev(S, P, **gen)
    tumours, _ = ctx.synth_counts_dev(T, P, somatic_rate=somatic_rate, vaf=vaf, sample_offset=1 << 20, want_ref=False, **gen)
    nxt, head = ctx.synth_twin_links_dev(P, seed=seed, twin_period=6)
    out = ctx.alloc_noise_outputs(P)
    ctx.estimate_thresholds_dev(normals, 0.002, CUT, out, nxt, head)
    return tumours, ref, ctx.thresholds_caller_view_dev(out["thr"])


@pytest.mark.parametrize("shape", ["c3", "c4"])
def test_generator_statistics(ctx, shape):
    """The HBM generator at the statistics of bench.py's c3 workload (2000x) and of configs[4] (50,000x, spiked SNVs at
    0.5-1 %), on 300 k / 20 k slots; tumour counts that are no multiple of the ring stage."""
    from scripts.forward_first_stats import rates
    if shape == "c3":
        args = dict(P=300_000, S=40, T=41, depth=2000.0, seed=20183, somatic_rate=2e-4, vaf=(0.01, 0.2))
    else:
        args = dict(P=20_000, S=40, T=403, depth=50000.0, seed=20185, somatic_rate=5e-4, vaf=(0.005, 0.01))
    tumours, ref, view = _generated(ctx, **args)
    r = rates(tumours, ref, view)
    assert 0 < r["fw_per_base"] <= r["fw_min_R"]          # reverse words were fetched
    got = assert_same([dev_calls(ctx, v, tumours, ref, view) for v in (0, 15, 13)])
    assert len(got) > 100


def _veto_panel(seed=5):
    """Slots in groups of eight kinds; the forward strand of alt C passes comfortably in every record, the reverse strand
    decides:  0 passes (a call)  1 BW < cut  2 reverse k = 0  3 reverse k within the integer pre-screen bound
    4 reverse mean just above the critical mean m*(k) (only the exact screen rejects)  5 reverse threshold -1
    6 forward threshold -1  7 forward strand absent.  Plus a reverse threshold of 0 (effective 0.0010008) in half the
    slots of kind 0."""
    rng = np.random.default_rng(seed)
    P, T = 8 * 25, 7                                       # P is no multiple of the 128-slot tile
    kind = np.arange(P) % 8
    ref = np.zeros(P, np.uint8)
    thr = np.full((P, 4, 2), 3e-4, np.float32)
    t = np.zeros((T, 2, P, 4), np.uint64)
    FW = rng.integers(1000, 3000, (T, P))
    t[:, 0, :, 1] = rng.integers(8, 20, (T, P))            # m = FW * 3e-4 < 1: k >= 8 is a call on the forward strand
    BW = rng.integers(1000, 3000, (T, P))
    kb = rng.integers(8, 20, (T, P))
    e4 = np.float32(2.0 ** -20)
    m4 = mcrit()[1] / (1 + 1e-9) * 1.05                    # k = 2: mean 5 % above m*(2), prescreen_k = 1
    for s in range(P):
        k = kind[s]
        if k == 1:
            BW[:, s] = rng.integers(20, CUT, T)
            kb[:, s] = 5
        elif k == 2:
            kb[:, s] = 0
        elif k == 3:
            thr[s, 1, 1] = 0.01                            # m = BW / 100 >= 10: k <= m is dropped by the pre-screen
            kb[:, s] = BW[:, s] // 200
        elif k == 4:
            thr[s, 1, 1] = e4
            BW[:, s] = int(np.rint(m4 * 2.0 ** 20))
            kb[:, s] = 2
        elif k == 5:
            thr[s, 1, 1] = -1.0
        elif k == 6:
            thr[s, 1, 0] = -1.0
        elif k == 0 and s % 16 == 0:
            thr[s, 1, 1] = 0.0
    t[:, 1, :, 1] = kb
    t[:, 0, :, 0] = FW - t[:, 0, :, 1]
    t[:, 1, :, 0] = BW - kb
    t = t.astype(np.uint32)
    t[:, 0, kind == 7, :] = ABSENT
    return t, ref, thr, kind


def test_reverse_strand_decides(ctx):
    tumours, ref, thr, kind = _veto_panel()
    cands = forward_fetches(tumours, ref, thr)
    # the reverse word was fetched for every kind the reverse strand has to reject, never for kinds 5-7
    assert cands[:, np.isin(kind, [0, 1, 2, 3, 4])].all() and not cands[:, np.isin(kind, [5, 6, 7])].any()
    got = assert_same([host_calls(ctx, v, tumours, ref, thr) for v in (0, 15, 13)])
    called = np.zeros(tumours.shape[2], bool)
    called[got["slot"]] = True
    assert called[kind == 0].all() and not called[kind != 0].any()
    assert (thr[got["slot"], 1, 1] == 0).any()


@pytest.mark.parametrize("pending_cap", [1, 2, 0])
def test_every_record_a_candidate(ctx, pending_cap):
    """Every record passes the forward screen (tiny thresholds, alt reads on every base): a warp has 192 candidate records
    per stage, more than its pending ring holds, so the ring is drained on the spot -- at the full ring and capped at 1
    and 2 entries.  The reverse strand carries zero and non-zero alt reads (calls and vetoes)."""
    rng = np.random.default_rng(31 + pending_cap)
    P, T = 300, 37
    ref = rng.integers(0, 4, P).astype(np.uint8)
    thr = np.full((P, 4, 2), 1e-6, np.float32)
    t = rng.integers(1, 6, (T, 2, P, 4)).astype(np.uint32)
    t[:, 1] = np.where(rng.random((T, P, 4)) < 0.4, 0, t[:, 1])
    t[:, :, np.arange(P), ref] = rng.integers(500, 900, (T, 2, P))
    cands = forward_fetches(t, ref, thr)
    assert cands.all()
    per_warp_stage = STAGE_SAMPLES * 32
    assert per_warp_stage > (pending_cap or RING)
    got = assert_same([host_calls(ctx, v, t, ref, thr, pending_cap=pending_cap) for v in (0, 15, 13)])
    assert 0 < len(got) < 3 * T * P


def test_tiles_chunks_and_slot_ranges(ctx):
    """Partial tiles (P = 1000), grid.y > 1 (101 tumours over 8 tiles: seven chunks, the last one a partial stage), slot
    ranges that do not start on a tile boundary on the device path, and 256-slot upload tiles on the host path."""
    tumours, ref, view = _generated(ctx, P=1000, S=20, T=101, depth=2000.0, seed=20191, somatic_rate=0.02, vaf=(0.01, 0.2))
    want = dev_calls(ctx, 0, tumours, ref, view)
    assert len(want) > 100
    for v in (15, 13):
        assert_same([want, dev_calls(ctx, v, tumours, ref, view, slot_ranges=[(0, 37), (37, 611), (611, 1000)])])
    h_t = tumours.cpu().numpy().view(np.uint32)
    h_ref, h_view = ref.cpu().numpy(), view.cpu().numpy()
    assert_same([want] + [host_calls(ctx, v, h_t, h_ref, h_view, tile_slots=256) for v in (15, 13)])


def test_counts_beyond_2_24(ctx):
    """Strand depths from 2^24 to 2^29 (2^28 and more saturate the pre-screen's 16 x depth), alt reads around the mean and
    well above it."""
    rng = np.random.default_rng(9)
    P, T = 260, 9
    ref = rng.integers(0, 4, P).astype(np.uint8)
    thr = rng.choice(np.array([1e-4, 3e-4, 1e-3, 0.0], np.float32), (P, 4, 2))
    depth = rng.choice([1 << 24, 3 << 24, 1 << 27, 5 << 26, 1 << 29], (T, 2, P)).astype(np.float64)
    e = _eff(thr).astype(np.float64)
    t = np.zeros((T, 2, P, 4), np.uint64)
    for st in (0, 1):
        m = depth[:, st, :, None] * e[None, :, :, st]
        t[:, st] = np.floor(m * rng.choice([0.9, 1.0, 1.0005, 1.01, 1.5], (T, P, 4))).astype(np.uint64)
        t[:, st, np.arange(P), ref] = 0
        t[:, st, np.arange(P), ref] = depth[:, st].astype(np.uint64) - t[:, st].sum(-1)
    t = t.astype(np.uint32)
    cands = forward_fetches(t, ref, thr)
    FW = t[:, 0].astype(np.uint64).sum(-1)
    assert cands[FW >= 1 << 28].any() and cands[FW < 1 << 28].any()
    got = assert_same([host_calls(ctx, v, t, ref, thr) for v in (0, 15, 13)])
    assert len(got) > 50
