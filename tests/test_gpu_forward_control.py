"""Branches of the forward-first caller's control warps (call kernel 13) that tests/test_gpu_forward_first.py does not
reach: stages whose records pass the scan warps' single bound R_min in numbers larger than one 32-lane pass of the control
warp, while few or none of them survive the per-base bounds R_b.  Call lists byte for byte against call kernels 0 and 15.
"""
import numpy as np
import pytest

from tests.test_gpu_forward_first import CUT, assert_same, forward_fetches, host_calls
from tests.test_gpu_sweep_paths import _eff, prescreen_k

pytestmark = pytest.mark.gpu


def scan_passes(tumours, ref, thr, cut=CUT):
    """[T][P] bool: the scan warps' test -- present, FW >= cut and the largest forward alt count over the callable bases
    above prescreen_k(FW, R_min), R_min the smallest forward bound of those bases."""
    fw = tumours[:, 0].astype(np.uint64)
    FW = fw.sum(-1) & np.uint64(0xFFFFFFFF)
    e = _eff(thr[..., 0]).astype(np.float64)
    R = np.where((e > 0) & (e < 1), np.floor(e * 2.0 ** 32), 0).astype(np.uint64)
    callable_ = (np.arange(4)[None, :] != ref[:, None]) & (ref[:, None] <= 3) & (thr[..., 0] != -1) & (thr[..., 1] != -1)
    Rmin = np.where(callable_, R, np.uint64(0xFFFFFFFF)).min(-1)
    kmax = np.where(callable_[None], fw, 0).max(-1)
    return (tumours[:, 0, :, 0] < 0x80000000) & (FW >= cut) & (kmax > prescreen_k(FW, Rmin[None]))


def _passer_panel(P, T, call_every, seed):
    """Alt C carries 10 forward reads at a forward mean of about 20 (threshold 0.01): the R_min bound, set by alt G's tiny
    threshold, passes every record and the per-base bound of C rejects it.  Every call_every-th slot instead has alt C at
    a threshold of 1e-4 (mean 0.2): a candidate and, with 10 reverse reads, a call."""
    rng = np.random.default_rng(seed)
    ref = np.zeros(P, np.uint8)
    thr = np.full((P, 4, 2), 0.01, np.float32)
    thr[:, 2, :] = 1e-6                                    # alt G: no reads, smallest threshold
    callers = np.arange(P) % call_every == 0 if call_every else np.zeros(P, bool)
    thr[callers, 1, :] = 1e-4
    t = np.zeros((T, 2, P, 4), np.uint32)
    depth = rng.integers(1900, 2100, (T, 2, P))
    t[..., 1] = 10
    t[..., 0] = depth - 10
    return t, ref, thr, callers


@pytest.mark.parametrize("call_every", [0, 7])
def test_passers_beyond_one_lane_pass(ctx, call_every):
    """Every record passes the scan and 4 x 128 = 512 records of each stage go through the control warp's per-base test,
    16 passes of 32 lanes; call_every = 0: none of them becomes a candidate (no reverse fetch, no call), 7: a seventh of
    the slots do and are called."""
    P, T = 300, 23                                         # a partial tile and a partial last stage
    t, ref, thr, callers = _passer_panel(P, T, call_every, seed=41 + call_every)
    assert scan_passes(t, ref, thr).all()
    fetch = forward_fetches(t, ref, thr)
    assert (fetch == callers[None]).all()
    got = assert_same([host_calls(ctx, v, t, ref, thr) for v in (0, 15, 13)])
    if call_every:
        assert len(got) == T * callers.sum() and callers[got["slot"]].all()
    else:
        assert len(got) == 0
