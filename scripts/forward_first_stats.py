"""Candidate rates and timing of the forward-first caller (call_forward_kernel, call kernel 13) against the both-strand
caller it replaced (call_staged_kernel<3,2,PRE>, call kernel 15), on the c3 and c4 workloads of bench.py.

    python scripts/forward_first_stats.py [--reps 5] [--variants 15,13] [--out FILE.json]

The tensors are built exactly as bench.py builds them (synth_counts_dev, the noise model, thresholds_caller_view_dev).  The
rates are plain tensor arithmetic on the device (__umulhi restated in int64), per record (tumour, slot):
  fw_min_R     forward strand only: present, FW >= cut, k > prescreen_k(FW, R_min) for some callable base
               (call_forward_kernel's scan)
  fw_per_base  the same with each base's own bound R_b (the records whose reverse word call_forward_kernel fetches)
  both_strand  call_staged_kernel's scan: present, min(FW, BW) >= cut, per base k > prescreen_k on both strands, R the
               smallest threshold of the strand
Bytes requested per record: 16 for the forward word, plus 16 per fetched reverse word (a 32-byte DRAM sector), against 32
for the both-strand kernel.  Timing: CUDA events around each caller variant, the variants alternating, `reps` rounds; the
sorted call lists of every variant must be equal.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

CUT = 100
WORKLOADS = {
    "c3": dict(P=2_000_000, S=100, T=500, seed=20183, depth=2000.0, somatic_rate=2e-4, vaf=(0.01, 0.2)),
    "c4": dict(P=100_000, S=100, T=10_000, seed=20185, depth=50000.0, somatic_rate=5e-4, vaf=(0.005, 0.01)),
}


def prescreen_k(depth, R):
    """as_call.cuh prescreen_k on int64 tensors (depth, R < 2^32)."""
    import torch
    d16 = torch.where(depth > 0x0FFFFFFF, torch.full_like(depth, 0xFFFFFFFF), depth << 4)
    m16 = (d16 * R) >> 32
    return (m16 + torch.where(m16 <= 1030, 9, 0)) >> 4


def bounds(view, ref):
    """Per slot: R_b [P][4][2] (0 = no screen), the callable-base mask [P][4] (alt != ref, no -1 on either strand) and
    the both-strand kernel's R_min per strand [P][2] (ref excluded, -1 puts no bound)."""
    import torch
    e = torch.where(view == 0, torch.tensor(0.0010008, dtype=torch.float32, device=view.device), view)
    R = torch.where((e > 0) & (e < 1), torch.floor(e.double() * 2.0 ** 32), torch.zeros_like(e, dtype=torch.float64)).long()
    not_ref = (torch.arange(4, device=view.device)[None, :] != ref[:, None].long()) & (ref[:, None] <= 3)
    callable_ = not_ref & (view[..., 0] != -1) & (view[..., 1] != -1)
    big = torch.full_like(R, 0xFFFFFFFF)
    R_old = torch.where(not_ref[..., None] & (view != -1), R, big).amin(dim=1) * (ref[:, None] <= 3)   # [P][2]
    return R, callable_, R_old


def rates(tumours, ref, view, block=10):
    import torch
    T = tumours.shape[0]
    R, callable_, R_old = bounds(view, ref)
    Rmin = torch.where(callable_, R[..., 0], torch.full_like(R[..., 0], 0xFFFFFFFF)).amin(dim=1)
    n = {"fw_min_R": 0, "fw_per_base": 0, "both_strand": 0}
    for s0 in range(0, T, block):
        c = tumours[s0:s0 + block].long() & 0xFFFFFFFF                                      # [t][2][P][4]
        fw, bw = c[:, 0], c[:, 1]
        FW, BW = fw.sum(-1) & 0xFFFFFFFF, bw.sum(-1) & 0xFFFFFFFF
        present = fw[..., 0] < 0x80000000
        ok = present & (FW >= CUT)
        kmax = torch.where(callable_[None], fw, torch.zeros_like(fw)).amax(-1)
        n["fw_min_R"] += int((ok & (kmax > prescreen_k(FW, Rmin[None]))).sum())
        per = (fw > prescreen_k(FW[..., None], R[None, ..., 0])) & callable_[None]
        n["fw_per_base"] += int((ok & per.any(-1)).sum())
        both = ((fw > prescreen_k(FW, R_old[None, :, 0])[..., None]) & (bw > prescreen_k(BW, R_old[None, :, 1])[..., None])
                & (torch.arange(4, device=c.device)[None, None, :] != ref[None, :, None].long()) & (ref[None, :, None] <= 3))
        n["both_strand"] += int((present & (torch.minimum(FW, BW) >= CUT) & both.any(-1)).sum())
    records = T * tumours.shape[2]
    out = {k: v / records for k, v in n.items()}
    out["bytes_per_record_forward"] = 16 + 32 * out["fw_per_base"]
    out["bytes_per_record_both_strand"] = 32
    return out


def build(ctx, wl):
    import torch
    gen = dict(seed=wl["seed"], mean_depth=wl["depth"], twin_period=6)
    normals, ref = ctx.synth_counts_dev(wl["S"], wl["P"], **gen)
    tumours, _ = ctx.synth_counts_dev(wl["T"], wl["P"], somatic_rate=wl["somatic_rate"], vaf=wl["vaf"], sample_offset=1 << 20,
                                      want_ref=False, **gen)
    nxt, head = ctx.synth_twin_links_dev(wl["P"], seed=wl["seed"], twin_period=6)
    out = ctx.alloc_noise_outputs(wl["P"])
    ctx.estimate_thresholds_dev(normals, 0.002, CUT, out, nxt, head)
    view = ctx.thresholds_caller_view_dev(out["thr"])
    del normals
    torch.cuda.synchronize()
    return tumours, ref, view


def main():
    import torch
    from amplisolve_b200 import CALL_DTYPE, Context, calls_from_device
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--variants", default="15,13")
    ap.add_argument("--workloads", default="c3,c4")
    ap.add_argument("--out")
    args = ap.parse_args()
    variants = [int(v) for v in args.variants.split(",")]
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": smi, "variants": variants, "reps": args.reps}
    ctx = Context(0)
    for name in args.workloads.split(","):
        wl = WORKLOADS[name]
        tumours, ref, view = build(ctx, wl)
        r = {"rates": rates(tumours, ref, view)}
        cap = max(1 << 16, int(wl["T"] * wl["P"] * 0.004))
        calls = torch.empty(cap * CALL_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        n = torch.zeros(1, dtype=torch.int64, device="cuda")
        times = {v: [] for v in variants}
        lists = {}
        for v in variants:   # warm-up, and the call list of each variant
            ctx.set_call_kernel(v)
            for _ in range(2):
                n.zero_()
                ctx.call_variants_dev(tumours, ref, view, CUT, calls, n)
            lists[v] = calls_from_device(calls, n)
        for _ in range(args.reps):
            for v in variants:
                ctx.set_call_kernel(v)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(5):
                    n.zero_()
                    ctx.call_variants_dev(tumours, ref, view, CUT, calls, n)
                b.record()
                torch.cuda.synchronize()
                times[v].append(a.elapsed_time(b) / 5)
        ctx.set_call_kernel(-1)
        first = lists[variants[0]]
        r["calls"] = len(first)
        r["calls_equal"] = all(len(l) == len(first) and l.tobytes() == first.tobytes() for l in lists.values())
        r["caller_ms"] = {str(v): {"median": float(np.median(t)), "min": float(np.min(t)), "max": float(np.max(t))} for v, t in times.items()}
        r["records"] = wl["T"] * wl["P"]
        res[name] = r
        print(name, json.dumps(r), flush=True)
        del tumours, ref, view, calls
        torch.cuda.empty_cache()
    ctx.close()
    print(json.dumps(res))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
