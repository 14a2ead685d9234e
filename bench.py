#!/usr/bin/env python
"""Benchmark of the AmpliSolve hot path on B200 (contract: see the task statement / DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (CUDA, one process per GPU)
    python bench.py --impl reference [--gpus N] ...                # the reference's CPU path on the host cores

A "step" is one pass of the hot path over one batch of synthetic input: the noise model over all normals
of the panel shard (as_noise_estimate_dev), the "%f" hand-over of the thresholds, and the Poisson caller
over all tumours (as_call_variants_dev).  Workload at every N: BASELINE.json configs[2] per GPU -- a
500-gene-panel-sized shard of 2,000,000 slots x 100 normals x 500 tumours at ~2000x (weak scaling: the
N-GPU job is N such shards = a slice of the exome-scale configs[3], position-sharded, no collective on
the data path).  Metric: Poisson strand tests per second (6 per (tumour, slot) record), whole job.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOAD = {"name": "c3: synthetic 500-gene panel shard per GPU", "slots": 2_000_000, "normals": 100, "tumours": 500,
            "depth": 2000.0, "C_value": 0.002, "coverage_cutoff": 100, "seed": 20183, "somatic_rate": 2e-4, "vaf": (0.01, 0.2),
            "twin_period": 6}
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md, used only when MEASURED_PEAKS.json is absent


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--slots", type=int, default=WORKLOAD["slots"], help="slots per GPU (default: the named workload)")
    ap.add_argument("--normals", type=int, default=WORKLOAD["normals"])
    ap.add_argument("--tumours", type=int, default=WORKLOAD["tumours"])
    ap.add_argument("--depth", type=float, default=WORKLOAD["depth"])
    ap.add_argument("--somatic-rate", type=float, default=WORKLOAD["somatic_rate"])
    ap.add_argument("--vaf", type=float, nargs=2, default=list(WORKLOAD["vaf"]))
    ap.add_argument("--twin-period", type=int, default=WORKLOAD["twin_period"], help="0 = no duplicated positions")
    ap.add_argument("--cuda-graph", action="store_true",
                    help="capture the device-resident step once and replay it (for small panels, where launches dominate)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the noise-floor sweep leg (C_value 0.001 .. 0.005, configs[3])")
    ap.add_argument("--no-config-legs", action="store_true",
                    help="skip the legs at configs[3]'s own dimensions (200 normals x 1000 tumours, sweep as the step) and at configs[4]'s "
                         "(100 k slots x 10,000 samples at 50,000x)")
    ap.add_argument("--no-e2e-text", action="store_true", help="skip the program-against-program leg (text in, text out)")
    ap.add_argument("--no-pileup-leg", action="store_true", help="skip the computeCounts leg (BAM -> PILEUP.ASEQ, SURVEY 8 f4)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--e2e-format", choices=["packed", "16", "32"], default="packed",
                    help="host layout of the e2e leg: the packed wire format (8 B/record), the 16-bit one (16 B) or uint32 (32 B)")
    ap.add_argument("--e2e-wide", action="store_true", help="same as --e2e-format 32")
    ap.add_argument("--call-kernel", type=int, default=13, help="include/amplisolve_b200.h as_set_call_kernel")
    ap.add_argument("--noise-kernel", type=int, default=1, help="include/amplisolve_b200.h as_set_noise_kernel")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (float32 / float64, a "
                         "seeded sample of the slots, at most 64 MB) for comparing two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA step's outputs: it does not apply to --impl reference")
    return args


# ------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's own programs (oracle/_ref) on the host cores
# ------------------------------------------------------------------------------------------------------
def _write_aseq(path, chrom, pos, counts_s):
    """counts_s uint32 [2][P][4] of one sample -> .PILEUP.ASEQ text (SURVEY.md C.2); absent rows skipped."""
    present = counts_s[0, :, 0] != 0xFFFFFFFF
    fw = counts_s[0, present].astype(np.int64)
    bw = counts_s[1, present].astype(np.int64)
    tot = fw + bw
    rd = tot.sum(axis=1)
    cols = np.column_stack([tot, rd, bw])
    lines = ["chr\tpos\tdbsnp\tMAF\tref\talt\tA\tC\tG\tT\tRD\tArs\tCrs\tGrs\tTrs"]
    ch = np.asarray(chrom)[present]
    po = np.asarray(pos)[present]
    for i in range(cols.shape[0]):
        lines.append(f"{ch[i]}\t{po[i]}\t.\t.\t.\t.\t" + "\t".join(map(str, cols[i])))
    Path(path).write_text("\n".join(lines) + "\n")
    return int(present.sum())


def make_reference_sample(workdir, n_slots, n_normals, n_tumours, depth, seed):
    """A bounded sample of the bench workload as the text inputs the reference reads."""
    from tests import synth
    workdir = Path(workdir)
    n_amp = max(1, n_slots // 125)
    bed, slots, pos_id, U = synth.make_panel(n_amp, amp_len=(125, 125), overlap_frac=0.17, seed=seed, chroms=("chr1",))
    P = len(slots)
    normals, ref = synth.make_counts(n_normals, P, depth=depth, seed=seed, pos_id=pos_id, absent_rate=0.0,
                                     low_cov_rate=0.0, edge_rate=0.0)
    tumours, _ = synth.make_counts(n_tumours, P, depth=depth, seed=seed + 1, ref=ref, pos_id=pos_id,
                                   somatic_rate=2e-4, absent_rate=0.0, low_cov_rate=0.0, edge_rate=0.0)
    chrom = [c for c, _ in slots]
    pos = [p for _, p in slots]
    (workdir / "N").mkdir()
    (workdir / "T").mkdir()
    with open(workdir / "panel.bed", "w") as fh:
        for i, (c, s, e) in enumerate(bed):
            fh.write(f"{c}\t{s}\t{e}\tAMP{i}\t.\tGENE\n")
    seen = {}
    with open(workdir / "rb_ref.txt", "w") as fh:
        for (c, p), r in zip(slots, ref):
            fh.write(f"{c}\t{p}\t{'ACGT'[r]}\n")
            seen[(c, p)] = seen.get((c, p), 0) + 1
    with open(workdir / "rb_dup.txt", "w") as fh:
        for (c, p), n in sorted(seen.items()):
            if n >= 2:
                fh.write(f"{c}\t{p}\n")
    rows_n = sum(_write_aseq(workdir / "N" / f"N{i}.PILEUP.ASEQ", chrom, pos, normals[i]) for i in range(n_normals))
    rows_t = sum(_write_aseq(workdir / "T" / f"T{i}.PILEUP.ASEQ", chrom, pos, tumours[i]) for i in range(n_tumours))
    return {"slots": P, "unique": U, "normal_rows": rows_n, "tumour_rows": rows_t, "normals": normals, "tumours": tumours,
            "ref": ref, "pos_id": pos_id}


def _ref_worker_cmds(workdir, out_tag):
    ref_dir = ROOT / "oracle" / "_ref"
    ee = [str(ref_dir / "ee_ref"), "panel.bed", "rb_ref.txt", "rb_dup.txt", "N", "0.002", "100", f"o{out_tag}",
          f"o{out_tag}/list.txt"]
    vc = [str(ref_dir / "AmpliSolveVariantCalling"), f"errorFile=o{out_tag}/positionSpecificNoise_0.0020.txt",
          "tumour_dir=T", f"output_dir=v{out_tag}", "coverage_cutoff=100", "p_value=0.05"]
    return ee, vc


def run_reference_pass(workdir, cores, kind, sample):
    """One pass of the reference's path on `cores` host cores (one single-threaded process per core, each
    over the same bounded sample).  Returns (wall seconds, noise seconds of the slowest worker)."""
    workdir = Path(workdir)
    if kind == "reference":
        t0 = time.perf_counter()
        procs = []
        for c in range(cores):
            (workdir / f"o{c}").mkdir(exist_ok=True)
            (workdir / f"v{c}").mkdir(exist_ok=True)
            ee, vc = _ref_worker_cmds(workdir, c)
            script = " ".join(ee) + " >/dev/null 2>&1 && date +%s.%N && " + " ".join(vc) + " >/dev/null 2>&1"
            procs.append(subprocess.Popen(["bash", "-c", script], cwd=workdir, stdout=subprocess.PIPE, text=True))
        mids = []
        for p in procs:
            out, _ = p.communicate()
            if p.returncode != 0:
                raise RuntimeError("reference worker failed")
            mids.append(float(out.strip().splitlines()[-1]))
        wall = time.perf_counter() - t0
        t0_epoch = time.time() - wall
        return wall, max(mids) - t0_epoch
    # "port": the in-repo CPU restatement (oracle/liboracle.so), one process per core
    import multiprocessing as mp
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(cores) as pool:
        res = pool.map(_port_worker, [sample] * cores)
    return time.perf_counter() - t0, max(res)


def _port_worker(sample):
    from oracle import pyoracle
    from tests import synth
    t0 = time.perf_counter()
    rows, off = pyoracle.dense_to_rows(synth.to_oracle_layout(sample["normals"]), sample["pos_id"])
    nz = pyoracle.noise_estimate(rows, off, sample["unique"], np.float32(0.002), 100)
    t_noise = time.perf_counter() - t0
    thr = pyoracle.thr_as_caller_sees(np.where(np.isnan(nz["thr"]), np.float32(0.01), nz["thr"]))
    ref_u = np.zeros(sample["unique"], np.uint8)
    ref_u[sample["pos_id"]] = sample["ref"]
    rows, off = pyoracle.dense_to_rows(synth.to_oracle_layout(sample["tumours"]), sample["pos_id"])
    pyoracle.call_variants(rows, off, sample["unique"], ref_u, thr, 100)
    return t_noise


def cpu_reference(steps, warmup, sample_slots=1000, sample_normals=100, sample_tumours=500):
    """Times the reference CPU path on all host cores over a bounded sample; returns the JSON fragments."""
    cores = os.cpu_count() or 1
    have_ref = (ROOT / "oracle" / "_ref" / "ee_ref").exists() and (ROOT / "oracle" / "_ref" / "AmpliSolveVariantCalling").exists()
    kind = "reference" if have_ref and not os.environ.get("AS_BENCH_FORCE_PORT") else "port"
    with tempfile.TemporaryDirectory(prefix="asb_", dir="/tmp") as td:
        sample = make_reference_sample(td, sample_slots, sample_normals, sample_tumours, WORKLOAD["depth"], WORKLOAD["seed"])
        walls, noises = [], []
        for i in range(warmup + steps):
            w, nz = run_reference_pass(td, cores, kind, sample)
            if i >= warmup:
                walls.append(w)
                noises.append(nz)
    wall = float(np.mean(walls))
    tests = 6.0 * sample["tumour_rows"] * cores
    desc = (f"{sample['slots']} slots x {sample_normals} normals x {sample_tumours} tumours at ~{int(WORKLOAD['depth'])}x, "
            f"the same sample on each of {cores} cores (one single-threaded process per core); "
            + ("oracle/_ref: reference sources compiled -O2, text in / text out" if kind == "reference"
               else "oracle/liboracle.so port (reference binaries not present)"))
    return {"value": tests / wall, "unit": "Poisson tests/s", "cores": cores, "kind": kind, "sample": desc,
            "noise_positions_per_s": sample["slots"] * cores / float(np.mean(noises)), "ms_per_step": wall * 1e3}


# ------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampled every 20 ms from before the warm-up; the report uses the samples whose timestamps fall inside
    the timed region (mark_start / mark_end), or the nearest ones when the region is shorter than the sampling period."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t0, self.t1 = index, [], None, None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
            deadline = time.time() + 3.0
            while not self.rows and time.time() < deadline:   # nvidia-smi takes a few hundred ms to produce its first line
                time.sleep(0.02)
        except OSError:
            self.proc = None

    def _read(self):
        import datetime
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                ts = time.time()
            self.rows.append((ts, time.time(), f[1:]))

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        self.th.join(timeout=2)
        inside = [r for r in self.rows if self.t0 is not None and self.t0 <= r[1] <= self.t1 + 0.03]
        if len(inside) < 2 and self.rows:   # region shorter than the sampling period: take the samples closest to it
            mid = 0.5 * ((self.t0 or 0) + (self.t1 or 0))
            inside = sorted(self.rows, key=lambda r: abs(r[1] - mid))[:3]
        rows = [r[2] for r in inside]
        sm = [float(r[0]) for r in rows if len(r) >= 8 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) >= 8:
                for nm, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def hbm_peak():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel, default_workload, key=None):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch (or another recorded figure) from the committed ncu capture
    of this workload (profiles/ncu_traffic.json, written by scripts/ncu_summary.py --traffic)."""
    f = ROOT / "profiles" / "ncu_traffic.json"
    if not default_workload or not f.exists():
        return None
    try:
        k = json.loads(f.read_text())["kernels"][kernel]
        return k[key] if key else k["dram_bytes_read"] + k["dram_bytes_write"]
    except Exception:
        return None


def bind_to_gpu_numa_node(index):
    """Pin this rank's threads to the CPUs next to its GPU (NVML's ideal affinity) so that the pinned host tensors of the
    end-to-end leg are first-touched on the GPU's own NUMA node.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n = (os.cpu_count() + 63) // 64
        words = pynvml.nvmlDeviceGetCpuAffinity(h, n)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


DUMP_BYTES = 64_000_000   # the whole dump, .npy headers included


def dump_outputs(path, out, view, calls, n_calls):
    """Writes what the step returns to its caller as path/<name>.npy, so that two builds can be compared output for output:
      per slot, at a sample of the slots (slots.npy): the noise model's thr, germ_val, germ_state, count and nrec, and thr_view
      (the thresholds as the caller reads them);
      calls_<field>.npy: the calls at those slots in the reference's row order (sample, slot, alt); n_calls.npy: all calls.
    Every array is float32 or float64 (integers are exact in float64) and finite: a threshold the noise model leaves undefined
    (NaN, printed "-1_-1" in the noise table) is written as -1, which no defined threshold (a ratio of counts) can be.  The
    sample is a prefix of one seeded permutation of the slots, halved until the files, headers included, fit in 64 MB
    (64,000,000 bytes): the same inputs give the same slots."""
    import io

    import torch

    from amplisolve_b200 import CALL_DTYPE, calls_from_device
    path.mkdir(parents=True, exist_ok=True)
    per_slot = dict(out, thr_view=view)
    all_calls = calls_from_device(calls, n_calls)
    order = np.random.default_rng(WORKLOAD["seed"]).permutation(view.shape[0])
    n = min(len(order), 1 << 18)
    while True:
        slots = np.sort(order[:n])
        idx = torch.from_numpy(slots).to(view.device)
        arrays = {"slots": slots.astype(np.float64)}
        for name, t in per_slot.items():
            a = t[idx].cpu().numpy()
            if a.dtype == np.int32:   # uint32 counts held in int32 tensors
                a = a.view(np.uint32)
            arrays[name] = a.astype(np.float32 if a.dtype in (np.float32, np.uint8) else np.float64)
        picked = all_calls[np.isin(all_calls["slot"], slots)]
        for field in CALL_DTYPE.names:
            arrays[f"calls_{field}"] = picked[field].astype(np.float64)
        arrays["n_calls"] = np.array([len(all_calls)], np.float64)
        arrays["thr"][np.isnan(arrays["thr"])] = -1.0
        files = {}
        for name, a in arrays.items():
            buf = io.BytesIO()
            np.save(buf, a)
            files[name] = buf.getvalue()
        if sum(len(b) for b in files.values()) <= DUMP_BYTES or n == 1:
            break
        n //= 2
    bad = [name for name, a in arrays.items() if not np.isfinite(a).all()]
    if bad:
        raise RuntimeError(f"the step computed values that are not finite: {bad}")
    for name, b in files.items():
        (path / f"{name}.npy").write_bytes(b)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from amplisolve_b200 import CALL_DTYPE, Context

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL writes its version banner to stdout when the communicator comes up; rank 0's stdout must carry ONE JSON
        # line, so file descriptor 1 points at stderr until the first collective has run
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    numa_cpus = bind_to_gpu_numa_node(local) if world > 1 else None
    dev = torch.device(f"cuda:{local}")
    ctx = Context(local)
    ctx.set_call_kernel(args.call_kernel)
    ctx.set_noise_kernel(args.noise_kernel)
    P, S, T = args.slots, args.normals, args.tumours
    C, cut = WORKLOAD["C_value"], WORKLOAD["coverage_cutoff"]

    # synthetic inputs generated in HBM, untimed; rank r owns global slots [r*P, (r+1)*P)
    if P % 125 != 0:
        raise SystemExit("--slots must be a multiple of the 125-slot synthetic amplicon")
    gen = dict(seed=WORKLOAD["seed"], mean_depth=args.depth, slot_offset=rank * P, twin_period=args.twin_period)
    normals, ref = ctx.synth_counts_dev(S, P, **gen)
    tumours, _ = ctx.synth_counts_dev(T, P, somatic_rate=args.somatic_rate, vaf=tuple(args.vaf), sample_offset=1 << 20,
                                      want_ref=False, **gen)
    twin_next = twin_head = None
    if args.twin_period > 0:   # ~1.6 % of the slots are second enumerations of a position (overlapping amplicons)
        twin_next, twin_head = ctx.synth_twin_links_dev(P, seed=WORKLOAD["seed"], slot_offset=rank * P,
                                                        twin_period=args.twin_period)
    out = ctx.alloc_noise_outputs(P)
    view = torch.empty_like(out["thr"])
    cap = max(1 << 16, int(T * P * 0.004))
    calls = torch.empty(cap * CALL_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    n_calls = torch.zeros(1, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def step(marks=None):
        if marks is not None:
            marks[0].record()
        ctx.estimate_thresholds_dev(normals, C, cut, out, twin_next, twin_head)
        if marks is not None:
            marks[1].record()
        ctx.thresholds_caller_view_dev(out["thr"], view)
        n_calls.zero_()
        if marks is not None:
            marks[2].record()
        ctx.call_variants_dev(tumours, ref, view, cut, calls, n_calls)
        if marks is not None:
            marks[3].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    launches0 = ctx.kernel_launches
    marks = [[ev() for _ in range(4)] for _ in range(args.steps)]
    e0, e1 = ev(), ev()
    graph = None
    if args.cuda_graph:
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                step()
        torch.cuda.synchronize()
        graph.replay()
    barrier()
    sampler.mark_start()
    e0.record()
    for i in range(args.steps):
        if graph is not None:
            graph.replay()
        else:
            step(marks[i])
    e1.record()
    barrier()
    sampler.mark_end()
    if graph is not None:       # per-kernel times from one eager pass after the timed region
        for i in range(args.steps):
            step(marks[i])
        torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    total_ms = e0.elapsed_time(e1)
    launches = ctx.kernel_launches - launches0 + args.steps  # + the n_calls.zero_() fill kernel of each step
    t_noise = float(np.mean([m[0].elapsed_time(m[1]) for m in marks]))
    t_call = float(np.mean([m[2].elapsed_time(m[3]) for m in marks]))
    found = int(n_calls.item())
    if found > cap:
        raise RuntimeError(f"call list overflow in the benchmark: {found} > {cap}")
    if args.dump_outputs:   # before the legs below reuse out, view and calls
        dump_outputs(Path(args.dump_outputs) / (f"rank{rank}" if world > 1 else ""), out, view, calls, n_calls)

    # the only cross-GPU traffic of the job: one final gather of the compacted calls on rank 0 (outside the math path),
    # device to device: counts exchanged, exact-size NCCL sends into rank 0's buffer, one radix sort there
    gather_ms = None
    n_merged = found
    if world > 1:
        from amplisolve_b200.shard import gather_calls_device
        gather_calls_device(ctx, calls, found, rank * P)      # warm-up: communicator set-up and scratch are not the gather
        barrier()
        tg = time.perf_counter()
        merged, n_total = gather_calls_device(ctx, calls, found, rank * P)
        barrier()
        gather_ms = (time.perf_counter() - tg) * 1e3
        gm = torch.tensor([gather_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(gm, op=dist.ReduceOp.MAX)
        gather_ms = float(gm.item())
        if rank == 0:
            head = merged[: n_total * CALL_DTYPE.itemsize].view(-1, CALL_DTYPE.itemsize)[:, :12].contiguous().view(torch.int32).to(torch.int64)
            key = (head[:, 0] << 33) | (head[:, 1] << 2) | head[:, 2]
            if n_total < found or not bool((key[1:] > key[:-1]).all()):
                raise RuntimeError("gathered call list is not the sorted union of the ranks' lists")
            del head, key
        n_merged = n_total
        del merged
    tmax = torch.tensor([total_ms, t_noise, t_call], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms, t_noise_max, t_call_max = [float(x) for x in tmax.tolist()]

    # ---- noise-floor sweep of configs[3] (C_value 0.001 .. 0.005) on the same resident shard: one pass over the
    # tumours for all five threshold tables vs one caller pass per value (reported beside the headline, not part of it)
    sweep = None
    default_wl_sweep = (P, S, T, args.depth) == (WORKLOAD["slots"], WORKLOAD["normals"], WORKLOAD["tumours"], WORKLOAD["depth"])
    if not args.no_sweep and args.call_kernel >= 2:
        c_values = [0.001, 0.002, 0.003, 0.004, 0.005]
        views = torch.empty((len(c_values),) + tuple(view.shape), dtype=torch.float32, device=dev)
        s_calls = torch.empty(len(c_values) * cap * CALL_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        s_n = torch.zeros(len(c_values), dtype=torch.int64, device=dev)

        thr_tables = torch.empty_like(views)

        def sweep_noise_separate():
            for ci, cv in enumerate(c_values):
                ctx.estimate_thresholds_dev(normals, cv, cut, out, twin_next, twin_head)
                ctx.thresholds_caller_view_dev(out["thr"], views[ci])

        def sweep_noise():   # shared passes over the normals: the first value alone, the other four together
            ctx.estimate_thresholds_sweep_dev(normals, c_values, cut, thr_tables, out, twin_next, twin_head)
            ctx.thresholds_caller_view_dev(thr_tables, views)

        def sweep_fused():
            s_n.zero_()
            ctx.call_variants_sweep_dev(tumours, ref, views, cut, s_calls, s_n)

        def sweep_separate():
            for ci in range(len(c_values)):
                n_calls.zero_()
                ctx.call_variants_dev(tumours, ref, views[ci], cut, calls, n_calls)

        def timed(fn, reps=5):
            for _ in range(2):
                fn()
            a, b = ev(), ev()
            torch.cuda.synchronize()
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / reps

        t_sns = timed(sweep_noise_separate)
        views_separate = views.clone()
        t_sn = timed(sweep_noise)
        if not torch.equal(views.view(torch.int32), views_separate.view(torch.int32)):
            raise RuntimeError("the fused noise sweep and the per-value passes disagree")
        del views_separate
        t_sf = timed(sweep_fused)
        found_fused = [int(x) for x in s_n.tolist()]
        t_ss = timed(sweep_separate)
        tt = torch.tensor([t_sn, t_sf, t_ss, t_sns], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_sn, t_sf, t_ss, t_sns = [float(x) for x in tt.tolist()]
        peak_s, _ = hbm_peak()
        nb = P * (32 * S + 72 + 32 * (len(c_values) - 1))                                   # normals once, five tables out
        cb = T * P * 32 + P * 33 * len(c_values) + sum(found_fused) * CALL_DTYPE.itemsize    # tumours once, five tables in
        sweep = {"C_values": c_values, "noise_ms_fused": t_sn, "noise_ms_one_pass_per_value": t_sns,
                 "caller_ms_fused_one_pass": t_sf, "caller_ms_one_pass_per_value": t_ss, "calls_per_value_rank0": found_fused,
                 "tests_per_s_fused": 6.0 * T * P * world * len(c_values) / ((t_sn + t_sf) * 1e-3),
                 "tests_per_s_separate": 6.0 * T * P * world * len(c_values) / ((t_sns + t_ss) * 1e-3),
                 "roofline_sweep": {"bound": "hbm", "peak": peak_s, "unit": "GB/s",
                                    "caller": {"kernel": "call_scan_kernel + call_resolve_kernel + call_series_kernel",
                                               "algorithmic_bytes": cb, "achieved": cb / (t_sf * 1e-3) / 1e9, "frac": cb / (t_sf * 1e-3) / 1e9 / peak_s,
                                               "traffic": ncu_traffic("call_scan_kernel", default_wl_sweep)},
                                    "noise": {"kernel": "noise_pattern_kernel<5> (+ twin-group kernels on the side stream)",
                                              "algorithmic_bytes": nb, "achieved": nb / (t_sn * 1e-3) / 1e9, "frac": nb / (t_sn * 1e-3) / 1e9 / peak_s,
                                              "traffic": ncu_traffic("noise_pattern_kernel", default_wl_sweep)}},
                 "api": "as_noise_estimate_sweep_dev (ONE pass over the normals for the five values) + as_call_variants_sweep_dev (ONE "
                        "pass over the tumour tensor for the five threshold tables)"}
        del views, s_calls, thr_tables

    # ---- end to end through the host-buffer C ABI ----------------------------------------------------
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, ctx, normals, tumours, ref, twin_next, twin_head, rank, world, barrier)
        if e2e["slots_per_gpu"] == P and e2e["calls_per_step"] != found:   # same data through the host C ABI: same call set
            raise RuntimeError(f"e2e leg found {e2e['calls_per_step']} calls, the device-resident step {found}")

    # ---- legs at the dimensions of configs[3] and configs[4] (reported beside the headline; the resident c3 tensors go first)
    config_legs = None
    if not args.no_config_legs and args.call_kernel >= 2:
        del normals, tumours, calls
        torch.cuda.empty_cache()
        config_legs = run_config_legs(ctx, rank, world, dev)
        torch.cuda.empty_cache()
    e2e_text = None
    if not args.no_e2e_text:
        barrier()
        if rank == 0:
            try:
                e2e_text = run_e2e_text(world)
            except Exception as exc:   # a failure here (a full /tmp, a parity break) is reported on the line, loudly, not by losing the line
                import traceback
                traceback.print_exc()
                e2e_text = {"error": f"{type(exc).__name__}: {exc}"}
        barrier()

    pileup_leg = None
    if not args.no_pileup_leg and world == 1:
        try:   # computeCounts on one sample of configs[1], checked against a numpy pileup (scripts/pileup_bench.py)
            import contextlib
            import io
            from scripts import pileup_bench
            with contextlib.redirect_stdout(io.StringIO()):
                pileup_leg = pileup_bench.run()
            pileup_leg.pop("stdout", None)
        except Exception as exc:
            import traceback
            traceback.print_exc()
            pileup_leg = {"error": f"{type(exc).__name__}: {exc}"}

    result = None
    if rank == 0:
        ms_per_step = total_ms / args.steps
        tests_per_step = 6.0 * T * P * world
        peak, peak_src = hbm_peak()
        default_wl = (P, S, T, args.depth) == (WORKLOAD["slots"], WORKLOAD["normals"], WORKLOAD["tumours"], WORKLOAD["depth"])
        call_bytes = T * P * 32 + P * 33 + found * CALL_DTYPE.itemsize
        noise_bytes = P * (32 * S + 72)
        result = {
            "metric": "Poisson tests/sec", "value": tests_per_step / (ms_per_step * 1e-3), "unit": "Poisson tests/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 scan + f64 incomplete gamma",
            "data": "synthetic (seeded generator in HBM, SURVEY.md 8d)",
            "config": {"workload": WORKLOAD["name"] if default_wl else "custom", "slots_per_gpu": P,
                       "normals": S, "tumours": T, "depth": args.depth, "C_value": C, "coverage_cutoff": cut,
                       "duplicated_slots": "none" if twin_next is None else f"one amplicon junction in {args.twin_period} overlaps by 2-10 positions (~1.6 % of slots at 6)",
                       "somatic_rate": args.somatic_rate, "vaf": list(args.vaf),
                       "sharding": f"positions x{world}, no collective on the data path",
                       "cpu_affinity": None if numa_cpus is None else f"each rank bound to the {numa_cpus} CPUs next to its GPU (NVML)",
                       "l2": "inputs (6.4 GB normals + 32 GB tumours per step) far larger than the 126 MB L2",
                       "calls_per_step_rank0": found, "call_kernel_variant": args.call_kernel, "noise_kernel_variant": args.noise_kernel,
                       "launch_mode": "CUDA graph replay" if args.cuda_graph else "eager launches"},
            "noise_positions_per_s": P * world / (t_noise_max * 1e-3),
            "kernel_ms": {"noise_model": t_noise_max, "caller": t_call_max},
            "roofline": {"bound": "hbm", "kernel": {0: "call_naive_kernel", 1: "call_queued_kernel"}.get(args.call_kernel, "call_staged_kernel"),
                         "achieved": call_bytes / (t_call * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": call_bytes / (t_call * 1e-3) / 1e9 / peak,
                         "traffic": ncu_traffic("call_staged_kernel", default_wl and args.call_kernel == 13), "peak_source": peak_src,
                         "algorithmic_bytes": call_bytes,
                         "ncu_dram_pct_of_hw_peak": ncu_traffic("call_staged_kernel", default_wl and args.call_kernel == 13, "dram_pct_of_peak"),
                         "note": "peak is the driver's copy measurement (read + write); a read-only stream can exceed it, hence frac > 1 is "
                                 "possible -- ncu's own gpu__dram_throughput percentage of the hardware peak is given beside it"},
            "roofline_noise": {"bound": "hbm", "kernel": "noise_main_kernel" if args.noise_kernel == 0 else "noise_staged_kernel", "achieved": noise_bytes / (t_noise * 1e-3) / 1e9,
                               "peak": peak, "unit": "GB/s", "frac": noise_bytes / (t_noise * 1e-3) / 1e9 / peak,
                               "traffic": ncu_traffic("noise_staged_kernel", default_wl and args.noise_kernel == 1),
                               "ncu_dram_pct_of_hw_peak": ncu_traffic("noise_staged_kernel", default_wl and args.noise_kernel == 1, "dram_pct_of_peak"),
                               "algorithmic_bytes": noise_bytes},
            "gpu_launches": int(launches * world), "clocks": clocks,
        }
        if gather_ms is not None:
            result["calls_gather"] = {"ms": gather_ms, "calls_total": n_merged,
                                      "transport": "device to device: one 8-byte all_gather of the counts, exact-size NCCL sends of the compacted "
                                                   "lists into rank 0's buffer, as_sort_calls_dev there; once per job, no host copy"}
            result["job_ms"] = {"value": args.steps * ms_per_step + gather_ms,
                                "note": "steps x ms_per_step + the one gather of the calls (the job's only collective)"}
        if sweep is not None:
            result["noise_floor_sweep"] = sweep
        if config_legs is not None:
            result["config_legs"] = config_legs
        if e2e_text is not None:
            result["e2e_text"] = e2e_text
        if pileup_leg is not None:
            result["pileup"] = pileup_leg
        if e2e is not None:
            result["e2e"] = e2e
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_reference(steps=1, warmup=0)
            result["cpu_baseline"] = cb
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return result


def run_config_legs(ctx, rank, world, dev):
    """The step at the dimensions BASELINE.json's configs[3] and configs[4] name, per GPU, device-resident:
      configs[3]: 200 normals x 1000 tumours, the five-value noise-floor sweep AS THE STEP (one pass over the normals, one pass
                  over the tumours), on a 1,000,000-slot position shard (38.4 GB; the 40 M-slot panel is 40 such shards)
      configs[4]: 100,000 slots x 10,000 samples at 50,000x with 0.5-1 % spiked SNVs, caller throughput (recall against the
                  reference is tests/test_gpu_configs.py's job)"""
    import torch
    import torch.distributed as dist

    from amplisolve_b200 import CALL_DTYPE
    peak, _ = hbm_peak()
    cut = WORKLOAD["coverage_cutoff"]

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def timed(fn, reps=5):
        for _ in range(3):
            fn()
        a, b = ev(), ev()
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b) / reps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    legs = {}
    # ---- configs[3] dimensions
    P, S, T = 1_000_000, 200, 1000
    c_values = [0.001, 0.002, 0.003, 0.004, 0.005]
    gen = dict(seed=20184, mean_depth=2000.0, slot_offset=rank * P, twin_period=6)
    normals, ref = ctx.synth_counts_dev(S, P, **gen)
    tumours, _ = ctx.synth_counts_dev(T, P, somatic_rate=2e-4, sample_offset=1 << 20, want_ref=False, **gen)
    nxt, head = ctx.synth_twin_links_dev(P, seed=20184, slot_offset=rank * P, twin_period=6)
    out = ctx.alloc_noise_outputs(P)
    thr = torch.empty((len(c_values), P, 4, 2), dtype=torch.float32, device=dev)
    views = torch.empty_like(thr)
    cap = int(T * P * 0.004)
    calls = torch.empty(len(c_values) * cap * CALL_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    n_calls = torch.zeros(len(c_values), dtype=torch.int64, device=dev)

    def noise():
        ctx.estimate_thresholds_sweep_dev(normals, c_values, cut, thr, out, nxt, head)
        ctx.thresholds_caller_view_dev(thr, views)

    def caller():
        n_calls.zero_()
        ctx.call_variants_sweep_dev(tumours, ref, views, cut, calls, n_calls)

    def step():
        noise()
        caller()

    t_noise, t_call, t_step = timed(noise), timed(caller), timed(step)
    found = [int(x) for x in n_calls.tolist()]
    if max(found) > cap:
        raise RuntimeError("call list overflow in the configs[3] leg")
    nb = P * (32 * S + 72 + 32 * (len(c_values) - 1))
    cb = T * P * 32 + P * 33 * len(c_values) + sum(found) * CALL_DTYPE.itemsize
    legs["config3_sweep_step"] = {
        "workload": f"configs[3] dimensions per GPU: {P} slots x {S} normals x {T} tumours at ~2000x, C_value 0.001..0.005 as the step",
        "ms_per_step": t_step, "noise_ms": t_noise, "caller_ms": t_call, "calls_per_value_rank0": found,
        "tests_per_s": 6.0 * T * P * world * len(c_values) / (t_step * 1e-3),
        "noise_positions_per_s": P * world * len(c_values) / (t_noise * 1e-3),
        "roofline_noise": {"bound": "hbm", "algorithmic_bytes": nb, "achieved": nb / (t_noise * 1e-3) / 1e9, "peak": peak,
                           "frac": nb / (t_noise * 1e-3) / 1e9 / peak},
        "roofline_caller": {"bound": "hbm", "algorithmic_bytes": cb, "achieved": cb / (t_call * 1e-3) / 1e9, "peak": peak,
                            "frac": cb / (t_call * 1e-3) / 1e9 / peak}}
    del normals, tumours, thr, views, calls, out
    torch.cuda.empty_cache()
    # ---- configs[4] dimensions
    P, S, T = 100_000, 100, 10_000
    gen = dict(seed=20185, mean_depth=50000.0, slot_offset=rank * P, twin_period=6)
    normals, ref = ctx.synth_counts_dev(S, P, **gen)
    tumours, _ = ctx.synth_counts_dev(T, P, somatic_rate=5e-4, vaf=(0.005, 0.01), sample_offset=1 << 20, want_ref=False, **gen)
    nxt, head = ctx.synth_twin_links_dev(P, seed=20185, slot_offset=rank * P, twin_period=6)
    out = ctx.alloc_noise_outputs(P)
    ctx.estimate_thresholds_dev(normals, WORKLOAD["C_value"], cut, out, nxt, head)
    view = ctx.thresholds_caller_view_dev(out["thr"])
    cap = int(T * P * 0.004)
    calls = torch.empty(cap * CALL_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    n1 = torch.zeros(1, dtype=torch.int64, device=dev)

    def caller5():
        n1.zero_()
        ctx.call_variants_dev(tumours, ref, view, cut, calls, n1)

    t5 = timed(caller5)
    found5 = int(n1.item())
    if found5 > cap:
        raise RuntimeError("call list overflow in the configs[4] leg")
    cb = T * P * 32 + P * 33 + found5 * CALL_DTYPE.itemsize
    legs["config4_caller"] = {
        "workload": f"configs[4] dimensions per GPU: {P} slots x {T} samples at ~50,000x, 0.5-1 % spiked SNVs",
        "caller_ms": t5, "calls_rank0": found5, "tests_per_s": 6.0 * T * P * world / (t5 * 1e-3),
        "roofline_caller": {"bound": "hbm", "algorithmic_bytes": cb, "achieved": cb / (t5 * 1e-3) / 1e9, "peak": peak,
                            "frac": cb / (t5 * 1e-3) / 1e9 / peak},
        "recall": "tests/test_gpu_configs.py::test_config4_slice_call_set_and_recall_equal_the_reference"}
    del normals, tumours, calls
    return legs


def run_e2e_text(world):
    """Text in, text out, the same files for both arms: the two drop-in programs against the compiled reference programs
    (oracle/_ref).  configs[1] at full size and a 200,000-slot slice of the configs[2] panel.  With several GPUs the programs
    use all of them (AS_DEVICES) and their outputs are compared with the one-GPU run; the reference arm runs at N=1 only
    (it is single-threaded and takes the same time at every N)."""
    from oracle import refrun
    from scripts import c2_cli_parity as cli
    shapes = {"config1_full_size": dict(),
              "config2_slice": dict(n_amplicons=1600, n_normals=20, n_tumours=20, depth=2000, amp_len=(125, 125), seed=20183,
                                    chroms=tuple(f"chr{i}" for i in range(1, 23)) + ("chrX",), somatic_rate=2e-4)}
    res = {}
    for name, shape in shapes.items():
        with tempfile.TemporaryDirectory(prefix="e2et_", dir="/tmp") as td:
            info = cli.stage(td, **shape)
            cli.run_ours(td, out_ee="w", out_vc="wv", devices=[0])            # warm the page cache and the driver
            runs = [cli.run_ours(td, devices=list(range(world))) for _ in range(2)]
            walls = [r["error_estimation_wall_s"] + r["variant_calling_wall_s"] for r in runs]
            ours = runs[int(np.argmin(walls))]
            leg = {"shape": info, "ours": ours, "devices": world, "ours_wall_s": min(walls), "ours_wall_s_runs": walls,
                   "ours_wall_note": "best of two runs after one warm-up run: CUDA start-up on the box varies between 0.2 and 4 s per "
                                     "process (cuda_context_wait in the phases), the arithmetic and the text handling do not"}
            rows = info["normal_rows"] + info["tumour_rows"]
            leg["ours_rows_per_s"] = rows / leg["ours_wall_s"]
            # the same programs with a resident service holding the CUDA context (AS_SERVER; as_serve.cpp): what a site that
            # runs many panels a day deploys.  The service is started before the clock, like a database would be.
            sock = str(Path(td) / "as.sock")
            srv = cli.start_service(sock, devices=list(range(world)) if world > 1 else None)
            try:
                served = [cli.run_ours(td, out_ee="so", out_vc="sv", devices=list(range(world)), server=sock) for _ in range(2)]
            finally:
                srv.terminate()
                srv.wait(timeout=30)
            swalls = [r["error_estimation_wall_s"] + r["variant_calling_wall_s"] for r in served]
            leg["ours_served"] = dict(served[int(np.argmin(swalls))], wall_s=min(swalls), wall_s_runs=swalls,
                                      identical_to_own_process=all(v for k, v in cli.compare(td, "o", "v", "so", "sv").items() if k.endswith("identical")),
                                      note="AS_SERVER=<socket of amplisolve_b200_serve>: same programs, same files, the CUDA context is resident")
            if not leg["ours_served"]["identical_to_own_process"]:
                raise RuntimeError("the programs' outputs through the resident service differ")
            # what the two processes waited for the CUDA driver (cuInit + primary context, started on a thread at program
            # entry and overlapped with the parse): profiles/r02_cuda_startup.txt times the same for an empty CUDA process
            leg["ours_cuda_startup_wait_s"] = sum(ours[k].get("cuda_context_wait", 0.0) for k in ("ee_phases_s", "vc_phases_s"))
            leg["ours_wall_without_cuda_startup_s"] = leg["ours_wall_s"] - leg["ours_cuda_startup_wait_s"]
            if world > 1:
                leg["identical_to_one_gpu"] = all(v for k, v in cli.compare(td, "o", "v", "w", "wv").items() if k.endswith("identical"))
                if not leg["identical_to_one_gpu"]:
                    raise RuntimeError("the programs' outputs on several GPUs differ from the one-GPU run")
            elif refrun.have_ref():
                ref = cli.run_reference(td)
                par = cli.compare(td)
                if not (par["noise_table_identical"] and par["summary_identical"] and par["vcfs_identical"]):
                    raise RuntimeError("program outputs differ from the reference's")
                leg.update(reference=ref, parity=par,
                           reference_wall_s=ref["error_estimation_wall_s"] + ref["variant_calling_wall_s"])
                leg["reference_rows_per_s"] = rows / leg["reference_wall_s"]
                leg["speedup_wall"] = leg["reference_wall_s"] / leg["ours_wall_s"]
                leg["speedup_wall_served"] = leg["reference_wall_s"] / leg["ours_served"]["wall_s"]
            res[name] = leg
    res["note"] = ("same ASEQ / BED / FASTA files in, same noise table / summary / VCF files out (byte-identical); wall clock of the two "
                   "processes per arm; the reference arm is single-threaded and skips only its samtools fork loop (ee_ref fast driver)")
    return res


def run_e2e(args, ctx, d_normals, d_tumours, d_ref, d_twin_next, d_twin_head, rank, world, barrier):
    """Same step through as_noise_estimate_host / as_call_variants_host: inputs start in pinned HOST memory;
    H2D of all counts and D2H of the noise table and the calls are inside the timed region."""
    import ctypes as C

    import psutil
    import torch

    from amplisolve_b200 import CALL_DTYPE, lib
    P, S, T = args.slots, args.normals, args.tumours
    # keep the pinned footprint of all ranks below a third of the free host memory
    avail = psutil.virtual_memory().available / max(1, world) / 3
    Pe = P
    while (S + T) * Pe * 32 > avail and Pe > 50_000:
        Pe //= 2
    L = lib()

    def pinned(nbytes):
        p = C.c_void_p()
        rc = L.as_host_alloc(C.byref(p), nbytes)
        if rc != 0:
            raise RuntimeError(L.as_last_error().decode())
        return p

    # host tensors: the packed wire format of the _host_packed entry points (8 bytes per record; records that do not fit
    # escaped into a side list of wide records: lossless), the 16-bit wire format, or uint32
    fmt = "32" if args.e2e_wide else args.e2e_format
    narrow = fmt == "16"
    packed = fmt == "packed"
    word = {"packed": 4, "16": 8, "32": 16}[fmt]            # bytes per (sample, strand, slot)
    bn, bt = S * 2 * Pe * word, T * 2 * Pe * word
    hp_n, hp_t = pinned(bn), pinned(bt)
    ctype, ndt = (C.c_uint16, np.int16) if narrow else (C.c_uint32, np.int32)
    shp = (lambda n: (n, 2, Pe)) if packed else (lambda n: (n, 2, Pe, 4))
    h_norm = np.ctypeslib.as_array(C.cast(hp_n, C.POINTER(ctype)), shape=shp(S))
    h_tum = np.ctypeslib.as_array(C.cast(hp_t, C.POINTER(ctype)), shape=shp(T))
    from amplisolve_b200.api import WIDE_DTYPE
    others = torch.tensor([[1, 2, 3], [0, 2, 3], [0, 1, 3], [0, 1, 2]], device=d_normals.device)

    def pack_block(blk):
        """torch statement of the packed wire format (api.to_wire_packed) for one block of samples, on the device"""
        v = blk.to(torch.int64) & 0xFFFFFFFF
        m, j = v[..., 0], torch.zeros_like(v[..., 0])
        for b in (1, 2, 3):                                  # first maximum: ties go to the lowest base index
            gt = v[..., b] > m
            j = torch.where(gt, b, j)
            m = torch.where(gt, v[..., b], m)
        mi = torch.gather(v, -1, others[j])
        fits = (m <= 0xFFFF) & (mi <= 15).all(-1)
        w = m | (j << 16) | (mi[..., 0] << 18) | (mi[..., 1] << 22) | (mi[..., 2] << 26)
        absent = blk[:, 0, :, 0] == -1
        esc = ~absent & ~(fits[:, 0] & fits[:, 1])
        w = torch.where(esc[:, None, :], 0xFFFFFFFE, w)
        w = torch.where(absent[:, None, :], 0xFFFFFFFF, w)
        return w.to(torch.int32), esc                        # int64 -> int32 keeps the low 32 bits

    def to_host(dst_np, src):
        """untimed: bring a slot prefix of a device tensor to the pinned host tensor (and its wide records)"""
        dst = torch.from_numpy(dst_np.view(ndt))
        wides = []
        for s0 in range(0, src.shape[0], 20):      # in sample blocks: bounded temporaries on the device
            blk = src[s0:s0 + 20, :, :Pe, :]
            if fmt == "32":
                dst[s0:s0 + 20].copy_(blk)
                continue
            if packed:
                w32, esc = pack_block(blk)
                smp, slot = esc.nonzero(as_tuple=True)
                w = np.zeros(len(smp), dtype=WIDE_DTYPE)
                w["sample"], w["slot"] = (smp + s0).cpu().numpy(), slot.cpu().numpy()
                w["fw"], w["bw"] = blk[smp, 0, slot].cpu().numpy(), blk[smp, 1, slot].cpu().numpy()
                wides.append(w)
                dst[s0:s0 + 20].copy_(w32)
                del w32, esc
                continue
            present = blk[:, 0, :, 0] >= 0                                   # absent words are -1 as int32
            big = present & ((blk[:, 0] >= 0xFFFE).any(-1) | (blk[:, 1] >= 0xFFFE).any(-1))
            smp, slot = big.nonzero(as_tuple=True)
            w = np.zeros(len(smp), dtype=WIDE_DTYPE)
            w["sample"], w["slot"] = (smp + s0).cpu().numpy(), slot.cpu().numpy()
            w["fw"], w["bw"] = blk[smp, 0, slot].cpu().numpy(), blk[smp, 1, slot].cpu().numpy()
            wides.append(w)
            n16 = blk.to(torch.int16)
            n16[smp, :, slot, :] = -2                                        # 0xFFFE: escaped
            dst[s0:s0 + 20].copy_(n16)
        return np.sort(np.concatenate(wides), order=["slot", "sample"]) if wides else np.zeros(0, WIDE_DTYPE)

    def pinned_copy(w):
        """the side lists live in pinned memory like the count tensors (the C ABI accepts pageable lists too, slower)"""
        if len(w) == 0:
            return w, None
        hp = pinned(w.nbytes)
        dst = np.frombuffer((C.c_char * w.nbytes).from_address(hp.value), dtype=WIDE_DTYPE)
        dst[:] = w
        return dst, hp

    w_norm, hp_wn = pinned_copy(to_host(h_norm, d_normals))
    w_tum, hp_wt = pinned_copy(to_host(h_tum, d_tumours))
    h_ref = d_ref[:Pe].cpu().numpy()
    h_tn = h_th = None
    if d_twin_next is not None:
        h_tn, h_th = d_twin_next[:Pe].cpu().numpy().copy(), d_twin_head[:Pe].cpu().numpy().copy()
        h_tn[h_tn >= Pe] = -1     # a slot prefix of the shard: a pair cut by the prefix end becomes two singletons
    torch.cuda.synchronize()
    cut, Cv = WORKLOAD["coverage_cutoff"], WORKLOAD["C_value"]
    cap = max(1 << 16, int(T * Pe * 0.004))
    stats = {}

    def one():
        ta = time.perf_counter()
        noise = ctx.estimate_thresholds(h_norm, Cv, cut, h_tn, h_th, wide_records=w_norm, with_view=True, pinned_outputs=True)
        tb = time.perf_counter()
        calls = ctx.call_variants(h_tum, h_ref, noise["thr_view"], cut, cap=cap, wide_records=w_tum, pinned_outputs=True)
        stats["calls"] = len(calls)
        stats["noise_ms"], stats["call_ms"] = (tb - ta) * 1e3, (time.perf_counter() - tb) * 1e3

    # context for the e2e number: what a plain pinned host -> device copy achieves on this box
    hb = torch.empty(1 << 30, dtype=torch.uint8).pin_memory()
    db = torch.empty(1 << 30, dtype=torch.uint8, device=d_normals.device)
    db.copy_(hb, non_blocking=True)
    ec = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ec[0].record()
    for _ in range(3):
        db.copy_(hb, non_blocking=True)
    ec[1].record()
    torch.cuda.synchronize()
    pcie_gbs = 3 * (1 << 30) / (ec[0].elapsed_time(ec[1]) * 1e-3) / 1e9
    del hb, db

    one()  # warm-up (allocates the tile buffers)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        one()
    barrier()
    dt = (time.perf_counter() - t0) / args.e2e_steps
    import torch.distributed as dist
    if world > 1:
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
    n_esc = len(w_norm) + len(w_tum)
    del w_norm, w_tum
    for hp in (hp_n, hp_t, hp_wn, hp_wt):
        if hp is not None:
            L.as_host_free(hp)
    return {"value": 6.0 * T * Pe * world / dt, "unit": "Poisson tests/s", "ms_per_step": dt * 1e3,
            "h2d_bytes_per_step": int(bn + bt + Pe * 33 + 40 * n_esc), "d2h_bytes_per_step": int(Pe * 72 + Pe * 32 + stats["calls"] * 48),
            "slots_per_gpu": Pe, "calls_per_step": stats["calls"], "noise_call_ms": stats["noise_ms"], "caller_call_ms": stats["call_ms"], "pcie_h2d_gbs_measured": pcie_gbs,
            "h2d_gbs_achieved": (bn + bt) / dt / 1e9,
            "host_dtype": {"packed": f"packed wire format (8 B/record: 16-bit major + three 4-bit minor counts per strand) + {n_esc} escaped wide records ({n_esc / ((S + T) * Pe):.2e} of the records; lossless)",
                           "16": f"uint16 wire format + {n_esc} escaped wide records (lossless)", "32": "uint32"}[fmt],
            "api": {"packed": "as_noise_estimate_host_packed + as_call_variants_host_packed", "16": "as_noise_estimate_host16 + as_call_variants_host16",
                    "32": "as_noise_estimate_host + as_call_variants_host"}[fmt] + ", pinned host count tensors",
            "timer": "host wall clock around the blocking C-ABI calls, max over ranks"}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        if rank != 0:
            return
        cb = cpu_reference(steps=args.steps, warmup=min(args.warmup, 1))
        line = {"impl": "reference", "metric": "Poisson tests/sec", "value": cb["value"], "unit": "Poisson tests/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": cb["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i32 + f64/x87 (CPU)",
                "data": "synthetic (bounded sample of the bench workload, written as ASEQ text)",
                "config": {"workload": WORKLOAD["name"], "sample": cb["sample"]},
                "noise_positions_per_s": cb["noise_positions_per_s"],
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": cb["value"], "unit": "Poisson tests/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return
    res = run_ours(args)
    if res is not None:
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
