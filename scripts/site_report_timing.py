#!/usr/bin/env python
"""Cost of the site report (sites= of AmpliSolveVariantCalling, as_site_tests_host*), in two parts.

    program : configs[1] size (synthetic ASEQ as scripts/c2_cli_parity.py writes it: ~41 k slots x 96 tumours at ~5000x, one
              noise table), AmpliSolveVariantCalling without and with sites= listing 1,000 SNVs, cold (a new process per run) and
              through the resident service, alternating over 3 repeats; every output but Site_Report.txt must be identical.
    entry   : as_site_tests_host alone at a configs[4]-like shape: 2,000 tumours x 100,000 slots at 50,000x (uint32 host tensor),
              1,000 sites, 5 tables; the host gather, the upload and site_test_kernel timed by CUDA events (AS_TIMING lines of
              the library), 5 calls after one warm-up.

Prints one JSON object with the GPU's name and power limit read in the same run.

    python scripts/site_report_timing.py [out.json]      (on a GPU box)
"""
import json
import os
import re
import shutil
import signal
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from scripts.c2_cli_parity import stage, start_service  # noqa: E402
from scripts.sweep_programs_timing import BIN, CUT, gpu_info, phases, run  # noqa: E402

REPEATS, N_SITES = 3, 1000


def site_lines(table_text, n):
    rows = [l.split("\t") for l in table_text.splitlines()[1:]]
    rows = [r for r in rows if r[2] in ("A", "C", "G", "T")]
    step = max(1, len(rows) // n)
    return [f"{r[0]}\t{r[1]}\t.\t{r[2]}\t{'ACGT'[('ACGT'.index(r[2]) + 1) % 4]}" for r in rows[::step][:n]]


def outputs(d):
    res = {}
    for p in sorted(Path(d).rglob("*")):
        if p.is_dir() or p.name == "Site_Report.txt":
            continue
        rel = "list" if p.name.endswith("_tumour_count_list_original.txt") else str(p.relative_to(d))
        text = p.read_text()
        res[rel] = "".join(l for l in text.splitlines(True) if not l.startswith("##fileDate")) if p.suffix == ".vcf" else text
    return res


def program_part(res):
    with tempfile.TemporaryDirectory(prefix="siterep_", dir="/tmp") as td:
        td = Path(td)
        res["staging"] = stage(td)
        run([BIN / "AmpliSolveErrorEstimation", "panel_design=panel.bed", "reference_genome=ref.fa", "germline_dir=N", "C_value=0.002",
             f"coverage_cutoff={CUT}", "default_error=0.01", "output_dir=o"], td)
        table = next((td / "o").glob("positionSpecificNoise_*.txt"))
        (td / "sites.vcf").write_text("\n".join(site_lines(table.read_text(), N_SITES)) + "\n")
        base = [BIN / "AmpliSolveVariantCalling", f"errorFile=o/{table.name}", "tumour_dir=T", None, f"coverage_cutoff={CUT}", "p_value=0.05"]
        sock_dir = tempfile.mkdtemp(prefix="as_sock_", dir="/tmp")
        sock = str(Path(sock_dir) / "as.sock")
        srv = start_service(sock)
        walls, last = {}, {}
        try:
            for rep in range(REPEATS):
                for mode, env in (("cold", {}), ("served", {"AS_SERVER": sock})):
                    arms = (("plain", []), ("sites", ["sites=sites.vcf"]))
                    for arm, extra in (arms if rep % 2 == 0 else arms[::-1]):
                        args = list(base)
                        args[3] = f"output_dir={mode}_{arm}_{rep}"
                        w, err = run(args + extra, td, env)
                        walls.setdefault(f"{mode}_{arm}_s", []).append(round(w, 3))
                        if mode == "cold":
                            last[arm] = phases(err)
            assert srv.poll() is None
        finally:
            srv.send_signal(signal.SIGTERM)
            srv.wait(timeout=30)
            shutil.rmtree(sock_dir, ignore_errors=True)
        res["program"] = {"sites": N_SITES, **walls, **{k[:-2] + "_min_s": min(v) for k, v in walls.items()}, "phases_last_cold_run_s": last}
        ref = outputs(td / "cold_plain_0")
        res["program"]["identical_outputs"] = all(outputs(td / f"{m}_{a}_{r}") == ref for m in ("cold", "served") for a in ("plain", "sites")
                                                  for r in range(REPEATS))
        rep_lines = (td / "cold_sites_0" / "Site_Report.txt").read_text().splitlines()[1:]
        res["program"]["report_rows"] = len(rep_lines)
        res["program"]["report_status"] = {s: sum(l.endswith("\t" + s) for l in rep_lines)
                                           for s in ("CALLED", "NOT_CALLED", "LOW_COVERAGE", "NO_DATA", "NOT_TESTABLE")}


def entry_part():
    """runs in a child process with AS_TIMING=1; prints the statuses as JSON"""
    import numpy as np
    import torch
    from amplisolve_b200 import api
    T, P, S, NC = 2000, 100_000, 100, 5
    with api.Context(0) as ctx:
        normals, ref = ctx.synth_counts_dev(S, P, seed=11, mean_depth=50_000, sample_offset=0)
        est = ctx.estimate_thresholds_sweep(normals.cpu().numpy().view(np.uint32), [0.001, 0.002, 0.003, 0.004, 0.005], CUT)
        del normals
        tumours, _ = ctx.synth_counts_dev(T, P, seed=11, mean_depth=50_000, somatic_rate=1e-3, sample_offset=S, want_ref=False)
        host = torch.empty(tumours.shape, dtype=torch.int32, pin_memory=True)
        host.copy_(tumours)
        del tumours
        torch.cuda.synchronize()
        counts = host.numpy().view(np.uint32)
        ref = ref.cpu().numpy()
        rng = np.random.default_rng(5)
        slot = np.sort(rng.choice(P, N_SITES, replace=False)).astype(np.int32)
        alt = ((ref[slot].astype(np.int32) + 1 + rng.integers(0, 3, N_SITES)) % 4).astype(np.int32)
        out = None
        for i in range(6):
            sys.stderr.write(f"AS_TIMING call {i}\n")
            sys.stderr.flush()
            out = ctx.site_tests(counts, ref, est["thr_view"][:NC], CUT, slot, alt)
        st = {int(s): int(n) for s, n in zip(*np.unique(out["status"], return_counts=True))}
        k0 = int(((out["alt_fw"] == 0) | (out["alt_bw"] == 0)).sum())
        print(json.dumps({"shape": {"tumours": T, "slots": P, "depth": 50_000, "sites": N_SITES, "tables": NC},
                          "entries": int(out.size), "status_counts": st, "entries_with_a_zero_alt_strand": k0}))


def entry_timing(res):
    env = dict(os.environ, AS_TIMING="1")
    t = time.perf_counter()
    r = subprocess.run([sys.executable, __file__, "--entry"], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    info = json.loads(r.stdout.strip().splitlines()[-1])
    calls = r.stderr.split("AS_TIMING call ")[2:]          # the first call is the warm-up
    per = {}
    for c in calls:
        for m in re.finditer(r"AS_TIMING capi\.(sites\.\S+) ([0-9.]+)", c):
            per.setdefault(m.group(1), []).append(float(m.group(2)))
    info["seconds"] = {k: {"min": min(v), "max": max(v)} for k, v in per.items()}
    info["child_wall_s"] = round(time.perf_counter() - t, 1)
    res["entry"] = info


def main(out_json=None):
    res = gpu_info()
    entry_timing(res)
    program_part(res)
    print(json.dumps(res, indent=1))
    if out_json:
        Path(out_json).parent.mkdir(parents=True, exist_ok=True)
        Path(out_json).write_text(json.dumps(res, indent=1) + "\n")
    assert res["program"]["identical_outputs"], "sites= changed another output"


if __name__ == "__main__":
    if sys.argv[1:] == ["--entry"]:
        entry_part()
    else:
        main(sys.argv[1] if len(sys.argv) > 1 else None)
