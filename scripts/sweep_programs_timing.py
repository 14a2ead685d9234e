#!/usr/bin/env python
"""The noise-floor sweep through the two programs against one run per value, at the size of BASELINE.json configs[1]:
~41 k slots x 40 normals x 96 tumours at ~5000x, synthetic ASEQ as scripts/c2_cli_parity.py writes it, five values of C.

    sweep     : AmpliSolveErrorEstimation C_value=0.001,...,0.005, then AmpliSolveVariantCalling errorFile=<that directory>
    per value : five AmpliSolveErrorEstimation runs (one value each), then five AmpliSolveVariantCalling runs (one table each)

Both arms run cold (a new process and CUDA context per program run) and through the resident service (AS_SERVER), and
alternate over 3 repeats.  The outputs of the two arms must be byte-identical (VCFs minus ##fileDate).  Prints one JSON
object: wall time of every run of each arm, the AS_TIMING phases of the last cold runs, and the GPU's name and power limit.

    python scripts/sweep_programs_timing.py [out.json]        (on a GPU box; staging the ASEQ files takes a minute or two)
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

BIN = ROOT / "amplisolve_b200" / "bin"
C_VALUES = ["0.001", "0.002", "0.003", "0.004", "0.005"]
CUT, REPEATS = 100, 3


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        name, power = r.stdout.strip().splitlines()[0].split(", ")
        return {"gpu": name, "power_limit": power}
    except Exception as exc:  # noqa: BLE001
        return {"gpu": "unknown", "power_limit": f"not read: {exc}"}


def run(args, cwd, env=None):
    t = time.perf_counter()
    r = subprocess.run([str(a) for a in args], cwd=cwd, capture_output=True, text=True, env=dict(os.environ, AS_TIMING="1", **(env or {})))
    wall = time.perf_counter() - t
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "Error from" not in r.stdout and "Error:" not in r.stdout, r.stdout[-3000:]
    return wall, r.stderr


def phases(stderr):
    out = {}
    for m in re.finditer(r"AS_TIMING (\S+) ([0-9.]+)", stderr):
        out[m.group(1)] = round(out.get(m.group(1), 0.0) + float(m.group(2)), 6)
    return out


def ee(c_value, out):
    return [BIN / "AmpliSolveErrorEstimation", "panel_design=panel.bed", "reference_genome=ref.fa", "germline_dir=N", f"C_value={c_value}",
            f"coverage_cutoff={CUT}", "default_error=0.01", f"output_dir={out}"]


def vc(error_file, out):
    return [BIN / "AmpliSolveVariantCalling", f"errorFile={error_file}", "tumour_dir=T", f"output_dir={out}", f"coverage_cutoff={CUT}",
            "p_value=0.05"]


def table(c):
    return "positionSpecificNoise_%.4f.txt" % float(c)


def outputs(td, tables_dir, calls_dir_of):
    """noise tables and every caller output per value (VCFs minus ##fileDate, the tumour list whatever its seed prefix)"""
    res = {}
    for c in C_VALUES:
        res[table(c)] = (td / tables_dir / table(c)).read_text()
        d = td / calls_dir_of(c)
        for p in sorted(d.rglob("*")):
            if p.is_dir():
                continue
            rel = str(p.relative_to(d))
            if rel.endswith("_tumour_count_list_original.txt"):
                rel = "tumour_count_list"
            text = p.read_text()
            if p.suffix == ".vcf":
                text = "".join(l for l in text.splitlines(True) if not l.startswith("##fileDate"))
            res[f"{c}/{rel}"] = text
    return res


def arm_sweep(td, tag, env):
    w1, e1 = run(ee(",".join(C_VALUES), f"{tag}_o"), td, env)
    w2, e2 = run(vc(f"{tag}_o", f"{tag}_v"), td, env)
    return w1 + w2, {"error_estimation": phases(e1), "variant_calling": phases(e2)}


def arm_per_value(td, tag, env):
    wall, err_ee, err_vc = 0.0, "", ""
    for c in C_VALUES:
        w, e = run(ee(c, f"{tag}_o"), td, env)
        wall += w
        err_ee += e
    for c in C_VALUES:
        w, e = run(vc(f"{tag}_o/{table(c)}", f"{tag}_v/{table(c)[:-4]}"), td, env)
        wall += w
        err_vc += e
    return wall, {"error_estimation": phases(err_ee), "variant_calling": phases(err_vc)}


def main(out_json=None):
    res = {"workload": "configs[1] size: synthetic ASEQ, ~41 k slots x 40 normals x 96 tumours at ~5000x; C_value " + ",".join(C_VALUES)}
    res.update(gpu_info())
    with tempfile.TemporaryDirectory(prefix="sweepprog_", dir="/tmp") as td:
        td = Path(td)
        t = time.time()
        res["staging"] = stage(td)
        res["setup_s"] = round(time.time() - t, 1)
        sock_dir = tempfile.mkdtemp(prefix="as_sock_", dir="/tmp")
        sock = str(Path(sock_dir) / "as.sock")
        srv = start_service(sock)
        try:
            walls = {f"{mode}_{arm}_s": [] for mode in ("cold", "served") for arm in ("sweep", "per_value")}
            last = {}
            for rep in range(REPEATS):
                for mode, env in (("cold", {}), ("served", {"AS_SERVER": sock})):
                    order = (("sweep", arm_sweep), ("per_value", arm_per_value))
                    for arm, fn in (order if rep % 2 == 0 else order[::-1]):
                        tag = f"{mode}_{arm}_{rep}"
                        w, ph = fn(td, tag, env)
                        walls[f"{mode}_{arm}_s"].append(round(w, 3))
                        if mode == "cold":
                            last[arm] = ph
            assert srv.poll() is None
        finally:
            srv.send_signal(signal.SIGTERM)
            srv.wait(timeout=30)
            shutil.rmtree(sock_dir, ignore_errors=True)
        res.update(walls)
        for k, v in walls.items():
            res[k[:-2] + "_min_s"] = min(v)
        res["phases_last_cold_run_s"] = last
        ref = outputs(td, "cold_per_value_0_o", lambda c: f"cold_per_value_0_v/{table(c)[:-4]}")
        same = True
        for mode in ("cold", "served"):
            for rep in range(REPEATS):
                same &= outputs(td, f"{mode}_sweep_{rep}_o", lambda c: f"{mode}_sweep_{rep}_v/{table(c)[:-4]}") == ref
                same &= outputs(td, f"{mode}_per_value_{rep}_o", lambda c: f"{mode}_per_value_{rep}_v/{table(c)[:-4]}") == ref
        res["identical_outputs"] = bool(same)
        res["calls_per_value"] = {c: ref[f"{c}/Summary_Variant_Info.txt"].count("\n") - 1 for c in C_VALUES}
    print(json.dumps(res, indent=1))
    if out_json:
        Path(out_json).parent.mkdir(parents=True, exist_ok=True)
        Path(out_json).write_text(json.dumps(res, indent=1) + "\n")
    assert res["identical_outputs"], "the sweep and the runs per value differ"
    return res


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
