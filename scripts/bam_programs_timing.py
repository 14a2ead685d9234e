#!/usr/bin/env python
"""The two programs on BAM input against the two-step run they replace, at the size of BASELINE.json configs[1]: 4 normals
and 4 tumours, each a synthetic amplicon BAM of 330 x 125 panel positions at ~5000x (scripts/pileup_bench.py's reads, here
carrying the FASTA's base with a 0.5 % error rate, plus spiked variants in the tumours).

    BAM mode : AmpliSolveErrorEstimation germline_dir=N, AmpliSolveVariantCalling tumour_dir=T (the directories hold BAMs)
    two-step : computeCounts for every BAM into the same directory, then both programs on the ASEQ files

The two paths run alternately, 3 times each.  Prints one JSON object: wall time of each path per run, the AS_TIMING phases
of the last BAM-mode run (capi.pileup.encode is pileup_encode_kernel, summed over the samples), the encode kernel's time
and bytes/s from U * 32 + P * 8 bytes per sample (the packed format; U unique positions read, P packed words written,
two strands), whether the outputs of the two paths are byte-identical, and the GPU's name and power limit.

    python scripts/bam_programs_timing.py [out.json]        (on a GPU box; a few minutes, most of it writing the BAMs)
"""
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from scripts.pileup_bench import READ_LEN, bam_bytes, make_reads  # noqa: E402
from tests import aseq_io, bam_io  # noqa: E402

BIN = ROOT / "amplisolve_b200" / "bin"
N_AMP, AMP_LEN, DEPTH = 330, 125, 5000
C_VALUE, CUT = 0.002, 100
TABLE = "positionSpecificNoise_%.4f.txt" % C_VALUE


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        name, power = r.stdout.strip().splitlines()[0].split(", ")
        return {"gpu": name, "power_limit": power}
    except Exception as exc:  # noqa: BLE001
        return {"gpu": "unknown", "power_limit": f"not read: {exc}"}


def write_sample(path, ref, seed, variants):
    starts, pos, flag, mapq, _, qual = make_reads(N_AMP, AMP_LEN, DEPTH, seed)
    rng = np.random.default_rng(seed + 1000)
    seq = np.empty((len(pos), READ_LEN), np.uint8)
    for r0 in range(0, len(pos), 100_000):  # in chunks: the whole sample's positions in 64 bits would be 1.7 GB
        g = pos[r0:r0 + 100_000, None].astype(np.int64) + np.arange(READ_LEN)[None, :]  # 0-based reference position of every base
        s = ref[g]
        bad = rng.random(s.shape, np.float32) < 0.005
        s[bad] = (s[bad] + rng.integers(1, 4, int(bad.sum()))) % 4
        for p0, alt, vaf in variants:
            hit = g == p0
            hit &= rng.random(s.shape, np.float32) < vaf
            s[hit] = alt
        seq[r0:r0 + 100_000] = s
    refs = [("chr1", len(ref))]
    path.write_bytes(bam_io.bgzf_compress(bam_bytes(refs, pos, flag, mapq, seq, qual), level=1))
    return starts


def run(args, cwd, env=None):
    t = time.perf_counter()
    r = subprocess.run([str(a) for a in args], cwd=cwd, capture_output=True, text=True, env=dict(os.environ, AS_TIMING="1", **(env or {})))
    wall = time.perf_counter() - t
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "Error from" not in r.stdout and "Error:" not in r.stdout, r.stdout[-3000:]
    return wall, r.stderr


def phases(stderr, into):
    for m in re.finditer(r"AS_TIMING (\S+) ([0-9.]+)", stderr):
        into[m.group(1)] = into.get(m.group(1), 0.0) + float(m.group(2))
    return into


def vc_outputs(d):
    out = {"Summary_Variant_Info.txt": (d / "Summary_Variant_Info.txt").read_text()}
    for v in sorted(d.glob("*.vcf")):
        out[v.name] = "".join(l for l in v.read_text().splitlines(True) if not l.startswith("##fileDate"))
    return out


def main(out_json=None):
    res = {"workload": f"4 normals + 4 tumours, {N_AMP} amplicons x {AMP_LEN} positions at ~{DEPTH}x, {READ_LEN}-base reads (configs[1] size)"}
    res.update(gpu_info())
    with tempfile.TemporaryDirectory(prefix="bamprog_", dir="/tmp") as td:
        td = Path(td)
        t = time.time()
        rng = np.random.default_rng(5)
        ref = rng.integers(0, 4, 10_000 + N_AMP * 1000 + 10_000).astype(np.uint8)
        starts = 10_000 + np.arange(N_AMP, dtype=np.int64) * 1000
        (td / "panel.bed").write_text("".join(f"chr1\t{s + 1}\t{s + AMP_LEN}\n" for s in starts))
        slots = [("chr1", int(s) + 1 + i) for s in starts for i in range(AMP_LEN)]
        aseq_io.write_fasta(td, slots, ["ACGT"[ref[p - 1]] for _, p in slots])
        spikes = [(int(starts[a]) + 30 + a % 50, (int(ref[int(starts[a]) + 30 + a % 50]) + 1) % 4, 0.1) for a in range(0, N_AMP, 17)]
        for sub in ("N", "T"):
            (td / sub).mkdir()
        for k in range(4):
            write_sample(td / "N" / f"N{k + 1}.bam", ref, 100 + k, [])
            write_sample(td / "T" / f"T{k + 1}.bam", ref, 200 + k, spikes)
        res["setup_s"] = round(time.time() - t, 1)
        res["bam_bytes_per_sample"] = (td / "N" / "N1.bam").stat().st_size
        (td / "positions_ee.txt").write_text("".join(f"{c}\t{p}\t.\t.\t.\n" for c, p in slots))
        ee = lambda ndir, out: [BIN / "AmpliSolveErrorEstimation", "panel_design=panel.bed", "reference_genome=ref.fa", f"germline_dir={ndir}",
                                f"C_value={C_VALUE}", f"coverage_cutoff={CUT}", "default_error=0.01", f"output_dir={out}"]
        vc = lambda tdir, out, table: [BIN / "AmpliSolveVariantCalling", f"errorFile={table}", f"tumour_dir={tdir}", f"output_dir={out}",
                                       f"coverage_cutoff={CUT}", "p_value=0.05"]
        cc = lambda vcf, sub: [BIN / "computeCounts", f"vcf={vcf}", "bam=" + ",".join(f"{sub}/{sub}{k + 1}.bam" for k in range(4)), f"out={sub}"]
        walls = {"bam_mode_s": [], "two_step_s": []}
        last_phases = {}
        # computeCounts writes into the BAM directories themselves: the reference orders samples by hashing
        # "<dir>/<name>.PILEUP.ASEQ", so another directory would give another sample order.  The ASEQ files go again
        # before the next BAM-mode run (a directory with an ASEQ file is read as ASEQ input).
        for rep in range(3):
            for d in ("o_bam", "v_bam", "o_two", "v_two"):
                shutil.rmtree(td / d, ignore_errors=True)
            for f in list((td / "N").glob("*.ASEQ")) + list((td / "T").glob("*.ASEQ")):
                f.unlink()
            w1, e1 = run(ee("N", "o_bam"), td)
            w2, e2 = run(vc("T", "v_bam", f"o_bam/{TABLE}"), td)
            walls["bam_mode_s"].append(w1 + w2)
            last_phases = {"error_estimation": phases(e1, {}), "variant_calling": phases(e2, {})}
            encode_s = phases(e1 + e2, {}).get("capi.pileup.encode", 0.0)
            w3, _ = run(cc("positions_ee.txt", "N"), td)
            w4, _ = run(ee("N", "o_two"), td)
            dummy = td / "v_bam" / "AmpliSolveVariantCalling_interm_files" / "dummyVCF_1.vcf"
            w5, _ = run(cc(dummy, "T"), td)
            w6, _ = run(vc("T", "v_two", f"o_two/{TABLE}"), td)
            walls["two_step_s"].append(w3 + w4 + w5 + w6)
        res.update(walls)
        res["bam_mode_min_s"], res["two_step_min_s"] = min(walls["bam_mode_s"]), min(walls["two_step_s"])
        res["phases_last_bam_mode_run_s"] = last_phases
        P = U = N_AMP * AMP_LEN
        enc_bytes = 8 * (U * 32 + P * 8)
        res["encode_kernel"] = {"samples": 8, "seconds": encode_s, "bytes": enc_bytes,
                                "bytes_per_s": enc_bytes / encode_s if encode_s > 0 else None}
        res["identical_noise_table"] = (td / "o_bam" / TABLE).read_text() == (td / "o_two" / TABLE).read_text()
        a, b = vc_outputs(td / "v_bam"), vc_outputs(td / "v_two")
        res["identical_calls"] = a == b
        res["calls"] = a["Summary_Variant_Info.txt"].count("\n") - 1
        res["identical_outputs"] = res["identical_noise_table"] and res["identical_calls"]
    print(json.dumps(res, indent=1))
    if out_json:
        Path(out_json).parent.mkdir(parents=True, exist_ok=True)
        Path(out_json).write_text(json.dumps(res, indent=1) + "\n")
    assert res["identical_outputs"], "BAM mode and the two-step run differ"
    return res


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
