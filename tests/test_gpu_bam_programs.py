"""The two programs on a directory of BAM files (germline_dir= / tumour_dir= with *.bam and no *.ASEQ) against the two-step
run they replace: computeCounts with the same mbq / mrq / mdc for a position file that lists the program's panel slots in
order, into the same directory, then the same program on the ASEQ files.  Outputs must be byte-identical.  Also the device
encoder behind it (as_pileup_end_wire) against as_pack_counts and the header's 16-bit rule."""
import os
import signal
import subprocess
from pathlib import Path

import numpy as np
import pytest

from amplisolve_b200 import AmpliSolveError, api
from tests import aseq_io, bam_io

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "amplisolve_b200" / "bin"

# the panel: two overlapping amplicons (twin slots), a low-coverage amplicon (absent slots), a second contig
AMPLICONS = [("chr1", 1001, 1060), ("chr1", 1041, 1100), ("chr1", 3001, 3040), ("chr2", 501, 560)]
LOW = 2
REF_LEN = {"chr1": 6000, "chr2": 3000}
BAM_REFS = [("chr2", 3000), ("chrM", 100), ("chr1", 6000)]   # another order than the panel's, one contig it lacks
NORMALS = ["N_a", "N10", "N2", "Nb", "N1"]                  # hash order != sorted order (asserted below)
TUMOURS = ["T_2", "T10", "T1", "Tb"]
EMPTY_TUMOUR = "Tempty"                                      # header only, no records
C_VALUE, CUT = 0.002, 50


def vcf_body(path):
    return "".join(l for l in Path(path).read_text().splitlines(True) if not l.startswith("##fileDate"))


def run(prog, args, cwd, env=None, ok=True):
    r = subprocess.run([str(BIN / prog)] + args, cwd=cwd, capture_output=True, text=True, env=dict(os.environ, **(env or {})))
    if ok:
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    return r


def bed_slots():
    return [(c, p) for c, s, e in AMPLICONS for p in range(s, e + 1)]


def sample_reads(rng, ref, depth, err, variants):
    """amplicon reads (one M block, 10 bases past the amplicon) carrying the reference base, sequencing errors at rate err
    and variants {(chrom, pos): (base, fraction)}; ~5 % of the reads carry a flag of 0x704, some a low mapping quality"""
    reads = []
    for k, (c, s, e) in enumerate(AMPLICONS):
        ref_id = [n for n, _ in BAM_REFS].index(c)
        for i in range(depth if k != LOW else 12):
            start = s - 1 + int(rng.integers(-5, 6))
            L = e - s + 11
            seq = np.array([("ACGT".index(b)) for b in ref[c][start:start + L]])
            for j in range(L):
                v = variants.get((c, start + j + 1))
                if v and rng.random() < v[1]:
                    seq[j] = "ACGT".index(v[0])
            bad = rng.random(L) < err
            seq[bad] = (seq[bad] + rng.integers(1, 4, int(bad.sum()))) % 4
            flag = 16 if rng.random() < 0.5 else 0
            if rng.random() < 0.05:
                flag |= int(rng.choice([0x4, 0x100, 0x200, 0x400]))
            reads.append(dict(ref_id=ref_id, pos=start, mapq=int(rng.choice([60, 60, 60, 60, 25, 10])), flag=flag, cigar=[("M", L)],
                              seq="".join("ACGT"[b] for b in seq), qual=rng.integers(12, 41, L).astype(np.uint8).tobytes(), name=f"r{k}.{i}"))
    order = rng.permutation(len(reads))
    return [reads[i] for i in order]


def make_case(td, seed=7, depth=300, err=0.004, n_normals=5, n_tumours=4):
    """panel.bed + ref.fa, normals in N/ (germline SNPs in two of them), tumours in T/ (spiked variants; plus a BAM without
    records).  Returns the reference sequence per contig."""
    td = Path(td)
    rng = np.random.default_rng(seed)
    ref = {c: "".join(rng.choice(list("ACGT"), size=n)) for c, n in REF_LEN.items()}
    (td / "panel.bed").write_text("".join(f"{c}\t{s}\t{e}\n" for c, s, e in AMPLICONS))
    slots = bed_slots()
    aseq_io.write_fasta(td, slots, [ref[c][p - 1] for c, p in slots])
    alt = lambda c, p: "ACGT"[("ACGT".index(ref[c][p - 1]) + 1) % 4]
    germ = {("chr1", 1020): (alt("chr1", 1020), 0.5), ("chr2", 530): (alt("chr2", 530), 1.0)}
    somatic = {("chr1", 1050): (alt("chr1", 1050), 0.2), ("chr1", 1090): (alt("chr1", 1090), 0.15), ("chr2", 510): (alt("chr2", 510), 0.3)}
    (td / "N").mkdir()
    (td / "T").mkdir()
    for i, nm in enumerate(NORMALS[:n_normals]):
        bam_io.write_bam(td / "N" / f"{nm}.bam", BAM_REFS, sample_reads(rng, ref, depth, err, germ if i in (0, 2) else {}), block_bytes=9000)
    for i, nm in enumerate(TUMOURS[:n_tumours]):
        bam_io.write_bam(td / "T" / f"{nm}.bam", BAM_REFS, sample_reads(rng, ref, depth, err, somatic if i != 1 else {}), block_bytes=9000)
    bam_io.write_bam(td / "T" / f"{EMPTY_TUMOUR}.bam", BAM_REFS, [])
    return ref


def ee_args(out, germline="N"):
    return ["panel_design=panel.bed", "reference_genome=ref.fa", f"germline_dir={germline}", f"C_value={C_VALUE}", f"coverage_cutoff={CUT}",
            "default_error=0.01", f"output_dir={out}"]


def vc_args(table, out, tumours="T"):
    return [f"errorFile={table}", f"tumour_dir={tumours}", f"output_dir={out}", f"coverage_cutoff={CUT}", "p_value=0.05"]


TABLE = "positionSpecificNoise_%.4f.txt" % C_VALUE


def two_step(td, positions_lines, sub, mbq=20, mrq=20, mdc=20):
    """computeCounts for every BAM of td/sub into td/sub (the directory is then read as ASEQ input)"""
    (Path(td) / "positions.txt").write_text("".join(f"{c}\t{p}\t.\t.\t.\n" for c, p in positions_lines))
    bams = sorted(p.name for p in (Path(td) / sub).glob("*.bam"))
    run("computeCounts", ["vcf=positions.txt", "bam=" + ",".join(f"{sub}/{b}" for b in bams), f"mbq={mbq}", f"mrq={mrq}", f"mdc={mdc}",
                          f"out={sub}"], td)


def outputs_vc(d, names):
    return (Path(d) / "Summary_Variant_Info.txt").read_text(), {n: vcf_body(Path(d) / f"{n}.vcf") for n in names}


# ---- 1. the encoder --------------------------------------------------------------------------------------------------
SPECIAL = np.array([0, 15, 16, 65533, 65534, 65535, 65536, (1 << 24) + 3, (1 << 31) - 1], np.uint64)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_encoder_equals_pack_counts_and_the_16_bit_rule(ctx, seed):
    rng = np.random.default_rng(seed)
    U = 700
    counts = rng.integers(0, 12, (2, U, 4)).astype(np.uint64)
    major = rng.integers(0, 4, U)
    counts[0, np.arange(U), major] += rng.integers(0, 3000, U).astype(np.uint64)
    counts[1, np.arange(U), major] += rng.integers(0, 3000, U).astype(np.uint64)
    hit = rng.random((2, U, 4)) < 0.08
    counts[hit] = rng.choice(SPECIAL, int(hit.sum()))
    counts[:, rng.random(U) < 0.05] = 0                             # positions without reads
    counts = counts.astype(np.uint32)
    slot_unique = np.concatenate([np.arange(U), rng.integers(0, U, 300)]).astype(np.int32)   # every position, plus twins
    rng.shuffle(slot_unique)
    P = len(slot_unique)
    for mdc in (0, 1, 20, 3000, 65536, (1 << 31) - 1):
        g = counts[:, slot_unique].copy()                            # gathered [2][P][4]
        absent = g.astype(np.uint64).sum(axis=(0, 2)) < mdc          # the mdc rule on the 64-bit depth
        g[:, absent] = api.ABSENT
        want_packed, want_wide = api.pack_counts(g[None])
        wire, wide, rows, _ = ctx.pileup_end_wire(slot_unique, mdc, "packed", sample=5, counts=counts)
        assert rows == int((~absent).sum())
        assert np.array_equal(wire, want_packed[0]), mdc
        assert np.array_equal(wide["slot"], want_wide["slot"]) and (wide["sample"] == 5).all()
        assert np.array_equal(wide["fw"], want_wide["fw"]) and np.array_equal(wide["bw"], want_wide["bw"])
        want16, want_wide16 = api.to_wire16(g[None])
        wire16, wide16, rows16, _ = ctx.pileup_end_wire(slot_unique, mdc, "16", sample=5, counts=counts)
        assert rows16 == rows
        assert np.array_equal(wire16, want16[0]), mdc
        assert np.array_equal(wide16["slot"], want_wide16["slot"])
        assert np.array_equal(wide16["fw"], want_wide16["fw"]) and np.array_equal(wide16["bw"], want_wide16["bw"])
    assert len(want_wide) > 2 and len(want_wide16) > 2, "the case must escape records in both formats"
    with pytest.raises(AmpliSolveError) as e:                        # too small a list: the true count comes back
        ctx.pileup_end_wire(slot_unique, 0, "packed", wide_cap=2, counts=counts)
    assert e.value.code == -5 and e.value.n_wide == len(api.pack_counts(counts[:, slot_unique][None])[1])
    wire, wide, _, _ = ctx.pileup_end_wire(slot_unique, 0, "packed")  # the pileup stayed open: the same call with room
    assert len(wide) == e.value.n_wide
    bad = slot_unique.copy()
    bad[7] = U
    with pytest.raises(AmpliSolveError) as e:
        ctx.pileup_end_wire(bad, 0, "packed", counts=counts)
    assert e.value.code == -1
    bad[7] = -1
    with pytest.raises(AmpliSolveError) as e:
        ctx.pileup_end_wire(bad, 0, "packed", counts=counts)
    assert e.value.code == -1


# ---- 2. the error estimation program ---------------------------------------------------------------------------------
def test_sample_names_hash_in_another_order_than_sorted():
    for d, names in (("N", NORMALS), ("T", TUMOURS + [EMPTY_TUMOUR])):
        keys = sorted(f"{d}/{n}.PILEUP.ASEQ" for n in names)
        assert api.hash_iteration_order(keys) != list(range(len(keys)))


@pytest.mark.parametrize("mbq,mrq,mdc", [(20, 20, 20), (30, 25, 60), (0, 0, 0)])
def test_error_estimation_bam_input_equals_two_step(tmp_path, mbq, mrq, mdc):
    make_case(tmp_path, n_tumours=0)
    env = {"AS_BAM_MBQ": str(mbq), "AS_BAM_MRQ": str(mrq), "AS_BAM_MDC": str(mdc)}
    r = run("AmpliSolveErrorEstimation", ee_args("o_bam"), tmp_path, env)
    assert f"{mbq} / {mrq} / {mdc}" in r.stdout
    listed = next((tmp_path / "o_bam" / "AmpliSolveErrorEstimation_interm_files").glob("*_germline_count_list_original.txt")).read_text()
    assert listed.count(".bam\n") == len(NORMALS)
    two_step(tmp_path, bed_slots(), "N", mbq, mrq, mdc)
    run("AmpliSolveErrorEstimation", ee_args("o_aseq"), tmp_path)
    want = (tmp_path / "o_aseq" / TABLE).read_text()
    assert (tmp_path / "o_bam" / TABLE).read_text() == want
    rows = (tmp_path / "N" / "N1.PILEUP.ASEQ").read_text().count("\n") - 1
    if mdc > 12:   # the low-coverage amplicon is absent, the other slots present
        assert 0 < rows < len(bed_slots())
    if mdc == 0:
        assert rows == len(bed_slots())


# ---- 3. the variant calling program ----------------------------------------------------------------------------------
def test_variant_calling_bam_input_equals_two_step(tmp_path):
    make_case(tmp_path)
    run("AmpliSolveErrorEstimation", ee_args("o"), tmp_path)
    table = f"o/{TABLE}"
    run("AmpliSolveVariantCalling", vc_args(table, "v_bam"), tmp_path)
    run("AmpliSolveVariantCalling", vc_args(table, "v_grouped"), tmp_path, {"AS_GROUP_SAMPLES": "1"})
    dummy = (tmp_path / "v_bam" / "AmpliSolveVariantCalling_interm_files" / "dummyVCF_1.vcf").read_text().splitlines()
    two_step(tmp_path, [tuple(l.split("\t")[:2]) for l in dummy], "T")
    run("AmpliSolveVariantCalling", vc_args(table, "v_aseq"), tmp_path)
    names = TUMOURS + [EMPTY_TUMOUR]
    want = outputs_vc(tmp_path / "v_aseq", names)
    assert want[0].count("\n") > 3, "the case must make calls"
    assert "Tempty" not in want[0] and want[1]["Tempty"].endswith("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n")
    assert outputs_vc(tmp_path / "v_bam", names) == want
    assert outputs_vc(tmp_path / "v_grouped", names) == want


# ---- 4. wire formats -------------------------------------------------------------------------------------------------
def test_noisy_bams_switch_to_16_bit_and_every_format_agrees(tmp_path):
    make_case(tmp_path, depth=600, err=0.25, n_normals=4, n_tumours=3)
    run("AmpliSolveErrorEstimation", ee_args("o"), tmp_path)
    table = f"o/{TABLE}"
    outs = {}
    for wire in ("auto", "packed", "16"):
        env = {} if wire == "auto" else {"AS_WIRE": wire}
        run("AmpliSolveVariantCalling", vc_args(table, f"v_{wire}"), tmp_path, env)
        run("AmpliSolveErrorEstimation", ee_args(f"o_{wire}"), tmp_path, env)
        outs[wire] = outputs_vc(tmp_path / f"v_{wire}", TUMOURS[:3]), (tmp_path / f"o_{wire}" / TABLE).read_text()
    dummy = (tmp_path / "v_auto" / "AmpliSolveVariantCalling_interm_files" / "dummyVCF_1.vcf").read_text().splitlines()
    two_step(tmp_path, [tuple(l.split("\t")[:2]) for l in dummy], "T")
    two_step(tmp_path, bed_slots(), "N")
    run("AmpliSolveVariantCalling", vc_args(table, "v_aseq"), tmp_path)
    run("AmpliSolveErrorEstimation", ee_args("o_aseq"), tmp_path)
    want = outputs_vc(tmp_path / "v_aseq", TUMOURS[:3]), (tmp_path / "o_aseq" / TABLE).read_text()
    # the data: more than 1 record in 16 has a minor count above 15 (the automatic choice is then the 16-bit format)
    rows = [l.split("\t") for l in (tmp_path / "T" / "T1.PILEUP.ASEQ").read_text().splitlines()[1:]]
    noisy = 0
    for r in rows:
        v = np.array([int(x) for x in r[6:]])
        fw, bw = v[:4] - v[5:], v[5:]
        noisy += int(np.sort(fw)[-2] > 15 or np.sort(bw)[-2] > 15)
    assert noisy * 16 > len(rows)
    for wire in outs:
        assert outs[wire] == want, wire


# ---- 5. errors -------------------------------------------------------------------------------------------------------
def test_unreadable_bams_report_the_compute_counts_message(tmp_path):
    make_case(tmp_path, depth=40, n_normals=2, n_tumours=0)
    good = (tmp_path / "N" / "N_a.bam").read_bytes()
    (tmp_path / "N" / "N_a.bam").write_bytes(b"not a BAM file at all, not even gzip" * 3)
    r = run("AmpliSolveErrorEstimation", ee_args("o1"), tmp_path)
    assert "is not a BGZF (BAM) file" in r.stdout and not (tmp_path / "o1" / TABLE).exists()
    bad = bytearray(good)
    bad[40] ^= 0xFF   # inside the deflate stream of the first block
    (tmp_path / "N" / "N_a.bam").write_bytes(bytes(bad))
    r = run("AmpliSolveErrorEstimation", ee_args("o2"), tmp_path)
    assert "does not inflate" in r.stdout and not (tmp_path / "o2" / TABLE).exists()
    (tmp_path / "N" / "N_a.bam").write_bytes(good[:len(good) // 2])   # cut inside a block
    r = run("AmpliSolveErrorEstimation", ee_args("o3"), tmp_path)
    assert "Error from computeCounts" in r.stdout and not (tmp_path / "o3" / TABLE).exists()
    (tmp_path / "N" / "N_a.bam").write_bytes(good)
    run("AmpliSolveErrorEstimation", ee_args("o4"), tmp_path)
    (tmp_path / "T" / "Tx.bam").write_bytes(b"\x1f\x8b" + b"garbage" * 10)
    r = run("AmpliSolveVariantCalling", vc_args(f"o4/{TABLE}", "v"), tmp_path)
    assert "is not a BGZF (BAM) file" in r.stdout and not (tmp_path / "v" / "Summary_Variant_Info.txt").exists()


# ---- 6. the resident service -----------------------------------------------------------------------------------------
def test_bam_input_through_the_resident_service(tmp_path, socket_path):
    make_case(tmp_path, n_normals=4, n_tumours=2)
    run("AmpliSolveErrorEstimation", ee_args("o"), tmp_path)
    run("AmpliSolveVariantCalling", vc_args(f"o/{TABLE}", "v"), tmp_path)
    names = TUMOURS[:2] + [EMPTY_TUMOUR]
    srv = subprocess.Popen([str(BIN / "amplisolve_b200_serve"), f"socket={socket_path}"], cwd="/", stderr=subprocess.PIPE, text=True)
    try:
        assert "ready" in srv.stderr.readline()
        for rnd in range(2):
            env = {"AS_SERVER": socket_path}
            run("AmpliSolveErrorEstimation", ee_args(f"os{rnd}"), tmp_path, env)
            assert (tmp_path / f"os{rnd}" / TABLE).read_text() == (tmp_path / "o" / TABLE).read_text()
            run("AmpliSolveVariantCalling", vc_args(f"o/{TABLE}", f"vs{rnd}"), tmp_path, env)
            assert outputs_vc(tmp_path / f"vs{rnd}", names) == outputs_vc(tmp_path / "v", names)
        assert srv.poll() is None
    finally:
        srv.send_signal(signal.SIGTERM)
        srv.wait(timeout=20)


# ---- 7. several GPUs -------------------------------------------------------------------------------------------------
def test_bam_input_on_two_gpus_equals_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")
    make_case(tmp_path, n_normals=4, n_tumours=3)
    names = TUMOURS[:3] + [EMPTY_TUMOUR]
    for tag, devs in (("one", "0"), ("two", "0,1")):
        run("AmpliSolveErrorEstimation", ee_args(f"o_{tag}"), tmp_path, {"AS_DEVICES": devs})
        run("AmpliSolveVariantCalling", vc_args(f"o_{tag}/{TABLE}", f"v_{tag}"), tmp_path, {"AS_DEVICES": devs, "AS_GROUP_SAMPLES": "2"})
    assert (tmp_path / "o_two" / TABLE).read_text() == (tmp_path / "o_one" / TABLE).read_text()
    assert outputs_vc(tmp_path / "v_two", names) == outputs_vc(tmp_path / "v_one", names)
