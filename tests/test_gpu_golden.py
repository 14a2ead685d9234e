"""GPU tests against the golden fixtures generated from the compiled reference (tests/golden/):
the CUDA path through the C ABI, and the two drop-in programs end to end, byte for byte."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import pyoracle
from tests import aseq_io
from tests import golden_util as gu

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "amplisolve_b200" / "bin"


@pytest.mark.parametrize("name", gu.CASES)
def test_noise_table_from_cuda_is_text_identical(ctx, name):
    from amplisolve_b200 import twin_links
    case = gu.load(name)
    normals = np.ascontiguousarray(case["normals"][case["normal_order"]])
    nxt, head = twin_links(case["pos_id"])
    got = ctx.estimate_thresholds(normals, float(case["c_value"]), int(case["cutoff"]), nxt, head)
    lines = gu.noise_table_lines(case, got["thr"], got["germ_val"].astype(np.float64), got["germ_state"])
    want = case["noise_table"].splitlines()
    bad = [i for i, (a, b) in enumerate(zip(lines, want)) if a != b]
    assert len(lines) == len(want) and not bad, (bad[:5], lines[bad[0]] if bad else "", want[bad[0]] if bad else "")


@pytest.mark.parametrize("name", gu.CASES)
def test_calls_from_cuda_match_reference_rows(ctx, name):
    case = gu.load(name)
    order = case["tumour_order"]
    tumours = np.ascontiguousarray(case["tumours"][order])
    thr_view = gu.parse_noise_thresholds(case)
    calls = ctx.call_variants(tumours, case["ref_code"], thr_view, int(case["cutoff"]))
    want = gu.golden_call_rows(case)
    assert len(calls) == len(want) > 0
    for c, w in zip(calls, want):
        chrom, pos = case["slots"][c["slot"]]
        cnt = tumours[c["sample"], :, c["slot"], :].astype(np.int64)
        FW, BW = int(cnt[0].sum()), int(cnt[1].sum())
        got = (case["tumour_names"][order[c["sample"]]], chrom, pos, "ACGT"[c["ref"]], "ACGT"[c["alt"]], FW + BW, FW, BW,
               int(cnt[0, c["alt"]]), int(cnt[1, c["alt"]]), gu.fmt_g(pyoracle.q_from_p(c["p_fw"])),
               gu.fmt_g(pyoracle.q_from_p(c["p_bw"])))
        assert got == w[:12]
        assert gu.fmt_g(c["q_fw"]) == w[10] and gu.fmt_g(c["q_bw"]) == w[11]   # the device's own fp64 Q prints alike


def run(prog, args, cwd, env=None):
    import os
    r = subprocess.run([str(BIN / prog)] + args, cwd=cwd, capture_output=True, text=True,
                       env=None if env is None else dict(os.environ, **env))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
    return r.stdout


def vcf_body(path):
    return "".join(l for l in open(path) if not l.startswith("##fileDate="))


@pytest.mark.parametrize("name", gu.CASES + ["toy_full"])
def test_programs_end_to_end_byte_identical(name, tmp_path):
    """BASELINE.json configs[0]/[1] shape: AmpliSolveErrorEstimation on N/ + BED, then AmpliSolveVariantCalling on T/
    with the table just written; every output file equals the reference's (VCF minus its ##fileDate line)."""
    case = gu.load(name)
    slots = aseq_io.stage_case(tmp_path, case)
    aseq_io.write_fasta(tmp_path, slots, list(case["ref_letters"]))
    c_text = "%g" % float(case["c_value"])
    out = run("AmpliSolveErrorEstimation", ["panel_design=panel.bed", "reference_genome=ref.fa", "germline_dir=N",
                                            f"C_value={c_text}", f"coverage_cutoff={int(case['cutoff'])}",
                                            "default_error=0.01", "output_dir=o"], tmp_path)
    tables = sorted((tmp_path / "o").glob("positionSpecificNoise_*.txt"))
    assert len(tables) == 1 and tables[0].name == "positionSpecificNoise_%.4f.txt" % float(case["c_value"]), out[-2000:]
    assert tables[0].read_text() == case["noise_table"]
    run("AmpliSolveVariantCalling", [f"errorFile=o/{tables[0].name}", "tumour_dir=T", "output_dir=v",
                                     f"coverage_cutoff={int(case['cutoff'])}", "p_value=0.05"], tmp_path)
    assert (tmp_path / "v" / "Summary_Variant_Info.txt").read_text() == case["summary"]
    for nm in case["tumour_names"]:
        assert vcf_body(tmp_path / "v" / f"{nm}.vcf") == case["vcfs"][nm], nm
    dummy = (tmp_path / "v" / "AmpliSolveVariantCalling_interm_files" / "dummyVCF_1.vcf").read_text().splitlines()
    assert len(dummy) == len(slots) and dummy[0] == f"{slots[0][0]}\t{slots[0][1]}\t.\t.\t.\t.\t.\t."


def test_programs_through_the_resident_service(tmp_path, socket_path):
    """amplisolve_b200_serve holds the CUDA context; the same programs, started with AS_SERVER, run inside it: outputs byte
    for byte those of the reference, twice in a row (every run gets and returns its own device memory), and the wait for
    CUDA is gone from the phases."""
    import os
    import re
    import signal
    sock = socket_path
    srv = subprocess.Popen([str(BIN / "amplisolve_b200_serve"), f"socket={sock}"], cwd="/", stderr=subprocess.PIPE, text=True)
    try:
        assert "ready" in srv.stderr.readline()
        for rnd, name in enumerate(["toy_full", gu.CASES[0], "toy_full"]):
            case = gu.load(name)
            wd = tmp_path / f"w{rnd}"
            wd.mkdir()
            slots = aseq_io.stage_case(wd, case)
            aseq_io.write_fasta(wd, slots, list(case["ref_letters"]))
            env = dict(os.environ, AS_SERVER=sock, AS_TIMING="1")
            r = subprocess.run([str(BIN / "AmpliSolveErrorEstimation"), "panel_design=panel.bed", "reference_genome=ref.fa", "germline_dir=N",
                                "C_value=%g" % float(case["c_value"]), f"coverage_cutoff={int(case['cutoff'])}", "default_error=0.01",
                                "output_dir=o"], cwd=wd, capture_output=True, text=True, env=env)
            assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-1000:]
            table = "positionSpecificNoise_%.4f.txt" % float(case["c_value"])
            assert (wd / "o" / table).read_text() == case["noise_table"]
            wait = float(re.search(r"AS_TIMING cuda_context_wait ([0-9.]+)", r.stderr).group(1))   # the client's stderr got the phases
            assert wait < 0.2, wait
            r = subprocess.run([str(BIN / "AmpliSolveVariantCalling"), f"errorFile=o/{table}", "tumour_dir=T", "output_dir=v",
                                f"coverage_cutoff={int(case['cutoff'])}", "p_value=0.05"], cwd=wd, capture_output=True, text=True, env=env)
            assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-1000:]
            assert (wd / "v" / "Summary_Variant_Info.txt").read_text() == case["summary"]
            for nm in case["tumour_names"]:
                assert vcf_body(wd / "v" / f"{nm}.vcf") == case["vcfs"][nm], nm
        assert srv.poll() is None
    finally:
        srv.send_signal(signal.SIGTERM)
        srv.wait(timeout=20)


@pytest.mark.parametrize("wire", ["16", "packed"])
def test_programs_byte_identical_in_either_wire_format(wire, tmp_path):
    """The loaders write the packed wire format and fall back to the 16-bit one for ultra-deep data; AS_WIRE forces one.
    Either way every output byte is the reference's (the Toy_data slice has 5000x rows: many records escape the packed
    form, none the 16-bit one)."""
    case = gu.load("toy_slice")
    slots = aseq_io.stage_case(tmp_path, case)
    aseq_io.write_fasta(tmp_path, slots, list(case["ref_letters"]))
    env = {"AS_WIRE": wire}
    run("AmpliSolveErrorEstimation", ["panel_design=panel.bed", "reference_genome=ref.fa", "germline_dir=N",
                                      "C_value=%g" % float(case["c_value"]), f"coverage_cutoff={int(case['cutoff'])}",
                                      "default_error=0.01", "output_dir=o"], tmp_path, env)
    table = tmp_path / "o" / ("positionSpecificNoise_%.4f.txt" % float(case["c_value"]))
    assert table.read_text() == case["noise_table"]
    run("AmpliSolveVariantCalling", [f"errorFile=o/{table.name}", "tumour_dir=T", "output_dir=v",
                                     f"coverage_cutoff={int(case['cutoff'])}", "p_value=0.05"], tmp_path, env)
    assert (tmp_path / "v" / "Summary_Variant_Info.txt").read_text() == case["summary"]
    for nm in case["tumour_names"]:
        assert vcf_body(tmp_path / "v" / f"{nm}.vcf") == case["vcfs"][nm], nm


def test_program_falls_back_to_16_bit_on_ultra_deep_panels(tmp_path):
    """At 50,000x (configs[4]) most records carry an error count above 15 and would escape the packed form: the loader
    notices (more than 1 record in 16) and parses into the 16-bit format instead.  The table must equal the one the
    forced formats give, and the oracle's."""
    from tests import synth
    bed, slots, pos_id, U = synth.make_panel(6, seed=71, chroms=("chr7",))
    P = len(slots)
    normals, ref = synth.make_counts(8, P, depth=50000, seed=71, pos_id=pos_id)
    from amplisolve_b200 import pack_counts
    _, wide = pack_counts(normals)
    assert len(wide) * 16 > (normals[:, 0, :, 0] != 0xFFFFFFFF).sum()          # the fallback condition holds
    ref_u = np.zeros(U, np.uint8)
    ref_u[pos_id] = ref
    case = {"bed": "".join(f"{c}\t{s}\t{e}\tA{i}\t.\tG\n" for i, (c, s, e) in enumerate(bed)),
            "ref_letters": "".join("ACGT"[r] for r in ref_u[pos_id]), "normal_names": [f"DEEP{i}" for i in range(8)],
            "normals": normals, "tumour_names": [], "tumours": np.zeros((0, 2, P, 4), np.uint32)}
    slots2 = aseq_io.stage_case(tmp_path, case)
    aseq_io.write_fasta(tmp_path, slots2, list(case["ref_letters"]))
    args = ["panel_design=panel.bed", "reference_genome=ref.fa", "germline_dir=N", "C_value=0.002", "coverage_cutoff=100",
            "default_error=0.01"]
    tables = {}
    for tag, env in (("auto", None), ("w16", {"AS_WIRE": "16"}), ("packed", {"AS_WIRE": "packed"})):
        run("AmpliSolveErrorEstimation", args + [f"output_dir=o_{tag}"], tmp_path, env)
        tables[tag] = (tmp_path / f"o_{tag}" / "positionSpecificNoise_0.0020.txt").read_text()
    assert tables["auto"] == tables["w16"] == tables["packed"]
    order = pyoracle.hash_iteration_order([f"N/{n}.PILEUP.ASEQ" for n in case["normal_names"]])
    rows, off = pyoracle.dense_to_rows(synth.to_oracle_layout(normals[order]), pos_id)
    nz = pyoracle.noise_estimate(rows, off, U, np.float32(0.002), 100)
    case.update(slots=slots2)
    want = gu.noise_table_lines(case, nz["thr"][pos_id], nz["germ_val"][pos_id], nz["germ_present"][pos_id])
    assert tables["auto"].splitlines() == want


def test_program_escapes_counts_beyond_the_16_bit_wire_format(tmp_path):
    """The loaders fill a wire format (packed, or 16-bit on ultra-deep data); a record that does not fit -- here counts of
    65534 or more, which escape both -- goes to the side list of wide records.  Checked end to end against the oracle's table on a panel with a few ultra-deep positions (incl.
    depths beyond 2^24, where int -> float stops being exact)."""
    from tests import synth
    bed, slots, pos_id, U = synth.make_panel(14, seed=61, chroms=("chr5",))
    P = len(slots)
    normals, ref = synth.make_counts(6, P, depth=3000, seed=61, pos_id=pos_id, big_rate=0.01)
    normals[2, 0, 7, :] = [70000, 3, 0, 1]          # one count just beyond 16 bits
    assert normals[normals != 0xFFFFFFFF].max() >= 1 << 24
    ref_u = np.zeros(U, np.uint8)
    ref_u[pos_id] = ref
    case = {"bed": "".join(f"{c}\t{s}\t{e}\tA{i}\t.\tG\n" for i, (c, s, e) in enumerate(bed)),
            "ref_letters": "".join("ACGT"[r] for r in ref_u[pos_id]), "normal_names": [f"BIG{i}" for i in range(6)],
            "normals": normals, "tumour_names": [], "tumours": np.zeros((0, 2, P, 4), np.uint32)}
    slots2 = aseq_io.stage_case(tmp_path, case)
    aseq_io.write_fasta(tmp_path, slots2, list(case["ref_letters"]))
    run("AmpliSolveErrorEstimation", ["panel_design=panel.bed", "reference_genome=ref.fa", "germline_dir=N", "C_value=0.002",
                                      "coverage_cutoff=100", "default_error=0.01", "output_dir=o"], tmp_path)
    got = (tmp_path / "o" / "positionSpecificNoise_0.0020.txt").read_text().splitlines()
    order = pyoracle.hash_iteration_order([f"N/{n}.PILEUP.ASEQ" for n in case["normal_names"]])
    rows, off = pyoracle.dense_to_rows(synth.to_oracle_layout(normals[order]), pos_id)
    nz = pyoracle.noise_estimate(rows, off, U, np.float32(0.002), 100)
    case.update(slots=slots2)
    want = gu.noise_table_lines(case, nz["thr"][pos_id], nz["germ_val"][pos_id], nz["germ_present"][pos_id])
    assert got == want


def _irregular():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_irregular", gu.GOLDEN / "make_irregular.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    z = np.load(gu.GOLDEN / "irregular_rows.npz", allow_pickle=False)
    return mod, {k: z[k] for k in z.files}


def _run_both_programs(case, workdir):
    run("AmpliSolveErrorEstimation", ["panel_design=panel.bed", "reference_genome=ref.fa", "germline_dir=N",
                                      "C_value=%g" % float(case["c_value"]), f"coverage_cutoff={int(case['cutoff'])}",
                                      "default_error=0.01", "output_dir=o"], workdir)
    table = workdir / "o" / ("positionSpecificNoise_%.4f.txt" % float(case["c_value"]))
    run("AmpliSolveVariantCalling", [f"errorFile=o/{table.name}", "tumour_dir=T", "output_dir=v",
                                     f"coverage_cutoff={int(case['cutoff'])}", "p_value=0.05"], workdir)
    return table.read_text()


def test_rows_beyond_the_panel_slots_and_rd_column_are_handled_like_the_reference(tmp_path):
    """VERDICT r01 missing item 4.  A file that lists a position more often than the panel enumerates it: the reference
    counts every such row in the noise model (EE:1241-1245: N, sums, count, Germ_Max) and tests every such row in the caller;
    a tumour row whose RD column is not A+C+G+T: the reference's AF and RD columns use the column (VC:814-817).  The
    programs reproduce both: every output byte equals the compiled reference's on the patched synth_small case
    (tests/golden/make_irregular.py: a repeated normal row, a third row of a duplicated position, a repeated called tumour
    row, a tumour RD column off by 9)."""
    mod, fx = _irregular()
    case = gu.load("synth_small")
    slots = aseq_io.stage_case(tmp_path, case)
    aseq_io.write_fasta(tmp_path, slots, list(case["ref_letters"]))
    mod.apply_patches(tmp_path, case, ee_rd=False)
    table = _run_both_programs(case, tmp_path)
    assert table != case["noise_table"]                       # the extra rows matter ...
    assert table == str(fx["noise_table"])                    # ... exactly as they do in the reference
    assert (tmp_path / "v" / "Summary_Variant_Info.txt").read_text() == str(fx["summary"])
    assert len(str(fx["summary"]).splitlines()) == len(case["summary"].splitlines()) + 1
    for nm, body in zip(fx["vcf_names"], fx["vcf_bodies"]):
        assert vcf_body(tmp_path / "v" / f"{nm}.vcf") == str(body), nm


def test_rd_column_of_a_normal_row_is_the_one_documented_deviation(tmp_path):
    """The dense tensor stores the eight strand counts, not the RD column.  In a NORMAL row whose RD column is not
    A+C+G+T the reference computes the total allele fractions of Germ_Max with the column (EE:1229-1232); this
    implementation uses the sum (DESIGN.md, known deviations) and says so on stdout.  This test pins where the outputs
    diverge: only the Germ_Max cells of that one position; thresholds, every other line and the line count are the
    reference's."""
    mod, fx = _irregular()
    case = gu.load("synth_small")
    slots = aseq_io.stage_case(tmp_path, case)
    aseq_io.write_fasta(tmp_path, slots, list(case["ref_letters"]))
    done = mod.apply_patches(tmp_path, case, ee_rd=True)
    chrom, pos = [d for d in done if d[0] == "normal RD column halved"][0][2]
    out = run("AmpliSolveErrorEstimation", ["panel_design=panel.bed", "reference_genome=ref.fa", "germline_dir=N",
                                            "C_value=%g" % float(case["c_value"]), f"coverage_cutoff={int(case['cutoff'])}",
                                            "default_error=0.01", "output_dir=o"], tmp_path)
    assert "RD column is not A+C+G+T" in out
    ours = (tmp_path / "o" / ("positionSpecificNoise_%.4f.txt" % float(case["c_value"]))).read_text().splitlines()
    ref = str(fx["noise_table_rd"]).splitlines()
    assert len(ours) == len(ref)
    diff = [(a.split("\t"), b.split("\t")) for a, b in zip(ours, ref) if a != b]
    assert 1 <= len(diff) <= 2
    for a, b in diff:
        assert a[:2] == [chrom, str(pos)] and a[:8] == b[:8] and a[8:] != b[8:]   # thresholds equal, Germ_Max differs
    assert ours == str(fx["noise_table"]).splitlines()        # = the table without the RD edit: the sum is what is used


def test_files_whose_rows_do_not_follow_the_panel_order(tmp_path):
    """ASEQ files normally list their rows in the panel's enumeration order, which the loader's cursor and the device's
    (sample, slot, alt) sort rely on.  A file that does not (rows reversed, halves swapped) takes the fall-back paths: hash
    lookup per row, a second parse with a row -> slot map, calls re-ordered by file row.  Outputs must still equal the
    compiled reference's, byte for byte (tests/golden/make_irregular.py shuffle_rows)."""
    mod, fx = _irregular()
    case = gu.load("synth_small")
    slots = aseq_io.stage_case(tmp_path, case)
    aseq_io.write_fasta(tmp_path, slots, list(case["ref_letters"]))
    mod.shuffle_rows(tmp_path, case)
    table = _run_both_programs(case, tmp_path)
    assert table == str(fx["shuffled_noise_table"])
    summary = (tmp_path / "v" / "Summary_Variant_Info.txt").read_text()
    assert summary == str(fx["shuffled_summary"]) and summary != case["summary"]      # same calls, another order
    for nm, body in zip(fx["shuffled_vcf_names"], fx["shuffled_vcf_bodies"]):
        assert vcf_body(tmp_path / "v" / f"{nm}.vcf") == str(body), nm


@pytest.mark.parametrize("group", [1, 2, 4])
def test_caller_program_in_sample_groups(group, tmp_path):
    """The variant-calling program parses and calls the tumours in groups (two pinned buffers: one group is parsed while the
    GPU works on the other).  Whatever the group size -- here 1, 2 and 4 of 6 tumours, incl. a last group that is not full --
    the outputs are the reference's."""
    case = gu.load("synth_small")
    slots = aseq_io.stage_case(tmp_path, case)
    aseq_io.write_fasta(tmp_path, slots, list(case["ref_letters"]))
    (tmp_path / "o").mkdir()
    table = tmp_path / "o" / ("positionSpecificNoise_%.4f.txt" % float(case["c_value"]))
    table.write_text(case["noise_table"])
    run("AmpliSolveVariantCalling", [f"errorFile=o/{table.name}", "tumour_dir=T", "output_dir=v",
                                     f"coverage_cutoff={int(case['cutoff'])}", "p_value=0.05"], tmp_path, {"AS_GROUP_SAMPLES": str(group)})
    assert (tmp_path / "v" / "Summary_Variant_Info.txt").read_text() == case["summary"]
    for nm in case["tumour_names"]:
        assert vcf_body(tmp_path / "v" / f"{nm}.vcf") == case["vcfs"][nm], nm
