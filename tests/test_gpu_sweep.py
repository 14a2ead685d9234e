"""Noise-floor sweep (several values of C in one run) through every layer above the two sweep kernels: the _host entry points
(as_noise_estimate_sweep_host*, as_call_variants_sweep_host*), AmpliSolveErrorEstimation with C_value=a,b,c and
AmpliSolveVariantCalling with errorFile=<directory>.  Every result must equal one single-value run per value."""
import os
import signal
import subprocess
from pathlib import Path

import numpy as np
import pytest

from amplisolve_b200 import api
from tests import aseq_io, synth
from tests import golden_util as gu
from tests import test_gpu_bam_programs as bp

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "amplisolve_b200" / "bin"
C_VALUES = [0.001, 0.0015, 0.002, 0.003, 0.004, 0.005, 0.0075, 0.01]
FORMATS = ["u32", "u16", "packed"]


def bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


def encode(counts, fmt):
    if fmt == "u32":
        return counts, None
    return api.to_wire16(counts) if fmt == "u16" else api.pack_counts(counts)


def sweep_data(seed=102):
    """twin pairs inside and across upload tiles, a position enumerated three times (its group spans the panel), ragged
    absent rows and counts beyond 2^24 (escaped by both wire formats)"""
    _, slots, pos_id, U = synth.make_panel(60, seed=seed, overlap_frac=0.6, amp_len=(20, 70))
    pos_id = pos_id.copy()
    pos_id[-3] = pos_id[5]
    P = len(slots)
    normals, ref = synth.make_counts(17, P, depth=3000, seed=seed, pos_id=pos_id, big_rate=0.01, ragged_twins=True)
    tumours, _ = synth.make_counts(23, P, depth=3000, seed=seed + 1, ref=ref, pos_id=pos_id, somatic_rate=0.02, big_rate=0.01)
    nxt, head = api.twin_links(pos_id)
    return normals, tumours, ref, nxt, head


# ---- 1. noise sweep on the host path ---------------------------------------------------------------------------------
@pytest.mark.parametrize("tile", [0, 256])
@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("n_c", [1, 2, 5, 8])
def test_noise_sweep_host_equals_one_run_per_value(ctx, n_c, fmt, tile):
    normals, _, _, nxt, head = sweep_data()
    counts, wide = encode(normals, fmt)
    cv = C_VALUES[:n_c]
    ctx.set_host_tile_slots(tile)
    try:
        before = ctx.kernel_launches
        got = ctx.estimate_thresholds_sweep(counts, cv, 100, nxt, head, wide_records=wide)
        sweep_launches = ctx.kernel_launches - before
        for i, c in enumerate(cv):
            before = ctx.kernel_launches
            one = ctx.estimate_thresholds(counts, c, 100, nxt, head, wide_records=wide, with_view=True)
            if n_c == 1:
                assert sweep_launches == ctx.kernel_launches - before     # a sweep of one is the single-value path
            assert np.array_equal(bits(got["thr"][i]), bits(one["thr"])), c
            assert np.array_equal(bits(got["thr_view"][i]), bits(one["thr_view"])), c
            for k in ("germ_val", "germ_state", "count", "nrec"):
                assert np.array_equal(bits(got[k]), bits(one[k])), (c, k)
    finally:
        ctx.set_host_tile_slots(0)
    assert n_c == 1 or not np.array_equal(bits(got["thr"][0]), bits(got["thr"][-1]))


def test_noise_sweep_host_rejects_bad_counts_of_values(ctx):
    normals, _, _, nxt, head = sweep_data()
    P = normals.shape[2]
    out = [np.empty(P * 8 * 9, np.float32), np.empty(P * 4, np.float32), np.empty(P * 4, np.uint8), np.empty(P * 4, np.uint32),
           np.empty(P, np.uint32)]
    cv = np.array(C_VALUES + [0.02], np.float32)
    for n_c in (0, 9):
        rc = api.lib().as_noise_estimate_sweep_host(ctx._h, api._hp(normals), normals.shape[0], P, api._hp(nxt), api._hp(head),
                                                    api._hp(cv), n_c, 100, *[api._hp(a) for a in out], None)
        assert rc == -1, n_c     # AS_EINVAL


# ---- 2. caller sweep on the host path --------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def caller_tables(ctx):
    normals, tumours, ref, nxt, head = sweep_data()
    views = ctx.estimate_thresholds_sweep(normals, C_VALUES, 100, nxt, head)["thr_view"]
    return tumours, ref, views


@pytest.mark.parametrize("mode", ["deferred", "deferred-overflow", "in-stage"])
@pytest.mark.parametrize("tile", [0, 256])
@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("n_c", [2, 5, 8])
def test_caller_sweep_host_equals_one_run_per_table(ctx, caller_tables, n_c, fmt, tile, mode):
    tumours, ref, views = caller_tables
    counts, wide = encode(tumours, fmt)
    ctx.set_host_tile_slots(tile)
    if mode == "in-stage":
        ctx.set_call_kernel(11)
    if mode == "deferred-overflow":
        ctx.set_option("deferred_capacity", 7)
    try:
        got = ctx.call_variants_sweep(counts, ref, views[:n_c], 100, wide_records=wide)
    finally:
        ctx.set_host_tile_slots(0)
        ctx.set_call_kernel(-1)
        ctx.set_option("deferred_capacity", 0)
    assert len(got) == n_c
    for i in range(n_c):
        want = ctx.call_variants(counts, ref, views[i], 100, wide_records=wide)
        assert len(want) > 0 and got[i].tobytes() == want.tobytes(), i
    assert len(got[0]) > len(got[-1])


def test_caller_sweep_host_overflow_and_range(ctx, caller_tables):
    tumours, ref, views = caller_tables
    T, _, P, _ = tumours.shape
    n_c = 5
    tv = np.ascontiguousarray(views[:n_c])
    full = [ctx.call_variants(tumours, ref, tv[i], 100) for i in range(n_c)]
    sizes = [len(f) for f in full]
    cap = (sizes[0] + sizes[-1]) // 2          # below the first table's count, above the last one's
    assert sizes[-1] < cap < sizes[0]
    calls = np.zeros((n_c, cap), api.CALL_DTYPE)
    n = np.zeros(n_c, np.int64)
    rc = api.lib().as_call_variants_sweep_host(ctx._h, api._hp(tumours), T, P, api._hp(ref), api._hp(tv), n_c, 100, api._hp(calls), cap,
                                               api._hp(n))
    assert rc == -5                            # AS_EOVERFLOW
    assert list(n) == sizes                    # the true count of every table
    for i in range(n_c):
        if sizes[i] <= cap:
            assert calls[i, :sizes[i]].tobytes() == full[i].tobytes(), i
        else:                                  # cap valid calls of the table (which ones is not specified), in row order
            kept = calls[i]
            assert set(kept.tobytes()[j * 48:(j + 1) * 48] for j in range(cap)) <= set(full[i].tobytes()[j * 48:(j + 1) * 48]
                                                                                      for j in range(sizes[i])), i
            assert np.array_equal(np.sort(kept, order=["sample", "slot", "alt"]), kept), i
    for bad in (0, 9):
        rc = api.lib().as_call_variants_sweep_host(ctx._h, api._hp(tumours), T, P, api._hp(ref), api._hp(tv), bad, 100, api._hp(calls),
                                                   cap, api._hp(n))
        assert rc == -1, bad                   # AS_EINVAL


# ---- 3. / 4. the programs on the golden cases ------------------------------------------------------------------------
def run(prog, args, cwd, env=None):
    r = subprocess.run([str(BIN / prog)] + args, cwd=cwd, capture_output=True, text=True, env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    return r.stdout


def ee(case, c_text, out, cwd, env=None, germline="N"):
    return run("AmpliSolveErrorEstimation", ["panel_design=panel.bed", "reference_genome=ref.fa", f"germline_dir={germline}",
                                             f"C_value={c_text}", f"coverage_cutoff={int(case['cutoff'])}", "default_error=0.01",
                                             f"output_dir={out}"], cwd, env)


def vc(case, error_file, out, cwd, env=None, tumours="T"):
    return run("AmpliSolveVariantCalling", [f"errorFile={error_file}", f"tumour_dir={tumours}", f"output_dir={out}",
                                            f"coverage_cutoff={int(case['cutoff'])}", "p_value=0.05"], cwd, env)


def table_name(c):
    return "positionSpecificNoise_%.4f.txt" % np.float32(c)


def vc_outputs(d):
    """every file a caller run writes: VCFs without their ##fileDate line, the tumour list whatever its seed prefix"""
    d = Path(d)
    out = {}
    for p in sorted(d.rglob("*")):
        if p.is_dir():
            continue
        rel = str(p.relative_to(d))
        if rel.endswith("_tumour_count_list_original.txt"):
            rel = "tumour_count_list"
        text = p.read_text()
        out[rel] = "".join(l for l in text.splitlines(True) if not l.startswith("##fileDate")) if p.suffix == ".vcf" else text
    return out


def stage(case, td):
    slots = aseq_io.stage_case(td, case)
    aseq_io.write_fasta(td, slots, list(case["ref_letters"]))


@pytest.mark.parametrize("name", gu.CASES)
def test_error_estimation_sweep_on_golden_cases(name, tmp_path):
    case = gu.load(name)
    stage(case, tmp_path)
    own = float(case["c_value"])
    values = ["%g" % own, "0.001", "0.004", "0.005"]
    ee(case, ",".join(values), "sw", tmp_path)
    tables = sorted(p.name for p in (tmp_path / "sw").glob("positionSpecificNoise_*.txt"))
    assert tables == sorted({table_name(float(v)) for v in values})
    assert (tmp_path / "sw" / table_name(own)).read_text() == case["noise_table"]
    for v in values:
        ee(case, v, f"one_{v}", tmp_path)
        assert (tmp_path / "sw" / table_name(float(v))).read_text() == (tmp_path / f"one_{v}" / table_name(float(v))).read_text(), v
    interm = list((tmp_path / "sw" / "AmpliSolveErrorEstimation_interm_files").iterdir())
    assert len(interm) == 3          # panel bases, duplicated positions, normal list: written once
    # ten values: two passes of the sweep kernels
    ten = ["0.001", "0.0015", "0.002", "0.0025", "0.003", "0.0035", "0.004", "0.0045", "0.005", "0.0075"]
    ee(case, ",".join(ten), "ten", tmp_path)
    for v in ten:
        if not (tmp_path / f"one_{v}").exists():
            ee(case, v, f"one_{v}", tmp_path)
        assert (tmp_path / "ten" / table_name(float(v))).read_text() == (tmp_path / f"one_{v}" / table_name(float(v))).read_text(), v
    # rejected lists: a value twice under one table name, an empty element
    for bad in ("0.002,0.00201", "0.002,,0.003"):
        out = ee(case, bad, "bad", tmp_path)
        assert "Error" in out and bad in out
        assert not (tmp_path / "bad").exists()


def sweep_dir(case, td):
    """the four-table directory of the EE sweep (the case's own value first in name order or not)"""
    own = "%g" % float(case["c_value"])
    ee(case, f"{own},0.001,0.004,0.005", "sw", td)
    return sorted((td / "sw").glob("positionSpecificNoise_*.txt"))


def check_vc_sweep(case, td, out, tables):
    """every <out>/<stem>/ equals errorFile=sw/<stem>.txt run alone"""
    for t in tables:
        single = f"single_{t.stem}"
        if not (td / single).exists():
            vc(case, f"sw/{t.name}", single, td)
        assert vc_outputs(td / out / t.stem) == vc_outputs(td / single), t.name


@pytest.mark.parametrize("name", gu.CASES)
def test_variant_calling_sweep_on_golden_cases(name, tmp_path):
    case = gu.load(name)
    stage(case, tmp_path)
    tables = sweep_dir(case, tmp_path)
    vc(case, "sw", "vsw", tmp_path)
    assert sorted(p.name for p in (tmp_path / "vsw").iterdir()) == [t.stem for t in tables]
    check_vc_sweep(case, tmp_path, "vsw", tables)
    own = tmp_path / "vsw" / table_name(float(case["c_value"]))[:-4]
    assert (own / "Summary_Variant_Info.txt").read_text() == case["summary"]
    for nm in case["tumour_names"]:
        assert "".join(l for l in (own / f"{nm}.vcf").read_text().splitlines(True) if not l.startswith("##fileDate")) == case["vcfs"][nm]
    for env in ({"AS_GROUP_SAMPLES": "1"}, {"AS_WIRE": "16"}, {"AS_WIRE": "packed"}):
        tag = "_".join(env.values())
        vc(case, "sw", f"venv_{tag}", tmp_path, env)
        for t in tables:
            assert vc_outputs(tmp_path / f"venv_{tag}" / t.stem) == vc_outputs(tmp_path / "vsw" / t.stem), (env, t.name)


def test_variant_calling_sweep_rejects_another_panel_and_an_empty_directory(tmp_path):
    case = gu.load("synth_small")
    stage(case, tmp_path)
    tables = sweep_dir(case, tmp_path)
    lines = tables[1].read_text().splitlines(True)
    f = lines[5].split("\t")
    f[1] = str(int(f[1]) + 100000)              # another BED: a row at another position
    lines[5] = "\t".join(f)
    (tmp_path / "other").mkdir()
    (tmp_path / "other" / tables[0].name).write_text(tables[0].read_text())
    (tmp_path / "other" / tables[1].name).write_text("".join(lines))
    out = vc(case, "other", "vbad", tmp_path)
    assert tables[1].name in out and "line 6" in out
    assert not (tmp_path / "vbad").exists()
    (tmp_path / "none").mkdir()
    out = vc(case, "none", "vnone", tmp_path)
    assert "Cannot open none" in out
    assert not (tmp_path / "vnone").exists()


def _irregular():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_irregular", gu.GOLDEN / "make_irregular.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("fixture", ["irregular", "shuffled"])
def test_variant_calling_sweep_on_irregular_rows(fixture, tmp_path):
    """extra rows beyond a position's slots and RD-column rows (irregular_rows.npz), or tumour rows out of panel order"""
    mod = _irregular()
    case = gu.load("synth_small")
    stage(case, tmp_path)
    if fixture == "irregular":
        mod.apply_patches(tmp_path, case, ee_rd=False)
    else:
        mod.shuffle_rows(tmp_path, case)
    tables = sweep_dir(case, tmp_path)
    vc(case, "sw", "vsw", tmp_path, {"AS_GROUP_SAMPLES": "2"})
    check_vc_sweep(case, tmp_path, "vsw", tables)


# ---- 5. BAM input ----------------------------------------------------------------------------------------------------
def test_both_programs_sweep_on_bam_directories(tmp_path):
    bp.make_case(tmp_path, n_normals=4, n_tumours=3)
    values = ["0.001", "0.002", "0.004"]
    bp.run("AmpliSolveErrorEstimation", [a if not a.startswith("C_value=") else "C_value=" + ",".join(values) for a in bp.ee_args("sw")],
           tmp_path)
    for v in values:
        bp.run("AmpliSolveErrorEstimation", [a if not a.startswith("C_value=") else f"C_value={v}" for a in bp.ee_args(f"one_{v}")],
               tmp_path)
        assert (tmp_path / "sw" / table_name(float(v))).read_text() == (tmp_path / f"one_{v}" / table_name(float(v))).read_text()
    bp.run("AmpliSolveVariantCalling", bp.vc_args("sw", "vsw"), tmp_path, {"AS_GROUP_SAMPLES": "2"})
    for v in values:
        t = table_name(float(v))
        bp.run("AmpliSolveVariantCalling", bp.vc_args(f"sw/{t}", f"v_{v}"), tmp_path)
        assert vc_outputs(tmp_path / "vsw" / t[:-4]) == vc_outputs(tmp_path / f"v_{v}"), v


# ---- 6. the resident service -----------------------------------------------------------------------------------------
def test_sweep_programs_through_the_resident_service(tmp_path, socket_path):
    case = gu.load("synth_small")
    stage(case, tmp_path)
    tables = sweep_dir(case, tmp_path)
    vc(case, "sw", "vcold", tmp_path)
    srv = subprocess.Popen([str(BIN / "amplisolve_b200_serve"), f"socket={socket_path}"], cwd="/", stderr=subprocess.PIPE, text=True)
    try:
        assert "ready" in srv.stderr.readline()
        own = "%g" % float(case["c_value"])
        for rnd in range(2):
            env = {"AS_SERVER": socket_path}
            ee(case, f"{own},0.001,0.004,0.005", f"sws{rnd}", tmp_path, env)
            for t in tables:
                assert (tmp_path / f"sws{rnd}" / t.name).read_text() == t.read_text()
            vc(case, "sw", f"vs{rnd}", tmp_path, env)
            assert vc_outputs(tmp_path / f"vs{rnd}") == vc_outputs(tmp_path / "vcold")
        assert srv.poll() is None
    finally:
        srv.send_signal(signal.SIGTERM)
        srv.wait(timeout=20)


# ---- 7. several GPUs -------------------------------------------------------------------------------------------------
def test_sweep_on_two_gpus_equals_one(ctx, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")
    normals, tumours, ref, nxt, head = sweep_data()
    with api.Context([0, 1]) as multi:
        for fmt in FORMATS:
            counts, wide = encode(normals, fmt)
            a = ctx.estimate_thresholds_sweep(counts, C_VALUES[:5], 100, nxt, head, wide_records=wide)
            b = multi.estimate_thresholds_sweep(counts, C_VALUES[:5], 100, nxt, head, wide_records=wide)
            for k in a:
                assert np.array_equal(bits(a[k]), bits(b[k])), (fmt, k)
            tc, tw = encode(tumours, fmt)
            x = ctx.call_variants_sweep(tc, ref, a["thr_view"], 100, wide_records=tw)
            y = multi.call_variants_sweep(tc, ref, a["thr_view"], 100, wide_records=tw)
            assert [l.tobytes() for l in x] == [l.tobytes() for l in y], fmt
    case = gu.load("synth_small")
    stage(case, tmp_path)
    own = "%g" % float(case["c_value"])
    for tag, devs in (("one", "0"), ("two", "0,1")):
        ee(case, f"{own},0.001,0.004", f"o_{tag}", tmp_path, {"AS_DEVICES": devs})
        vc(case, f"o_{tag}", f"v_{tag}", tmp_path, {"AS_DEVICES": devs, "AS_GROUP_SAMPLES": "2"})
    for p in (tmp_path / "o_one").glob("positionSpecificNoise_*.txt"):
        assert (tmp_path / "o_two" / p.name).read_text() == p.read_text()
    assert vc_outputs(tmp_path / "v_two") == vc_outputs(tmp_path / "v_one")
