"""CPU tests of the product's host side: the C-ABI library loads and exports every symbol the header
declares, the parts of the two programs that need no GPU (usage text, default-error mode, hash order) behave
like the reference, and compute entry points fail loudly without a GPU."""
import re
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import pyoracle
from tests import aseq_io
from tests import golden_util as gu

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "amplisolve_b200" / "bin"


def test_library_exports_every_declared_symbol():
    import ctypes as C
    from amplisolve_b200 import api
    L = api.lib()
    header = (ROOT / "include" / "amplisolve_b200.h").read_text()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = sorted(set(re.findall(r"\b(as_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(L, name), f"{name} is declared in include/amplisolve_b200.h but not exported"
    assert set(api.EXPORTS) == set(declared)
    assert C.sizeof(api.SynthParams) == 56 and api.CALL_DTYPE.itemsize == 48


def test_no_cpu_fallback():
    import torch
    from amplisolve_b200 import AmpliSolveError, Context
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(AmpliSolveError, match="no CPU fallback|CUDA"):
        Context(0)


def test_hash_iteration_order_equals_libstdcxx_model():
    from amplisolve_b200 import hash_iteration_order
    rng = np.random.default_rng(3)
    for n in (1, 2, 3, 5, 12, 13, 29, 30, 97, 200):
        keys = [f"dir{n}/S{int(x):05d}_{i}.PILEUP.ASEQ" for i, x in enumerate(rng.integers(0, 99999, n))]
        assert hash_iteration_order(keys) == pyoracle.hash_iteration_order(keys)
    n5 = [f"N/N{i}.PILEUP.ASEQ" for i in range(1, 6)]
    assert [n5[i][2:4] for i in hash_iteration_order(n5)] == ["N5", "N3", "N2", "N4", "N1"]   # SURVEY.md A.5


def unpack_numpy(word):
    """numpy decoder of the packed wire format (include/amplisolve_b200.h), independent of the library's."""
    word = np.asarray(word, np.uint32)
    m, j = word & 0xFFFF, (word >> 16) & 3
    minors = np.stack([(word >> 18) & 15, (word >> 22) & 15, (word >> 26) & 15], -1)
    out = np.empty(word.shape + (4,), np.uint32)
    for b in range(4):
        k = np.where(b < j, b, b - 1).clip(0, 2)                 # index among the minors of base b when b != j
        out[..., b] = np.where(j == b, m, np.take_along_axis(minors, k[..., None], -1)[..., 0])
    out[word >= 0xFFFFFFFE] = 0xFFFFFFFF
    return out


def test_packed_wire_format_is_lossless():
    """as_pack_counts (the library's threaded encoder, host code) == the numpy statement of the format, and decoding the
    words + patching the escaped records gives back the uint32 tensor bit for bit."""
    from amplisolve_b200 import pack_counts, to_wire_packed
    from tests import synth
    rng = np.random.default_rng(8)
    _, slots, pos_id, U = synth.make_panel(20, seed=8)
    P = len(slots)
    counts, _ = synth.make_counts(9, P, depth=3000, seed=8, pos_id=pos_id, big_rate=0.02, somatic_rate=0.02)
    edge = np.array([[65535, 15, 15, 15], [15, 65535, 15, 15], [0, 0, 0, 0], [16, 16, 16, 16], [65536, 0, 0, 0], [1, 1, 1, 1],
                     [0, 16, 0, 70000], [15, 15, 15, 15], [0x7FFFFFFF, 0, 0, 0]], np.uint32)
    for i, e in enumerate(edge):
        counts[i % 9, rng.integers(0, 2), 3 + i] = e
    packed, wide = pack_counts(counts)
    ref_packed, ref_wide = to_wire_packed(counts)
    assert np.array_equal(packed, ref_packed) and wide.tobytes() == ref_wide.tobytes()
    assert 0 < len(wide) < counts.shape[0] * P // 4
    back = unpack_numpy(packed)
    assert (back[wide["sample"], 0, wide["slot"]] == 0xFFFFFFFF).all()     # escaped words decode as absent until patched
    back[wide["sample"], 0, wide["slot"]] = wide["fw"]
    back[wide["sample"], 1, wide["slot"]] = wide["bw"]
    assert np.array_equal(back, counts)
    # capacity protocol: too small a list reports the count and AS_EOVERFLOW
    import ctypes as C
    from amplisolve_b200 import api
    n = C.c_int64(0)
    small = np.zeros(1, api.WIDE_DTYPE)
    rc = api.lib().as_pack_counts(counts.ctypes.data_as(C.c_void_p), counts.shape[0], P, packed.ctypes.data_as(C.c_void_p),
                                  small.ctypes.data_as(C.c_void_p), 1, C.byref(n))
    assert rc == -5 and n.value == len(wide)


def test_critical_means_table_and_prescreen_bound():
    """AS_MCRIT of as_call.cuh is what scripts/critical_means.py computes (m*(k)(1 + 1e-9), P(X >= k | m*) = P*), the
    reference's own p (oracle) is above P* at the table value and at most P* a hair below the critical mean, and the
    scan's bound K - 9/16 >= AS_MCRIT[K-1] holds for K = 1..64."""
    import sys
    sys.path.insert(0, str(ROOT / "scripts"))
    from critical_means import critical_means
    want = critical_means()
    src = (ROOT / "amplisolve_b200" / "csrc" / "as_call.cuh").read_text()
    body = src[src.index("AS_MCRIT[64] = {") + len("AS_MCRIT[64] = {"):]
    body = body[:body.index("};")]
    have = [float(x) for x in body.replace("\n", " ").split(",") if x.strip()]
    assert have == want and len(have) == 64
    p_star = np.frombuffer(np.uint64(0x3FD43D136248490E).tobytes(), dtype=np.float64)[0]
    err = np.float32(2.0 ** -20)
    for k in range(1, 65):
        assert have[k - 1] <= k - 9 / 16
        above = int(np.ceil(have[k - 1] * 2 ** 20))                   # the first depth whose mean is >= the table value
        below = int(np.floor(have[k - 1] / (1 + 1e-9) * (1 - 3e-6) * 2 ** 20))
        assert pyoracle.poisson_p(k, above, err) > p_star
        assert pyoracle.poisson_p(k, below, err) <= p_star


def test_twin_links():
    from amplisolve_b200 import twin_links
    nxt, head = twin_links([0, 1, 2, 1, 3, 0, 1])
    assert nxt.tolist() == [5, 3, -1, 6, -1, -1, -1]
    assert head.tolist() == [0, 1, 2, 1, 4, 0, 1]


@pytest.mark.parametrize("prog,n", [("AmpliSolveErrorEstimation", 8), ("AmpliSolveVariantCalling", 6)])
def test_usage_on_wrong_argc_returns_zero(prog, n):
    """EE:266-273, VC:216-223: wrong argc prints the usage text and returns 0."""
    r = subprocess.run([str(BIN / prog), "x=1"], capture_output=True, text=True)
    assert r.returncode == 0
    assert "Your input arguments are not correct" in r.stdout and "Please type the following" in r.stdout


@pytest.mark.parametrize("name", gu.CASES)
def test_default_error_mode_is_byte_identical(name, tmp_path):
    """germline_dir=not_available (EE:349, EE:472-506, EE:2948-3043): BED enumeration, reference bases read from
    the .fai-indexed FASTA, duplicated positions -- no GPU involved."""
    case = gu.load(name)
    slots = aseq_io.stage_case(tmp_path, case)
    aseq_io.write_fasta(tmp_path, slots, list(case["ref_letters"]))
    r = subprocess.run([str(BIN / "AmpliSolveErrorEstimation"), "panel_design=panel.bed", "reference_genome=ref.fa",
                        "germline_dir=not_available", "C_value=0.002", "coverage_cutoff=100", "default_error=0.02",
                        "output_dir=od"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout
    got = (tmp_path / "od" / "positionSpecificNoise_default.txt").read_text()
    assert got == case["default_table"]
    interm = list((tmp_path / "od" / "AmpliSolveErrorEstimation_interm_files").glob("*_panelReferenceBases.txt"))
    assert len(interm) == 1 and interm[0].read_text() == (tmp_path / "rb_ref.txt").read_text()
    dups = list((tmp_path / "od" / "AmpliSolveErrorEstimation_interm_files").glob("*_ampliconDuplicatedPositions.txt"))
    assert sorted(dups[0].read_text().splitlines()) == sorted((tmp_path / "rb_dup.txt").read_text().splitlines())


def test_noise_mode_without_gpu_fails_loudly(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    case = gu.load("synth_small")
    slots = aseq_io.stage_case(tmp_path, case)
    aseq_io.write_fasta(tmp_path, slots, list(case["ref_letters"]))
    r = subprocess.run([str(BIN / "AmpliSolveErrorEstimation"), "panel_design=panel.bed", "reference_genome=ref.fa",
                        "germline_dir=N", "C_value=0.0035", "coverage_cutoff=150", "default_error=0.01", "output_dir=o"],
                       cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode != 0 and "no CPU fallback" in r.stdout
    assert not list((tmp_path / "o").glob("positionSpecificNoise_0*.txt"))


def test_compute_counts_reads_the_container_and_fails_loudly_without_gpu(tmp_path):
    """computeCounts (SURVEY.md 8 f4): usage and container errors need no GPU; a valid BAM without a GPU is an error that
    says so -- there is no CPU pileup behind the program."""
    import torch
    from tests import bam_io
    prog = str(BIN / "computeCounts")
    r = subprocess.run([prog], capture_output=True, text=True)
    assert r.returncode == 0 and "Usage: computeCounts" in r.stdout
    (tmp_path / "positions.txt").write_text("chr1\t1000\t.\t.\t.\n")
    (tmp_path / "x.bam").write_bytes(b"plain text, not BGZF" * 4)
    r = subprocess.run([prog, "vcf=positions.txt", "bam=x.bam", "out=o"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 1 and "not a BGZF" in r.stdout
    read = dict(ref_id=0, pos=990, mapq=60, flag=0, cigar=[("M", 30)], seq="ACGT" * 7 + "AC", qual=bytes([30]) * 30)
    bam_io.write_bam(tmp_path / "ok.bam", [("chr1", 5000)], [read] * 25)
    r = subprocess.run([prog, "vcf=positions.txt", "bam=ok.bam", "out=o"], cwd=tmp_path, capture_output=True, text=True)
    if torch.cuda.is_available():
        assert r.returncode == 0
        rows = (tmp_path / "o" / "ok.PILEUP.ASEQ").read_text().splitlines()
        assert rows[1].split("\t")[:2] == ["chr1", "1000"] and rows[1].split("\t")[10] == "25"
    else:
        assert r.returncode == 1 and "no CPU fallback" in r.stdout
        assert not (tmp_path / "o" / "ok.PILEUP.ASEQ").exists()


def test_resident_service_runs_the_programs_for_its_clients(tmp_path, socket_path):
    """amplisolve_b200_serve + AS_SERVER: argv, working directory, stdout / stderr and the exit status travel; the output is
    the one of a run in the program's own process; no service listening -> the program runs by itself.  (Default-error mode
    and usage errors need no GPU, so the plumbing is tested here; the GPU paths through the service in test_gpu_golden.py.)"""
    import os
    import signal
    import time
    case = gu.load("synth_small")
    slots = aseq_io.stage_case(tmp_path, case)
    aseq_io.write_fasta(tmp_path, slots, list(case["ref_letters"]))
    args = [str(BIN / "AmpliSolveErrorEstimation"), "panel_design=panel.bed", "reference_genome=ref.fa", "germline_dir=not_available",
            "C_value=0.002", "coverage_cutoff=100", "default_error=0.02"]
    sock = socket_path
    env = dict(os.environ, AS_SERVER=sock)
    # nobody listens: the program runs by itself
    r0 = subprocess.run(args + ["output_dir=alone"], cwd=tmp_path, capture_output=True, text=True, env=env)
    assert r0.returncode == 0 and (tmp_path / "alone" / "positionSpecificNoise_default.txt").read_text() == case["default_table"]
    srv = subprocess.Popen([str(BIN / "amplisolve_b200_serve"), f"socket={sock}"], cwd="/", stderr=subprocess.PIPE, text=True,
                           env=dict(os.environ, AS_SERVE_NO_WARMUP="1"))
    try:
        assert "ready" in srv.stderr.readline()
        r1 = subprocess.run(args + ["output_dir=served"], cwd=tmp_path, capture_output=True, text=True, env=env)
        assert r1.returncode == 0
        assert (tmp_path / "served" / "positionSpecificNoise_default.txt").read_text() == case["default_table"]
        strip = lambda t: re.sub(r"(alone|served)", "X", t)   # noqa: E731
        assert strip(r1.stdout) == strip(r0.stdout) and "Running function" in r1.stdout      # the client's stdout got the program's text
        r2 = subprocess.run(args[:2], cwd=tmp_path, capture_output=True, text=True, env=env)  # wrong argc: usage, status 0
        assert r2.returncode == 0 and "Your input arguments are not correct" in r2.stdout
        r3 = subprocess.run([str(BIN / "computeCounts"), "vcf=nope.txt", "bam=nope.bam"], cwd=tmp_path, capture_output=True, text=True, env=env)
        assert r3.returncode == 1 and "Cannot open file" in r3.stdout                           # exit status travels
        # several clients at once: served one after the other, each with its own directory and output
        from concurrent.futures import ThreadPoolExecutor
        def one(k):
            return subprocess.run(args + [f"output_dir=par{k}"], cwd=tmp_path, capture_output=True, text=True, env=env).returncode
        with ThreadPoolExecutor(4) as pool:
            assert list(pool.map(one, range(4))) == [0, 0, 0, 0]
        for k in range(4):
            assert (tmp_path / f"par{k}" / "positionSpecificNoise_default.txt").read_text() == case["default_table"]
        assert srv.poll() is None
    finally:
        srv.send_signal(signal.SIGTERM)
        srv.wait(timeout=10)


def test_shard_bounds_keep_twin_groups_whole():
    """as_shard_bounds (what as_create_multi contexts split a panel by): contiguous, covering, and no twin group straddles a
    boundary -- also with a group that spans almost the whole panel; equal to amplisolve_b200.shard.shard_ranges."""
    import numpy as np
    from amplisolve_b200 import shard_bounds, twin_links
    from amplisolve_b200.shard import shard_ranges
    from tests import synth
    for seed, n in ((1, 2), (2, 3), (3, 8)):
        _, slots, pos_id, U = synth.make_panel(70, seed=seed, overlap_frac=0.6, amp_len=(20, 70))
        pos_id = pos_id.copy()
        if seed == 3:
            pos_id[-5] = pos_id[300]
        nxt, head = twin_links(pos_id)
        P = len(slots)
        b = shard_bounds(P, n, nxt, head)
        assert b[0] == 0 and b[-1] == P and all(x <= y for x, y in zip(b, b[1:]))
        for cut in b[1:-1]:
            assert not np.any((head[cut:] < cut)), cut          # no member at or after the cut belongs to a group that starts before it
        assert [(b[i], b[i + 1]) for i in range(n)] == shard_ranges(P, n, head, nxt)
    assert shard_bounds(1000, 4) == [0, 128, 384, 640, 1000] or shard_bounds(1000, 4)[-1] == 1000


def test_aseq_loader_fast_and_general_paths_agree(tmp_path):
    """The ASEQ loader (as_host.cpp parse_aseq) has a fast row scanner for the usual row shape and a general parser for
    everything sscanf("%s %s %s %s %s %s %d ...") of the reference accepts (EE:1149, VC:752).  The same counts written with
    tabs, with CRLF line ends, with runs of blanks instead of tabs, with blank lines in between and with the rows in reverse
    order must give the same packed tensor (scripts/parse_bench.cpp: the loader alone, no GPU; checksum over all words)."""
    import json
    import numpy as np
    from tests import synth
    exe = _build_parse_bench(tmp_path)
    bed, slots, pos_id, U = synth.make_panel(30, seed=9)
    P = len(slots)
    counts, _ = synth.make_counts(5, P, depth=3000, seed=9, pos_id=pos_id)
    counts[1, 0, 3, :] = [70000, 1, 0, 2]            # escapes the packed format
    counts[2, 1, 5, :] = [123456789, 0, 17, 2]       # nine digits: beyond the vector scanner's eight
    counts[3, 0, 7, :] = [99999999, 3, 0, 0]         # eight digits
    counts[3, 1, 7, :] = [0, 0, 0, 0]
    (tmp_path / "panel.bed").write_text("".join(f"{c}\t{s}\t{e}\tA{i}\n" for i, (c, s, e) in enumerate(bed)))

    def variant(name, transform):
        d = tmp_path / name
        d.mkdir()
        for i in range(counts.shape[0]):
            aseq_io.write_aseq(d / f"S{i}.PILEUP.ASEQ", slots, counts[i])
            text = (d / f"S{i}.PILEUP.ASEQ").read_text()
            head, rows = text.split("\n", 1)
            (d / f"S{i}.PILEUP.ASEQ").write_text(head + "\n" + transform(rows))
        got = []
        for scan in ("scalar", "avx2"):  # the byte-wise row scanner and the vector one (taken when the CPU has AVX2)
            out = subprocess.run([str(exe), str(tmp_path / "panel.bed"), str(d), "1"], capture_output=True, text=True,
                                 env=dict(os.environ, AS_ROW_SCAN=scan))
            assert out.returncode == 0, out.stderr
            res = json.loads(out.stdout)
            got.append((res["checksum"], res["rows"], res["escaped"], res["outside"]))
        assert got[0] == got[1], (name, got)
        return got[0]

    base = variant("tabs", lambda t: t)
    assert base[1] == int((counts[:, 0, :, 0] != 0xFFFFFFFF).sum()) and base[2] >= 1 and base[3] == 0
    assert variant("crlf", lambda t: t.replace("\n", "\r\n")) == base
    assert variant("blanks", lambda t: t.replace("\t", "   ")) == base
    assert variant("blank_lines", lambda t: t.replace("\n", "\n\n")) == base
    assert variant("reversed", lambda t: "\n".join(t.strip("\n").split("\n")[::-1]) + "\n") == base
    assert variant("no_final_newline", lambda t: t.rstrip("\n")) == base


_PARSE_BENCH = []


def _build_parse_bench(tmp_path):
    """scripts/parse_bench.cpp (as_host.cpp's host logic behind a small command line), built once per test session."""
    import shutil
    import tempfile
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    if _PARSE_BENCH:
        return _PARSE_BENCH[0]
    exe = Path(tempfile.mkdtemp(prefix="as_parse_bench_")) / "parse_bench"
    lib_dir = ROOT / "amplisolve_b200" / "lib"
    from amplisolve_b200 import lib
    lib()
    r = subprocess.run(["g++", "-O1", "-std=c++17", "-pthread", "-I", str(ROOT / "include"), str(ROOT / "scripts" / "parse_bench.cpp"),
                        f"-L{lib_dir}", "-lamplisolve_b200", f"-Wl,-rpath,{lib_dir}", "-Wl,-rpath,/usr/local/cuda/lib64", "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    _PARSE_BENCH.append(exe)
    return exe


def test_noise_table_parser_in_pieces_equals_an_independent_reading(tmp_path):
    """The caller program reads the noise table (storeInputFile, VC:430-576) in pieces on all host threads, with its own
    decimal -> float conversion for the cells "%f" writes (as_host.cpp parse_noise_table, threshold_text_to_float).  Whatever
    the number of pieces, every row must hold what a plain reading of the table gives: chromosome ids in order of first
    appearance, position, texts, flag, std::stof of the eight threshold parts (compared as float bit patterns against
    numpy's correctly rounded conversion), the Germ_Max texts, the twin links of repeated positions and the dummy VCF."""
    import json
    import numpy as np
    exe = _build_parse_bench(tmp_path)
    table = str(np.load(ROOT / "tests" / "golden" / "toy_slice.npz", allow_pickle=True)["noise_table"])
    head, body = table.split("\n", 1)
    rows = [r for r in body.split("\n") if r.strip()]
    # cells the golden table does not hold: empty parts, a second underscore, exponents, nan, many digits, blanks, CRLF
    odd = ["chrZ\t77\tN\tNO\t_0.5\t1e-05_2.5e-3\tnan_inf\t0.123456789_12345678.5\t-\t0\t1.5\t-888",
           "chrZ  78 \t A  YES\t0.25_\t-2_-2\t0.01_0.01\t0.000001_9.999999\t-\t-\t-\t-\r",
           "chr8\t77\tC\tNO\t0.1_0.2_0.3\t7_8\t.5_5.\t-0.000000_0.000000\t1\t2\t3\t4",
           "chrZ\t77\tG\tYES\t1_1\t1_1\t1_1\t1_1\t-\t-\t-\t-"]
    rows = rows[:1500] + odd[:2] + rows[1500:] + odd[2:]
    path = tmp_path / "table.txt"
    path.write_text(head + "\n" + "\n".join(rows) + "\n\n")

    # the independent reading
    chrom_ids, first, last, expect, dummy = {}, {}, {}, [], []
    heads, nexts = [], []
    for i, r in enumerate(rows):
        f = r.split()
        f += [""] * (12 - len(f))
        cid = chrom_ids.setdefault(f[0], len(chrom_ids))
        bits = []
        for cell in f[4:8]:
            parts = cell.split("_")
            for part in (parts[:2] if len(parts) >= 2 else ["", ""]):
                v = np.float32(0) if part == "" else np.float32(part)
                bits.append("%08x" % np.array(v, np.float32).view(np.uint32))
        key = (cid, int(f[1]))
        heads.append(first.setdefault(key, i))
        nexts.append(-1)
        if key in last:
            nexts[last[key]] = i
        last[key] = i
        expect.append([str(cid), f[0], f[1], f[1], f[2] or "~", "1" if f[3] == "YES" else "0"] + bits + [g or "~" for g in f[8:12]])
        dummy.append(f"{f[0]}\t{f[1]}\t.\t.\t.\t.\t.\t.\n")
    for i in range(len(rows)):
        expect[i] += [str(heads[i]), str(nexts[i]), str(heads[i])]

    for pieces in (1, 2, 7, 64, 0):
        dump = tmp_path / f"dump{pieces}.txt"
        out = subprocess.run([str(exe), "--noise-table", str(path), str(pieces), str(dump)], capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        res = json.loads(out.stdout)
        assert res["rows"] == len(rows) and res["positions"] == len(first)
        got, got_dummy = dump.read_text().split("DUMMY\n")
        got = [g.split(" ") for g in got.strip("\n").split("\n")]
        assert len(got) == len(expect)
        for g, x in zip(got, expect):
            assert g == x, (pieces, g, x)
        assert got_dummy == "".join(dummy)


def test_noise_table_writer_percent_f_equals_printf(tmp_path):
    """The noise-table writer formats "%f" of a float threshold (EE:1787) itself: v * 10^6 is exact in a double, rint() is the
    round-half-even printf performs (as_host.cpp append_percent_f).  Against snprintf: every float of the thresholds' range
    with a stride, the neighbourhood of the 6-decimal ties, both zeros, negative values, huge values, nan and inf."""
    import json
    exe = _build_parse_bench(tmp_path)
    for first, last, stride in ((0x00000000, 0x3D800000, 211),       # 0 .. 0.0625
                                (0x3A800000, 0x3A810000, 1),         # every float around 0.001
                                (0x3D800000, 0x4A000000, 4099),      # 0.0625 .. 2^21 (the fall-back from 2^20 on)
                                (0x7F700000, 0x80000100, 101) ):     # huge, inf, nan, -0, negative denormals
        out = subprocess.run([str(exe), "--percent-f", hex(first), hex(last), str(stride)], capture_output=True, text=True)
        res = json.loads(out.stdout)
        assert out.returncode == 0 and res["differences"] == 0 and res["tried"] > 50000, res


def test_row_scanners_agree_with_the_general_parser_on_random_rows(tmp_path):
    """as_host.cpp has three readers of an ASEQ row (EE:1149, VC:752): the vector scanner (AVX2: bit masks of one 64-byte
    window, ten numbers converted in vector lanes), the byte-wise scanner and the general sscanf-like parser.  A faster one
    may decline a row, never read it differently: random rows with positions up to 2^31, counts of up to ten digits, long
    chromosome names, CRLF ends and tokens in the unused columns."""
    import json
    exe = _build_parse_bench(tmp_path)
    out = subprocess.run([str(exe), "--row-scan", "300000", "11"], capture_output=True, text=True)
    res = json.loads(out.stdout)
    assert out.returncode == 0 and res["differences"] == 0, res
    assert res["bytewise_scanner_took"] > 250000, res


def test_noise_table_writer_percent_g_equals_printf(tmp_path):
    """The Germ_Max cells of the noise table are ostream << double = "%g" (EE:2815); the writer formats the values of
    [1e-4, 1) itself, exactly (integer round-half-even of m * 10^D / 2^s: as_host.cpp append_percent_g), and leaves the rest to
    snprintf.  Against snprintf: the whole range with a stride, every float around the decade boundaries 1e-4, 1e-3, 1e-2,
    1e-1 and 1 (where the number of decimals changes and 9.999995 rounds into the next decade), and values it must decline."""
    import json
    import struct
    exe = _build_parse_bench(tmp_path)

    def bits(x):
        return struct.unpack("<I", struct.pack("<f", x))[0]

    out = subprocess.run([str(exe), "--percent-g", hex(bits(1e-4) - 5000), hex(bits(1.0) + 5000), "613"], capture_output=True, text=True)
    res = json.loads(out.stdout)
    assert out.returncode == 0 and res["differences"] == 0 and res["tried"] - res["declined"] > 150000, res
    for edge in (1e-4, 1e-3, 1e-2, 1e-1, 1.0, 0.05, 0.0123455, 0.00999995):
        out = subprocess.run([str(exe), "--percent-g", hex(bits(edge) - 20000), hex(bits(edge) + 20000), "1"], capture_output=True, text=True)
        res = json.loads(out.stdout)
        assert out.returncode == 0 and res["differences"] == 0, (edge, res)
    out = subprocess.run([str(exe), "--percent-g", hex(bits(-888.0) - 50), hex(bits(-888.0) + 50), "1"], capture_output=True, text=True)
    res = json.loads(out.stdout)
    assert out.returncode == 0 and res["declined"] == res["tried"], res


def test_host_thread_pool_under_concurrent_phases(tmp_path):
    """as_host.cpp runs every parallel phase on one pool of host threads that stay (HostPool); a phase that finds the pool busy
    starts threads of its own.  Three threads starting 15,000 phases between them: every item of every phase runs exactly once
    and nothing hangs."""
    import json
    exe = _build_parse_bench(tmp_path)
    out = subprocess.run([str(exe), "--pool-stress", "5000"], capture_output=True, text=True, timeout=300)
    res = json.loads(out.stdout)
    assert out.returncode == 0 and res["bad"] == 0 and res["phases"] == 15000, res


def test_noise_table_threshold_text_to_float_equals_strtof(tmp_path):
    """The caller program reads a threshold cell through std::stof (VC:889-890); as_host.cpp converts texts of the form
    [-]digits[.digits] with at most eight digits itself -- double(n) / 10^s narrowed to float is the correctly rounded float --
    and leaves the rest to strtof.  Against strtof: every "%f" text below 2.0, and random texts incl. longer ones, exponents
    and words."""
    import json
    exe = _build_parse_bench(tmp_path)
    out = subprocess.run([str(exe), "--stof", "2000000", "5"], capture_output=True, text=True)
    res = json.loads(out.stdout)
    assert out.returncode == 0 and res["differences"] == 0 and res["tried"] > 4000000, res
