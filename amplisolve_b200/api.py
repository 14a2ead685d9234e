"""ctypes face of libamplisolve_b200.so (include/amplisolve_b200.h).

The function names mirror the reference code each one replaces:

    Context.estimate_thresholds   estimateThresholds + the Germ_Max part of storeGermlineStatistics
                                  (AmpliSolveErrorEstimation.cpp:1484-2544, :1247-1467)
    Context.thresholds_caller_view  the "%f" -> std::stof hand-over (EE:1787 -> VC:889-890)
    Context.call_variants         the row loop of callVariants (AmpliSolveVariantCalling.cpp:723-3296)
    Context.site_tests            VC:895-898 for listed sites in every tumour, called or not
    Context.mutation_rules_poisson_quality_score   VC:3834-3884, element-wise
    Context.kf_gammaq             VC:3726, element-wise

Host arrays are numpy, device arrays are torch CUDA tensors (torch is used for device memory and
streams only).  There is no CPU fallback: without the built library or without a B200 every compute
call raises AmpliSolveError.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

ABSENT = 0xFFFFFFFF
CALL_DTYPE = np.dtype([("sample", "<i4"), ("slot", "<i4"), ("alt", "<i4"), ("ref", "<i4"), ("p_fw", "<f8"),
                       ("p_bw", "<f8"), ("q_fw", "<f8"), ("q_bw", "<f8")])
assert CALL_DTYPE.itemsize == 48
# as_site_test and its statuses (include/amplisolve_b200.h)
SITE_TEST_DTYPE = np.dtype([("depth_fw", "<u4"), ("depth_bw", "<u4"), ("alt_fw", "<u4"), ("alt_bw", "<u4"), ("p_fw", "<f8"),
                            ("p_bw", "<f8"), ("status", "<i4"), ("pad", "<i4")])
assert SITE_TEST_DTYPE.itemsize == 40
SITE_CALLED, SITE_NOT_CALLED, SITE_LOW_COVERAGE, SITE_NO_DATA, SITE_NOT_TESTABLE = 1, 2, 3, 4, 5

EXPORTS = [
    "as_last_error", "as_version", "as_device_count", "as_create", "as_create_multi", "as_context_devices", "as_shard_bounds", "as_destroy", "as_host_alloc", "as_host_free",
    "as_set_call_kernel", "as_set_noise_kernel", "as_set_host_tile_slots", "as_set_option", "as_kernel_launches", "as_noise_estimate_dev", "as_noise_estimate_host",
    "as_noise_estimate_host16", "as_thresholds_caller_view_dev", "as_call_variants_dev", "as_call_variants_host",
    "as_call_variants_host16", "as_sort_calls_dev", "as_call_variants_sweep_dev", "as_noise_estimate_sweep_dev", "as_pack_counts", "as_noise_estimate_host_packed", "as_call_variants_host_packed",
    "as_noise_estimate_sweep_host", "as_noise_estimate_sweep_host16", "as_noise_estimate_sweep_host_packed", "as_call_variants_sweep_host",
    "as_call_variants_sweep_host16", "as_call_variants_sweep_host_packed", "as_site_tests_host", "as_site_tests_host16",
    "as_site_tests_host_packed", "as_poisson_test_host",
    "as_kf_gammaq_host", "as_synth_counts_dev", "as_synth_twin_links_dev", "as_hash_iteration_order", "as_fisher_test", "as_fisher_tests_host", "as_error_estimation_main",
    "as_variant_calling_main", "as_pileup_begin", "as_pileup_add_host", "as_pileup_end_host", "as_pileup_end_wire", "as_pileup_set_host", "as_compute_counts_main", "as_serve_main", "as_client_run", "as_process_is_resident",
]


class AmpliSolveError(RuntimeError):
    pass


WIDE_DTYPE = np.dtype([("sample", "<i4"), ("slot", "<i4"), ("fw", "<u4", (4,)), ("bw", "<u4", (4,))])
assert WIDE_DTYPE.itemsize == 40
WIRE_ABSENT, WIRE_ESCAPE = 0xFFFF, 0xFFFE


def to_wire16(counts):
    """uint32 [S][2][P][4] -> (uint16 wire tensor, wide records) of the _host16 entry points (include/amplisolve_b200.h):
    absent records are 0xFFFF, records with a count >= 65534 are escaped (0xFFFE) into the side list sorted by slot."""
    counts = np.asarray(counts, dtype=np.uint32)
    absent = counts[:, 0, :, 0] == ABSENT                                       # [S][P]
    big = (~absent) & ((counts[:, 0] >= WIRE_ESCAPE).any(-1) | (counts[:, 1] >= WIRE_ESCAPE).any(-1))
    out = counts.astype(np.uint16)
    out[:, 0][absent] = WIRE_ABSENT
    out[:, 1][absent] = WIRE_ABSENT
    out[:, 0][big] = WIRE_ESCAPE
    out[:, 1][big] = WIRE_ESCAPE
    smp, slot = np.nonzero(big)
    wide = np.zeros(len(smp), dtype=WIDE_DTYPE)
    wide["sample"], wide["slot"] = smp, slot
    wide["fw"], wide["bw"] = counts[smp, 0, slot], counts[smp, 1, slot]
    return out, np.sort(wide, order=["slot", "sample"])


PACKED_ABSENT, PACKED_ESCAPE = 0xFFFFFFFF, 0xFFFFFFFE


def to_wire_packed(counts):
    """uint32 [S][2][P][4] -> (packed uint32 [S][2][P], wide records): numpy statement of the packed wire format of the
    _host_packed entry points (include/amplisolve_b200.h); as_pack_counts is the library's own (threaded) encoder."""
    counts = np.asarray(counts, dtype=np.uint32)
    absent = counts[:, 0, :, 0] == ABSENT                                       # [S][P]
    j = counts.argmax(-1)                                                       # first maximum = lowest base index on ties
    major = np.take_along_axis(counts, j[..., None], -1)[..., 0]
    others = np.array([[1, 2, 3], [0, 2, 3], [0, 1, 3], [0, 1, 2]])[j]          # [S][2][P][3]
    minor = np.take_along_axis(counts, others, -1)
    fits = (major <= 0xFFFF) & (minor <= 15).all(-1)
    word = (major | (j.astype(np.uint32) << 16) | (minor[..., 0] << 18) | (minor[..., 1] << 22) | (minor[..., 2] << 26)).astype(np.uint32)
    escaped = (~absent) & ~(fits[:, 0] & fits[:, 1])
    for st in (0, 1):
        word[:, st][escaped] = PACKED_ESCAPE
        word[:, st][absent] = PACKED_ABSENT
    smp, slot = np.nonzero(escaped)
    wide = np.zeros(len(smp), dtype=WIDE_DTYPE)
    wide["sample"], wide["slot"] = smp, slot
    wide["fw"], wide["bw"] = counts[smp, 0, slot], counts[smp, 1, slot]
    return word, np.sort(wide, order=["slot", "sample"])


def pack_counts(counts):
    """as_pack_counts: uint32 [S][2][P][4] -> (packed uint32 [S][2][P], wide records sorted by (slot, sample))."""
    counts = _np(counts, np.uint32)
    S, two, P, four = counts.shape
    assert two == 2 and four == 4
    packed = np.empty((S, 2, P), np.uint32)
    cap = max(1024, S * P // 64)
    while True:
        wide = np.zeros(cap, dtype=WIDE_DTYPE)
        n = C.c_int64(0)
        rc = lib().as_pack_counts(_hp(counts), S, P, _hp(packed), _hp(wide), cap, C.byref(n))
        if rc == -5:
            cap = int(n.value)
            continue
        _check(rc)
        return packed, wide[:n.value]


class SynthParams(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("mean_depth", C.c_float), ("depth_sigma", C.c_float),
                ("germline_rate", C.c_float), ("somatic_rate", C.c_float), ("somatic_vaf_lo", C.c_float),
                ("somatic_vaf_hi", C.c_float), ("absent_rate", C.c_float), ("sample_offset", C.c_int32),
                ("slot_offset", C.c_int64), ("twin_period", C.c_int32), ("reserved", C.c_int32)]


_lib = None


def lib_path() -> Path:
    return Path(__file__).resolve().parent / "lib" / "libamplisolve_b200.so"


def lib():
    """Load (building first if the sources are newer) the shared library.  Never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build as _build
    try:
        path = _build.build()
    except Exception as exc:  # no nvcc (e.g. the GPU box): use the prebuilt library that travelled with the tree
        path = lib_path()
        if not path.exists():
            raise AmpliSolveError(f"libamplisolve_b200.so is missing and cannot be built: {exc}") from exc
    L = C.CDLL(str(path))
    vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
    L.as_last_error.restype = C.c_char_p
    L.as_version.restype = C.c_char_p
    L.as_device_count.argtypes = [C.POINTER(C.c_int)]
    L.as_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.as_create_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    L.as_context_devices.argtypes = [vp, C.POINTER(C.c_int), C.c_int]
    L.as_shard_bounds.argtypes = [i64, i32, vp, vp, vp]
    L.as_destroy.argtypes = [vp]
    L.as_destroy.restype = None
    L.as_host_alloc.argtypes = [C.POINTER(vp), C.c_size_t]
    L.as_host_free.argtypes = [vp]
    L.as_set_call_kernel.argtypes = [vp, C.c_int]
    L.as_set_noise_kernel.argtypes = [vp, C.c_int]
    L.as_set_host_tile_slots.argtypes = [vp, i64]
    L.as_set_option.argtypes = [vp, C.c_char_p, i64]
    L.as_kernel_launches.argtypes = [vp]
    L.as_kernel_launches.restype = i64
    L.as_noise_estimate_dev.argtypes = [vp, vp, i32, i64, i64, i64, vp, vp, f32, i32, vp, vp, vp, vp, vp, vp]
    L.as_noise_estimate_sweep_dev.argtypes = [vp, vp, i32, i64, i64, i64, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp]
    L.as_noise_estimate_host.argtypes = [vp, vp, i32, i64, vp, vp, f32, i32, vp, vp, vp, vp, vp, vp]
    L.as_noise_estimate_host16.argtypes = [vp, vp, vp, i64, i32, i64, vp, vp, f32, i32, vp, vp, vp, vp, vp, vp]
    L.as_thresholds_caller_view_dev.argtypes = [vp, vp, vp, i64, vp]
    L.as_call_variants_dev.argtypes = [vp, vp, i32, i64, i64, i64, vp, vp, i32, vp, i64, vp, vp]
    L.as_call_variants_sweep_dev.argtypes = [vp, vp, i32, i64, i64, i64, vp, vp, i32, i32, vp, i64, vp, vp]
    L.as_call_variants_host.argtypes = [vp, vp, i32, i64, vp, vp, i32, vp, i64, C.POINTER(i64)]
    L.as_sort_calls_dev.argtypes = [vp, vp, i64, i32, vp, vp]
    L.as_call_variants_host16.argtypes = [vp, vp, vp, i64, i32, i64, vp, vp, i32, vp, i64, C.POINTER(i64)]
    L.as_noise_estimate_host_packed.argtypes = L.as_noise_estimate_host16.argtypes
    L.as_call_variants_host_packed.argtypes = L.as_call_variants_host16.argtypes
    L.as_noise_estimate_sweep_host.argtypes = [vp, vp, i32, i64, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp]
    L.as_noise_estimate_sweep_host16.argtypes = [vp, vp, vp, i64, i32, i64, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp]
    L.as_noise_estimate_sweep_host_packed.argtypes = L.as_noise_estimate_sweep_host16.argtypes
    L.as_call_variants_sweep_host.argtypes = [vp, vp, i32, i64, vp, vp, i32, i32, vp, i64, vp]
    L.as_call_variants_sweep_host16.argtypes = [vp, vp, vp, i64, i32, i64, vp, vp, i32, i32, vp, i64, vp]
    L.as_call_variants_sweep_host_packed.argtypes = L.as_call_variants_sweep_host16.argtypes
    L.as_site_tests_host.argtypes = [vp, vp, i32, i64, vp, vp, i32, vp, vp, i64, i32, vp]
    L.as_site_tests_host16.argtypes = [vp, vp, vp, i64, i32, i64, vp, vp, i32, vp, vp, i64, i32, vp]
    L.as_site_tests_host_packed.argtypes = L.as_site_tests_host16.argtypes
    L.as_pack_counts.argtypes = [vp, i32, i64, vp, vp, i64, C.POINTER(i64)]
    L.as_poisson_test_host.argtypes = [vp, vp, vp, vp, i64, vp, vp]
    L.as_kf_gammaq_host.argtypes = [vp, vp, vp, i64, vp]
    L.as_synth_counts_dev.argtypes = [vp, vp, i32, i64, vp, C.POINTER(SynthParams), vp]
    L.as_synth_twin_links_dev.argtypes = [vp, i64, C.POINTER(SynthParams), vp, vp, vp]
    L.as_hash_iteration_order.argtypes = [C.POINTER(C.c_char_p), i32, vp]
    L.as_fisher_tests_host.argtypes = [vp, vp, i64, vp]
    L.as_fisher_test.restype = C.c_double
    L.as_fisher_test.argtypes = [i32, i32, i32, i32]
    L.as_pileup_begin.argtypes = [vp, vp, i32, vp, i64]
    L.as_pileup_add_host.argtypes = [vp, vp, i64, vp, i64, vp, i32, i32, i32, C.c_uint32]
    L.as_pileup_end_host.argtypes = [vp, vp, vp]
    L.as_pileup_end_wire.argtypes = [vp, vp, i64, i32, i32, i32, vp, vp, i64, C.POINTER(i64), C.POINTER(i64), vp]
    L.as_pileup_set_host.argtypes = [vp, vp]
    for name in ("as_error_estimation_main", "as_variant_calling_main", "as_compute_counts_main"):
        if hasattr(L, name):
            getattr(L, name).argtypes = [C.c_int, C.POINTER(C.c_char_p)]
    _lib = L
    return L


def _check(rc: int, allow_overflow: bool = False) -> int:
    if rc == 0 or (allow_overflow and rc == -5):
        return rc
    raise AmpliSolveError(f"amplisolve_b200 error {rc}: {lib().as_last_error().decode(errors='replace')}")


def _np(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _hp(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _dp(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def hash_iteration_order(keys) -> list:
    """Order in which libstdc++ iterates an unordered_map<string,string> filled with `keys`
    (the reference's file order, EE:1081 / VC:672).  Host-only, needs no GPU."""
    arr = (C.c_char_p * len(keys))(*[k.encode() for k in keys])
    out = np.empty(max(1, len(keys)), dtype=np.int32)
    n = lib().as_hash_iteration_order(arr, len(keys), _hp(out))
    if n < 0:
        raise AmpliSolveError("as_hash_iteration_order failed")
    return [int(i) for i in out[:n]]


def fisher_test(fw: int, bw: int, alt_fw: int, alt_bw: int) -> float:
    """fisherTest(FW, BW, alt_fw, alt_bw) of VC:3797-3814 (host arithmetic of the variant-calling program)."""
    return float(lib().as_fisher_test(int(fw), int(bw), int(alt_fw), int(alt_bw)))


def shard_bounds(n_slots: int, n_shards: int, twin_next=None, twin_head=None) -> list:
    """as_shard_bounds: the slot ranges a multi-device context splits a panel into (twin groups kept whole)."""
    out = np.zeros(n_shards + 1, dtype=np.int64)
    tn = None if twin_next is None else _np(twin_next, np.int32)
    th = None if twin_head is None else _np(twin_head, np.int32)
    _check(lib().as_shard_bounds(int(n_slots), int(n_shards), None if tn is None else _hp(tn), None if th is None else _hp(th), _hp(out)))
    return [int(x) for x in out]


def twin_links(pos_id) -> tuple[np.ndarray, np.ndarray]:
    """twin_next / twin_head arrays from a slot -> unique-position map (slots in panel order)."""
    pos_id = np.asarray(pos_id)
    P = len(pos_id)
    nxt = np.full(P, -1, dtype=np.int32)
    head = np.arange(P, dtype=np.int32)
    last: dict = {}
    for p in range(P):
        u = int(pos_id[p])
        if u in last:
            nxt[last[u]] = p
            head[p] = head[last[u]]
        last[u] = p
    return nxt, head


def _host_format(counts) -> str:
    a = np.asarray(counts)
    if a.dtype == np.uint16:
        return "u16"
    return "packed" if a.ndim == 3 else "u32"


class Context:
    """One per device (as_ctx)."""

    def __init__(self, device=0):
        """device: one ordinal (as_create) or a list of ordinals (as_create_multi: the host entry points shard the panel's
        slots over them; device-resident entry points use the first)."""
        self._h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            arr = (C.c_int * len(device))(*device)
            self.device = int(device[0])
            _check(lib().as_create_multi(arr, len(device), C.byref(self._h)))
        else:
            self.device = device
            _check(lib().as_create(device, C.byref(self._h)))

    def close(self):
        if self._h:
            for p, _ in self.__dict__.pop("_pool", {}).values():
                lib().as_host_free(p)
            lib().as_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def kernel_launches(self) -> int:
        return int(lib().as_kernel_launches(self._h))

    def set_call_kernel(self, variant: int):
        _check(lib().as_set_call_kernel(self._h, variant))

    def set_noise_kernel(self, variant: int):
        _check(lib().as_set_noise_kernel(self._h, variant))

    def set_host_tile_slots(self, slots: int):
        _check(lib().as_set_host_tile_slots(self._h, slots))

    def set_option(self, name: str, value: int):
        _check(lib().as_set_option(self._h, name.encode(), int(value)))

    # ---- host-buffer entry points --------------------------------------------------------------
    def _pinned_array(self, name, shape, dtype):
        """a numpy view of pinned host memory owned by this context, reused by the next call that asks for `name`"""
        nbytes = max(16, int(np.prod(shape)) * np.dtype(dtype).itemsize)
        pool = self.__dict__.setdefault("_pool", {})
        have = pool.get(name)
        if have is None or have[1] < nbytes:
            if have is not None:
                lib().as_host_free(have[0])
            p = C.c_void_p()
            _check(lib().as_host_alloc(C.byref(p), nbytes))
            pool[name] = have = (p, nbytes)
        buf = (C.c_char * nbytes).from_address(have[0].value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def estimate_thresholds(self, counts, c_value, coverage_cutoff, twin_next=None, twin_head=None, wide_records=None,
                            with_view=False, pinned_outputs=False):
        """counts: uint32 [S][2][P][4] host array, the uint16 wire format [S][2][P][4] with its wide_records (to_wire16)
        or the packed wire format uint32 [S][2][P] with its wide_records (pack_counts); normals in the reference's file
        order."""
        fmt = _host_format(counts)
        wide = fmt == "u32"
        counts = _np(counts, np.uint16 if fmt == "u16" else np.uint32)
        wr = _np(wide_records if wide_records is not None else np.zeros(0, WIDE_DTYPE), WIDE_DTYPE)
        S, two, P = counts.shape[:3]
        assert two == 2 and (fmt == "packed" or counts.shape[3] == 4)
        # pinned_outputs: the arrays live in pinned memory owned by the context (the D2H copies of the tile pipeline are
        # then truly asynchronous) and are OVERWRITTEN by the next call with pinned_outputs
        new = (lambda name, shape, dt: self._pinned_array(name, shape, dt)) if pinned_outputs else (lambda name, shape, dt: np.empty(shape, dt))
        out = {"thr": new("thr", (P, 4, 2), np.float32), "germ_val": new("germ_val", (P, 4), np.float32),
               "germ_state": new("germ_state", (P, 4), np.uint8), "count": new("count", (P, 4), np.uint32),
               "nrec": new("nrec", (P,), np.uint32)}
        view = new("thr_view", (P, 4, 2), np.float32) if with_view else None
        tn = th = None
        if twin_next is not None:
            tn, th = _np(twin_next, np.int32), _np(twin_head, np.int32)
        tail = (None if tn is None else _hp(tn), None if th is None else _hp(th), np.float32(c_value), int(coverage_cutoff),
                _hp(out["thr"]), _hp(out["germ_val"]), _hp(out["germ_state"]), _hp(out["count"]), _hp(out["nrec"]),
                None if view is None else _hp(view))
        if wide:
            _check(lib().as_noise_estimate_host(self._h, _hp(counts), S, P, *tail))
        else:
            fn = lib().as_noise_estimate_host16 if fmt == "u16" else lib().as_noise_estimate_host_packed
            _check(fn(self._h, _hp(counts), _hp(wr), len(wr), S, P, *tail))
        if view is not None:
            out["thr_view"] = view   # thresholds as the caller parses them ("%f" text round trip, -1_-1 -> 0.01)
        return out

    def call_variants(self, counts, ref, thr_view, coverage_cutoff, cap=None, wide_records=None, pinned_outputs=False):
        """counts: uint32 [T][2][P][4] host array, or one of the two wire formats with its wide_records (see
        estimate_thresholds).  Returns calls sorted by (sample, slot, alt)."""
        fmt = _host_format(counts)
        wide = fmt == "u32"
        counts = _np(counts, np.uint16 if fmt == "u16" else np.uint32)
        wr = _np(wide_records if wide_records is not None else np.zeros(0, WIDE_DTYPE), WIDE_DTYPE)
        T, two, P = counts.shape[:3]
        assert two == 2 and (fmt == "packed" or counts.shape[3] == 4)
        ref = _np(ref, np.uint8)
        thr_view = _np(thr_view, np.float32)
        assert ref.shape == (P,) and thr_view.shape == (P, 4, 2)
        if cap is None:
            cap = max(1024, T * P // 8)
        # only the first n entries are written and returned; pinned_outputs: see estimate_thresholds
        calls = self._pinned_array("calls", (cap,), CALL_DTYPE) if pinned_outputs else np.empty(cap, dtype=CALL_DTYPE)
        n = C.c_int64(0)
        tail = (T, P, _hp(ref), _hp(thr_view), int(coverage_cutoff), _hp(calls), cap, C.byref(n))
        if wide:
            rc = lib().as_call_variants_host(self._h, _hp(counts), *tail)
        else:
            fn = lib().as_call_variants_host16 if fmt == "u16" else lib().as_call_variants_host_packed
            rc = fn(self._h, _hp(counts), _hp(wr), len(wr), *tail)
        _check(rc, allow_overflow=True)
        if rc == -5:
            return self.call_variants(counts, ref, thr_view, coverage_cutoff, cap=int(n.value), wide_records=wide_records,
                                      pinned_outputs=pinned_outputs)
        return calls[:n.value]

    def estimate_thresholds_sweep(self, counts, c_values, coverage_cutoff, twin_next=None, twin_head=None, wide_records=None):
        """Noise-floor sweep on the host path (as_noise_estimate_sweep_host*): the dict of estimate_thresholds(with_view=True)
        with thr / thr_view of shape [n_c][P][4][2], table i bit for bit that of c_values[i].  One upload of counts."""
        fmt = _host_format(counts)
        counts = _np(counts, np.uint16 if fmt == "u16" else np.uint32)
        wr = _np(wide_records if wide_records is not None else np.zeros(0, WIDE_DTYPE), WIDE_DTYPE)
        cv = _np(c_values, np.float32).reshape(-1)
        S, two, P = counts.shape[:3]
        assert two == 2 and (fmt == "packed" or counts.shape[3] == 4)
        n_c = len(cv)
        out = {"thr": np.empty((n_c, P, 4, 2), np.float32), "germ_val": np.empty((P, 4), np.float32),
               "germ_state": np.empty((P, 4), np.uint8), "count": np.empty((P, 4), np.uint32), "nrec": np.empty(P, np.uint32),
               "thr_view": np.empty((n_c, P, 4, 2), np.float32)}
        tn = th = None
        if twin_next is not None:
            tn, th = _np(twin_next, np.int32), _np(twin_head, np.int32)
        tail = (None if tn is None else _hp(tn), None if th is None else _hp(th), _hp(cv), n_c, int(coverage_cutoff),
                _hp(out["thr"]), _hp(out["germ_val"]), _hp(out["germ_state"]), _hp(out["count"]), _hp(out["nrec"]),
                _hp(out["thr_view"]))
        if fmt == "u32":
            _check(lib().as_noise_estimate_sweep_host(self._h, _hp(counts), S, P, *tail))
        else:
            fn = lib().as_noise_estimate_sweep_host16 if fmt == "u16" else lib().as_noise_estimate_sweep_host_packed
            _check(fn(self._h, _hp(counts), _hp(wr), len(wr), S, P, *tail))
        return out

    def call_variants_sweep(self, counts, ref, thr_views, coverage_cutoff, cap=None, wide_records=None):
        """Caller sweep on the host path (as_call_variants_sweep_host*): thr_views [n_c][P][4][2]; returns one call array
        per table, each what call_variants returns for that table.  One upload of counts."""
        fmt = _host_format(counts)
        counts = _np(counts, np.uint16 if fmt == "u16" else np.uint32)
        wr = _np(wide_records if wide_records is not None else np.zeros(0, WIDE_DTYPE), WIDE_DTYPE)
        T, two, P = counts.shape[:3]
        assert two == 2 and (fmt == "packed" or counts.shape[3] == 4)
        ref = _np(ref, np.uint8)
        thr_views = _np(thr_views, np.float32)
        n_c = thr_views.shape[0]
        assert ref.shape == (P,) and thr_views.shape == (n_c, P, 4, 2)
        if cap is None:
            cap = max(1024, T * P // 8)
        calls = np.empty((n_c, cap), dtype=CALL_DTYPE)
        n = np.zeros(n_c, np.int64)
        tail = (T, P, _hp(ref), _hp(thr_views), n_c, int(coverage_cutoff), _hp(calls), cap, _hp(n))
        if fmt == "u32":
            rc = lib().as_call_variants_sweep_host(self._h, _hp(counts), *tail)
        else:
            fn = lib().as_call_variants_sweep_host16 if fmt == "u16" else lib().as_call_variants_sweep_host_packed
            rc = fn(self._h, _hp(counts), _hp(wr), len(wr), *tail)
        _check(rc, allow_overflow=True)
        if rc == -5:
            return self.call_variants_sweep(counts, ref, thr_views, coverage_cutoff, cap=int(n.max()), wide_records=wide_records)
        return [calls[i, :n[i]].copy() for i in range(n_c)]

    def site_tests(self, counts, ref, thr_view, coverage_cutoff, site_slot, site_alt, wide_records=None):
        """Site report (as_site_tests_host*): the strand tests of the listed sites (site_slot[i], site_alt[i]) in every tumour,
        called or not.  counts / wide_records as in call_variants, thr_view [P][4][2] or [n_c][P][4][2].  Returns a
        SITE_TEST_DTYPE array [n_c][T][H]: strand depths, alt reads, p_fw / p_bw (NaN where not evaluated) and status
        (SITE_CALLED is the caller's decision)."""
        fmt = _host_format(counts)
        counts = _np(counts, np.uint16 if fmt == "u16" else np.uint32)
        wr = _np(wide_records if wide_records is not None else np.zeros(0, WIDE_DTYPE), WIDE_DTYPE)
        T, two, P = counts.shape[:3]
        assert two == 2 and (fmt == "packed" or counts.shape[3] == 4)
        ref = _np(ref, np.uint8)
        tv = _np(thr_view, np.float32)
        tv = tv.reshape((-1, P, 4, 2)) if tv.size or P == 0 else tv.reshape((0, P, 4, 2))
        n_c = tv.shape[0]
        slot, alt = _np(site_slot, np.int32).reshape(-1), _np(site_alt, np.int32).reshape(-1)
        assert ref.shape == (P,) and slot.shape == alt.shape
        H = len(slot)
        out = np.zeros((n_c, T, H), SITE_TEST_DTYPE)
        tail = (T, P, _hp(ref), _hp(tv), n_c, _hp(slot), _hp(alt), H, int(coverage_cutoff), _hp(out))
        if fmt == "u32":
            _check(lib().as_site_tests_host(self._h, _hp(counts), *tail))
        else:
            fn = lib().as_site_tests_host16 if fmt == "u16" else lib().as_site_tests_host_packed
            _check(fn(self._h, _hp(counts), _hp(wr), len(wr), *tail))
        return out

    def mutation_rules_poisson_quality_score(self, k, rd, err):
        k, rd, err = _np(k, np.int32), _np(rd, np.int32), _np(err, np.float32)
        p, q = np.empty(k.shape, np.float64), np.empty(k.shape, np.float64)
        _check(lib().as_poisson_test_host(self._h, _hp(k), _hp(rd), _hp(err), k.size, _hp(p), _hp(q)))
        return p, q

    def fisher_tests(self, tables):
        """tables [n][4] = (FW, BW, alt_fw, alt_bw) -> p [n]: fisherTest of VC:3797-3814 for every row, on the device."""
        tables = _np(tables, np.int32).reshape(-1, 4)
        p = np.empty(len(tables), np.float64)
        _check(lib().as_fisher_tests_host(self._h, _hp(tables), len(tables), _hp(p)))
        return p

    def kf_gammaq(self, s, z):
        s, z = _np(s, np.float64), _np(z, np.float64)
        out = np.empty(s.shape, np.float64)
        _check(lib().as_kf_gammaq_host(self._h, _hp(s), _hp(z), s.size, _hp(out)))
        return out

    # ---- device-resident entry points (torch CUDA tensors) -------------------------------------
    @staticmethod
    def _stream(stream=None):
        import torch
        return C.c_void_p((stream or torch.cuda.current_stream()).cuda_stream)

    def alloc_noise_outputs(self, P):
        import torch
        dev = f"cuda:{self.device}"
        return {"thr": torch.empty((P, 4, 2), dtype=torch.float32, device=dev),
                "germ_val": torch.empty((P, 4), dtype=torch.float32, device=dev),
                "germ_state": torch.empty((P, 4), dtype=torch.uint8, device=dev),
                "count": torch.empty((P, 4), dtype=torch.int32, device=dev),
                "nrec": torch.empty(P, dtype=torch.int32, device=dev)}

    def estimate_thresholds_dev(self, counts, c_value, coverage_cutoff, out, twin_next=None, twin_head=None,
                                slot_range=None, stream=None):
        """counts: torch int32 CUDA tensor [S][2][P][4] (bit pattern of the uint32 counts)."""
        S, two, P, four = counts.shape
        b, e = slot_range if slot_range is not None else (0, P)
        _check(lib().as_noise_estimate_dev(self._h, _dp(counts), S, P, b, e, _dp(twin_next), _dp(twin_head),
                                           np.float32(c_value), int(coverage_cutoff), _dp(out["thr"]),
                                           _dp(out["germ_val"]), _dp(out["germ_state"]), _dp(out["count"]),
                                           _dp(out["nrec"]), self._stream(stream)))
        return out

    def thresholds_caller_view_dev(self, thr, view=None, stream=None):
        import torch
        if view is None:
            view = torch.empty_like(thr)
        _check(lib().as_thresholds_caller_view_dev(self._h, _dp(thr), _dp(view), thr.numel(), self._stream(stream)))
        return view

    def estimate_thresholds_sweep_dev(self, counts, c_values, coverage_cutoff, thr, out, twin_next=None, twin_head=None,
                                      slot_range=None, stream=None):
        """Noise-floor sweep: thr torch float32 [n_c][P][4][2] receives one threshold table per C value; out (as from
        alloc_noise_outputs) the outputs that do not depend on C (its "thr" entry is not written)."""
        S, two, P, four = counts.shape
        cv = _np(c_values, np.float32)
        assert thr.shape == (len(cv), P, 4, 2) and thr.is_contiguous()
        b, e = slot_range if slot_range is not None else (0, P)
        _check(lib().as_noise_estimate_sweep_dev(self._h, _dp(counts), S, P, b, e, _dp(twin_next), _dp(twin_head), _hp(cv),
                                                 len(cv), int(coverage_cutoff), _dp(thr), _dp(out["germ_val"]),
                                                 _dp(out["germ_state"]), _dp(out["count"]), _dp(out["nrec"]),
                                                 self._stream(stream)))

    def call_variants_dev(self, counts, ref, thr_view, coverage_cutoff, calls, n_calls, slot_range=None, stream=None):
        """calls: torch uint8 CUDA tensor of cap*48 bytes; n_calls: torch int64 CUDA tensor [1] (added to)."""
        T, two, P, four = counts.shape
        b, e = slot_range if slot_range is not None else (0, P)
        cap = calls.numel() * calls.element_size() // CALL_DTYPE.itemsize
        _check(lib().as_call_variants_dev(self._h, _dp(counts), T, P, b, e, _dp(ref), _dp(thr_view),
                                          int(coverage_cutoff), _dp(calls), cap, _dp(n_calls), self._stream(stream)))

    def call_variants_sweep_dev(self, counts, ref, thr_views, coverage_cutoff, calls, n_calls, slot_range=None, stream=None):
        """Noise-floor sweep: thr_views torch float32 [n_c][P][4][2]; calls torch uint8 CUDA tensor of n_c*cap*48 bytes
        (list ci at [ci*cap, (ci+1)*cap)); n_calls torch int64 CUDA tensor [n_c] (added to).  One pass over counts."""
        T, two, P, four = counts.shape
        n_c = thr_views.shape[0]
        assert thr_views.shape == (n_c, P, 4, 2) and thr_views.is_contiguous() and n_calls.numel() == n_c
        b, e = slot_range if slot_range is not None else (0, P)
        cap = calls.numel() * calls.element_size() // CALL_DTYPE.itemsize // n_c
        _check(lib().as_call_variants_sweep_dev(self._h, _dp(counts), T, P, b, e, _dp(ref), _dp(thr_views), n_c,
                                                int(coverage_cutoff), _dp(calls), cap, _dp(n_calls), self._stream(stream)))
        return cap

    def sort_calls_dev(self, calls, n, sorted_out, slot_offset=0, stream=None):
        """calls / sorted_out: torch uint8 CUDA tensors of >= n*48 bytes; the first n calls of `calls` get slot_offset added
        and land in sorted_out in the reference's row order (sample, slot, alt)."""
        _check(lib().as_sort_calls_dev(self._h, _dp(calls), int(n), int(slot_offset), _dp(sorted_out), self._stream(stream)))

    def pileup(self, pieces, ref_contig, contig_first, slot_pos, mbq=20, mrq=20, skip_flags=0x704):
        """BAM records -> counts uint32 [2 strands][P][4 bases] of one sample (as_pileup_*).  pieces: iterable of
        (records uint8 array, rec_off int64 array) of the uncompressed record stream; ref_contig[refID] = panel contig or -1;
        the panel as sorted unique 0-based positions slot_pos[contig_first[c]:contig_first[c+1]].  Returns (counts, (reads
        used, bases counted))."""
        first = np.ascontiguousarray(contig_first, np.int64)
        pos = np.ascontiguousarray(slot_pos, np.int32)
        refc = np.ascontiguousarray(ref_contig, np.int32)
        P = len(pos)
        _check(lib().as_pileup_begin(self._h, first.ctypes.data, len(first) - 1, pos.ctypes.data, P))
        for rec, off in pieces:
            rec = np.ascontiguousarray(rec, np.uint8)
            off = np.ascontiguousarray(off, np.int64)
            _check(lib().as_pileup_add_host(self._h, rec.ctypes.data, len(rec), off.ctypes.data, len(off), refc.ctypes.data, len(refc),
                                            int(mbq), int(mrq), int(skip_flags)))
        counts = np.zeros((2, P, 4), np.uint32)
        stats = np.zeros(2, np.uint64)
        _check(lib().as_pileup_end_host(self._h, counts.ctypes.data, stats.ctypes.data))
        return counts, (int(stats[0]), int(stats[1]))

    def pileup_end_wire(self, slot_unique, mdc, fmt="packed", sample=0, wide_cap=None, counts=None):
        """as_pileup_end_wire: ends the open pileup in the wire form of one sample of the programs' host tensor.  slot_unique
        [P] = position (0..U-1) of every panel slot; a slot whose depth is below mdc is absent.  counts: uint32 [2][U][4]
        put in place of the pileup's counts first (as_pileup_set_host; a pileup over positions 0..U-1 of one contig is opened
        for them).  fmt "packed" -> wire uint32 [2][P], "16" -> uint16 [2][P][4].  Returns (wire, wide records sorted by slot,
        present slots, (reads used, bases counted)).  More than wide_cap (default P) escaped records raise AmpliSolveError
        with .code -5 and .n_wide = the true count; the pileup then stays open."""
        slot_unique = np.ascontiguousarray(slot_unique, np.int32)
        P = len(slot_unique)
        if counts is not None:
            counts = _np(counts, np.uint32)
            U = counts.shape[1]
            first = np.array([0, U], np.int64)
            pos = np.arange(U, dtype=np.int32)
            _check(lib().as_pileup_begin(self._h, first.ctypes.data, 1, pos.ctypes.data, U))
            _check(lib().as_pileup_set_host(self._h, counts.ctypes.data))
        f = {"packed": 1, "16": 2}[fmt]
        wire = np.empty((2, P), np.uint32) if f == 1 else np.empty((2, P, 4), np.uint16)
        cap = P if wide_cap is None else int(wide_cap)
        wide = np.zeros(max(cap, 1), dtype=WIDE_DTYPE)
        n, rows = C.c_int64(0), C.c_int64(0)
        stats = np.zeros(2, np.uint64)
        rc = lib().as_pileup_end_wire(self._h, slot_unique.ctypes.data, P, int(mdc), f, int(sample), wire.ctypes.data, wide.ctypes.data, cap,
                                      C.byref(n), C.byref(rows), stats.ctypes.data)
        if rc != 0:
            err = AmpliSolveError(f"amplisolve_b200 error {rc}: {lib().as_last_error().decode(errors='replace')}")
            err.code, err.n_wide = rc, int(n.value)
            raise err
        return wire, wide[:n.value], int(rows.value), (int(stats[0]), int(stats[1]))

    def synth_counts_dev(self, n_samples, P, *, seed, mean_depth, somatic_rate=0.0, sample_offset=0, slot_offset=0,
                         depth_sigma=0.5, germline_rate=1e-3, vaf=(0.01, 0.2), absent_rate=0.0, want_ref=True,
                         twin_period=0, stream=None):
        """Synthetic panel generated in HBM (SURVEY.md 8d).  Returns (counts int32 [n][2][P][4], ref uint8 [P])."""
        import torch
        dev = f"cuda:{self.device}"
        counts = torch.empty((n_samples, 2, P, 4), dtype=torch.int32, device=dev)
        ref = torch.empty(P, dtype=torch.uint8, device=dev) if want_ref else None
        prm = SynthParams(seed, mean_depth, depth_sigma, germline_rate, somatic_rate, vaf[0], vaf[1], absent_rate,
                          sample_offset, slot_offset, twin_period, 0)
        _check(lib().as_synth_counts_dev(self._h, _dp(counts), n_samples, P, _dp(ref), C.byref(prm),
                                         self._stream(stream)))
        return counts, ref

    def synth_twin_links_dev(self, P, *, seed, slot_offset=0, twin_period=6, stream=None):
        """twin_next / twin_head (int32 CUDA tensors [P]) of the synthetic panel geometry."""
        import torch
        dev = f"cuda:{self.device}"
        nxt = torch.empty(P, dtype=torch.int32, device=dev)
        head = torch.empty(P, dtype=torch.int32, device=dev)
        prm = SynthParams(seed, 0, 0, 0, 0, 0, 0, 0, 0, slot_offset, twin_period, 0)
        _check(lib().as_synth_twin_links_dev(self._h, P, C.byref(prm), _dp(nxt), _dp(head), self._stream(stream)))
        return nxt, head


def calls_from_device(calls, n_calls) -> np.ndarray:
    """Download a device call list and sort it into the reference's row order."""
    n = int(n_calls.item())
    cap = calls.numel() * calls.element_size() // CALL_DTYPE.itemsize
    if n > cap:
        raise AmpliSolveError(f"call list overflow: {n} calls, capacity {cap}")
    raw = calls.view(-1)[: n * CALL_DTYPE.itemsize].cpu().numpy().view(CALL_DTYPE)
    return sort_calls(raw)


def sort_calls(calls: np.ndarray) -> np.ndarray:
    """Reference row order: sample (file), slot (row), alt (AmpliSolveVariantCalling.cpp:672, :869-3288)."""
    return calls[np.lexsort((calls["alt"], calls["slot"], calls["sample"]))]
