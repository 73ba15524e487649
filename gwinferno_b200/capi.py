"""ctypes binding of libgwi.so (include/gwi.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is present, the
calls raise :class:`GwiError` -- they never route to NumPy.
"""

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GWI_LIBRARY", os.path.join(_HERE, "libgwi.so"))  # override: another build of the library, e.g. to compare two builds on the same GPU

GWI_VERSION = 5  # include/gwi.h: GWI_VERSION (device-resident catalogs, device plan builder, plan timings in gwi_model_info)
GWI_LIKE_HEADER = 8
LIKE_FIELDS = ("log_l", "passed", "log_mu", "logNeff_inj", "min_logNeff", "sum_logBF", "variance", "status")
PARTIAL_HEADER = 8


class GwiError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libgwi error {code}: {msg}")
        self.code = code


class gwi_term(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("feature", C.c_int32),
        ("outside", C.c_int32),
        ("logx", C.c_int32),
        ("col", C.c_int32 * 2),
        ("slot", C.c_int32 * 6),
        ("cst", C.c_double * 4),
        ("n_splines", C.c_int32),
        ("norm_group", C.c_int32),
        ("x_lo", C.c_double),
        ("x_hi", C.c_double),
        ("xi_lo", C.c_double),
        ("xi_hi", C.c_double),
        ("grid", C.POINTER(C.c_double)),
        ("knots", C.POINTER(C.c_double)),
        ("n_knots", C.c_int32),
        ("order", C.c_int32),
    ]


class gwi_norm_group(C.Structure):
    _fields_ = [("n_grid", C.c_int32), ("log_w", C.POINTER(C.c_double))]


class gwi_cut(C.Structure):
    _fields_ = [("kind", C.c_int32), ("col", C.c_int32 * 2), ("lo", C.c_double), ("hi", C.c_double)]


class gwi_nuts_opts(C.Structure):
    _fields_ = [("n_warmup", C.c_int32), ("n_samples", C.c_int32), ("max_depth", C.c_int32), ("flags", C.c_int32), ("seed", C.c_int64), ("target_accept", C.c_double)]


class gwi_nuts_info(C.Structure):
    _fields_ = [
        ("step_size", C.c_double),
        ("mean_accept", C.c_double),
        ("sampling_seconds", C.c_double),
        ("leapfrogs_sampling", C.c_int64),
        ("leapfrogs_total", C.c_int64),
        ("n_evals", C.c_int64),
    ]


class gwi_prior_block(C.Structure):
    _fields_ = [("first", C.c_int32), ("count", C.c_int32), ("sigma", C.c_double), ("tau", C.c_double), ("diff_degree", C.c_int32), ("fix_first_zero", C.c_int32)]


# double (*)(void* ctx, const double* theta, double* grad)
POTENTIAL_FN = C.CFUNCTYPE(C.c_double, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double))


class gwi_model_desc(C.Structure):
    _fields_ = [
        ("n_terms", C.c_int32),
        ("terms", C.POINTER(gwi_term)),
        ("n_groups", C.c_int32),
        ("groups", C.POINTER(gwi_norm_group)),
        ("n_cuts", C.c_int32),
        ("cuts", C.POINTER(gwi_cut)),
        ("n_params", C.c_int32),
        ("need_neff_grad", C.c_int32),
        ("chunk_steps", C.c_int32),
        ("n_deep", C.c_int32),
        ("batch_hint", C.c_int32),
        ("keep_sample_index", C.c_int32),
    ]


class gwi_catalog_desc(C.Structure):
    _fields_ = [
        ("n_columns", C.c_int32),
        ("n_events", C.c_int32),
        ("pe_offsets", C.POINTER(C.c_int64)),
        ("pe_columns", C.POINTER(C.POINTER(C.c_double))),
        ("n_inj", C.c_int64),
        ("inj_columns", C.POINTER(C.POINTER(C.c_double))),
        ("total_inj", C.c_double),
        ("device", C.c_int32),
        ("columns_on_device", C.c_int32),
    ]


class gwi_outputs(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("logBF", "logNeff", "log_mu", "logNeff_inj", "J_logBF", "J_logNeff", "J_log_mu", "J_logNeff_inj", "logZ")]


class gwi_like_opts(C.Structure):
    _fields_ = [("Nobs", C.c_int32), ("marginalize_selection", C.c_int32), ("min_neff_cut", C.c_int32), ("max_variance_cut", C.c_int32)]


class gwi_model_info(C.Structure):
    _fields_ = [
        ("n_samples_pe", C.c_int64),
        ("n_samples_inj", C.c_int64),
        ("n_valid_pe", C.c_int64),
        ("n_valid_inj", C.c_int64),
        ("n_padded", C.c_int64),
        ("bytes_per_eval", C.c_int64),
        ("n_chunks", C.c_int32),
        ("n_stream_columns", C.c_int32),
        ("n_spline_dims", C.c_int32),
        ("n_deep", C.c_int32),
        ("n_linear", C.c_int32),
        ("n_param_terms", C.c_int32),
        ("grid_blocks", C.c_int32),
        ("block_threads", C.c_int32),
        ("kernel_launches_per_eval", C.c_int32),
        ("active_switches", C.c_int32),
        ("plan_on_device", C.c_int32),
        ("reserved_", C.c_int32),
        ("plan_seconds", C.c_double * 5),
    ]


# every symbol include/gwi.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "gwi_comm_local_handle",
    "gwi_comm_connect",
    "gwi_loglike_sharded",
    "gwi_sharded_push",
    "gwi_sharded_combine",
    "gwi_model_last_sites",
    "gwi_sample_log_weights",
    "gwi_draw_samples",
    "gwi_catalog_create",
    "gwi_catalog_destroy",
    "gwi_model_create",
    "gwi_model_destroy",
    "gwi_eval",
    "gwi_loglike",
    "gwi_loglike_host",
    "gwi_loglike_batch",
    "gwi_loglike_batch_host",
    "gwi_partial_size",
    "gwi_partial",
    "gwi_combine",
    "gwi_model_get_info",
    "gwi_model_batch_hint",
    "gwi_model_set_exact_shift",
    "gwi_model_set_timing",
    "gwi_model_stream_times",
    "gwi_last_error",
    "gwi_version",
    "gwi_debug_plan_build",
    "gwi_debug_plan_destroy",
    "gwi_debug_plan_read",
    "gwi_debug_model_read",
    "gwi_synth_injections",
    "gwi_device_minmax",
    "gwi_nuts_sample",
    "gwi_posterior_create",
    "gwi_posterior_destroy",
    "gwi_posterior_dim",
    "gwi_posterior_potential",
    "gwi_nuts_sample_posterior",
    "gwi_nuts_sample_posterior_chains",
]

_lib = None
_cudart = None


def load_library(_allow_emulator=False):
    """Load libgwi.so (built in-tree by ``__graft_entry__.build()`` / ``make -C gwinferno_b200/csrc``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GwiError(-2, f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` " "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    if hasattr(lib, "gwi_emu_marker") and not _allow_emulator:
        # tests/emu builds the kernel sources for a host warp emulator (CPU test suite only)
        raise GwiError(-2, f"{LIB_PATH} is the test suite's host-emulator build, not the CUDA library (there is no CPU path)")
    if lib.gwi_version() != GWI_VERSION:  # the structs below would not match the library's
        raise GwiError(-1, f"{LIB_PATH} has ABI version {lib.gwi_version()}, this binding expects {GWI_VERSION}: rebuild it")
    lib.gwi_last_error.restype = C.c_char_p
    lib.gwi_partial_size.restype = C.c_int64
    lib.gwi_partial_size.argtypes = [C.c_void_p]
    lib.gwi_debug_plan_read.restype = C.c_int64
    lib.gwi_debug_plan_read.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64]
    lib.gwi_synth_injections.argtypes = [C.c_int32, C.c_uint64, C.c_int64, C.c_int64, C.POINTER(C.c_void_p), C.c_void_p]
    lib.gwi_device_minmax.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.POINTER(C.c_double)]
    lib.gwi_debug_model_read.restype = C.c_int64
    lib.gwi_debug_model_read.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64]
    lib.gwi_catalog_create.argtypes = [C.POINTER(gwi_catalog_desc), C.POINTER(C.c_void_p)]
    lib.gwi_catalog_destroy.argtypes = [C.c_void_p]
    lib.gwi_catalog_destroy.restype = None
    lib.gwi_model_create.argtypes = [C.c_void_p, C.POINTER(gwi_model_desc), C.POINTER(C.c_void_p)]
    lib.gwi_model_destroy.argtypes = [C.c_void_p]
    lib.gwi_model_destroy.restype = None
    lib.gwi_eval.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(gwi_outputs), C.c_void_p]
    lib.gwi_loglike.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(gwi_like_opts), C.c_void_p, C.c_void_p]
    lib.gwi_loglike_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(gwi_like_opts), C.c_void_p, C.c_void_p]
    lib.gwi_loglike_host.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(gwi_like_opts), C.POINTER(C.c_double)]
    lib.gwi_partial.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gwi_combine.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(gwi_like_opts), C.c_void_p, C.c_void_p]
    lib.gwi_model_get_info.argtypes = [C.c_void_p, C.POINTER(gwi_model_info)]
    lib.gwi_comm_local_handle.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    lib.gwi_comm_connect.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
    lib.gwi_loglike_sharded.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(gwi_like_opts), C.c_void_p, C.c_void_p]
    lib.gwi_sharded_push.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gwi_sharded_combine.argtypes = [C.c_void_p, C.POINTER(gwi_like_opts), C.c_void_p, C.c_void_p]
    lib.gwi_model_last_sites.restype = C.c_int64
    lib.gwi_model_last_sites.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.c_int64]
    lib.gwi_model_set_exact_shift.argtypes = [C.c_void_p, C.c_int32]
    lib.gwi_sample_log_weights.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gwi_draw_samples.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.gwi_model_set_timing.argtypes = [C.c_void_p, C.c_int32]
    lib.gwi_model_stream_times.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.c_int32]
    lib.gwi_debug_plan_build.argtypes = [C.c_void_p, C.POINTER(gwi_model_desc), C.c_int32, C.POINTER(C.c_void_p)]
    lib.gwi_debug_plan_destroy.argtypes = [C.c_void_p]
    lib.gwi_debug_plan_destroy.restype = None
    lib.gwi_nuts_sample.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_double), C.POINTER(gwi_nuts_opts), C.POINTER(C.c_double), C.POINTER(gwi_nuts_info)]
    lib.gwi_posterior_create.argtypes = [C.c_void_p, C.POINTER(gwi_like_opts), C.POINTER(gwi_prior_block), C.c_int32, C.POINTER(C.c_void_p)]
    lib.gwi_posterior_destroy.argtypes = [C.c_void_p]
    lib.gwi_posterior_destroy.restype = None
    lib.gwi_posterior_dim.argtypes = [C.c_void_p]
    lib.gwi_posterior_potential.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.gwi_posterior_potential.restype = C.c_double
    lib.gwi_nuts_sample_posterior.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(gwi_nuts_opts), C.POINTER(C.c_double), C.POINTER(gwi_nuts_info)]
    lib.gwi_nuts_sample_posterior_chains.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_double), C.POINTER(gwi_nuts_opts), C.POINTER(C.c_double), C.POINTER(gwi_nuts_info)]
    lib.gwi_loglike_batch_host.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.c_int32, C.POINTER(gwi_like_opts), C.POINTER(C.c_double)]
    _lib = lib
    return lib


def _check(rc):
    if rc != 0:
        raise GwiError(rc, load_library().gwi_last_error().decode())


def _dptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


# ---- minimal CUDA runtime access for device buffers (same libcudart libgwi.so links) -----------
def cudart():
    global _cudart
    if _cudart is None:
        load_library()
        for name in ("libcudart.so.12", "libcudart.so", "/usr/local/cuda/lib64/libcudart.so.12"):
            try:
                _cudart = C.CDLL(name)
                break
            except OSError:
                continue
        if _cudart is None:
            raise GwiError(-2, "libcudart not found")
        _cudart.cudaMalloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
        _cudart.cudaFree.argtypes = [C.c_void_p]
        _cudart.cudaMemcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
        _cudart.cudaGetErrorString.restype = C.c_char_p
        _cudart.cudaGetErrorString.argtypes = [C.c_int]
    return _cudart


def _cuda_check(rc, what):
    if rc != 0:
        raise GwiError(-2, f"{what}: {cudart().cudaGetErrorString(rc).decode()}")


def _is_device_array(a):
    return not isinstance(a, np.ndarray) and hasattr(a, "__cuda_array_interface__")


class DeviceBuffer:
    """fp64 device array (cudaMalloc) with host <-> device copies."""

    def __init__(self, n, device=0):
        rt = cudart()
        _cuda_check(rt.cudaSetDevice(int(device)), "cudaSetDevice")
        self.n = int(n)
        self.device = device
        p = C.c_void_p()
        _cuda_check(rt.cudaMalloc(C.byref(p), max(1, self.n) * 8), "cudaMalloc")
        self.ptr = p.value
        self._rt = rt  # freed by the runtime that allocated it

    def upload(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        assert a.size == self.n
        _cuda_check(cudart().cudaMemcpy(self.ptr, a.ctypes.data, a.size * 8, 1), "cudaMemcpy H2D")

    def download(self):
        out = np.empty(self.n, dtype=np.float64)
        _cuda_check(cudart().cudaMemcpy(out.ctypes.data, self.ptr, self.n * 8, 2), "cudaMemcpy D2H")
        return out

    def free(self):
        if self.ptr:
            self._rt.cudaFree(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def synchronize():
    _cuda_check(cudart().cudaDeviceSynchronize(), "cudaDeviceSynchronize")


class DeviceArray:
    """A float64 array in device memory exposing ``__cuda_array_interface__`` -- what a jax / torch / cupy array looks like
    to this package (tests and the bench use it to hand device-resident sample columns to the model classes)."""

    def __init__(self, a, device=0):
        a = np.ascontiguousarray(a, dtype=np.float64)
        self.shape = tuple(a.shape)
        self._buf = DeviceBuffer(a.size, device)
        if a.size:
            self._buf.upload(a.reshape(-1))

    @classmethod
    def empty(cls, shape, device=0):
        self = cls.__new__(cls)
        self.shape = tuple(int(x) for x in np.atleast_1d(shape))
        self._buf = DeviceBuffer(int(np.prod(self.shape)), device)
        return self

    @property
    def __cuda_array_interface__(self):
        return {"shape": self.shape, "typestr": "<f8", "data": (int(self._buf.ptr or 0), False), "version": 3, "strides": None}

    def download(self):
        return self._buf.download().reshape(self.shape)

    def minmax(self):
        """(min, max) computed on the device (gwi_device_minmax), NaN entries ignored."""
        out = (C.c_double * 2)()
        _check(load_library().gwi_device_minmax(int(self._buf.device), C.c_void_p(self._buf.ptr), int(np.prod(self.shape)), out))
        return float(out[0]), float(out[1])


INJ_COLUMNS = ["mass_1", "mass_ratio", "mass_2", "a_1", "a_2", "cos_tilt_1", "cos_tilt_2", "redshift", "prior"]


def synth_injections_device(seed, first, count, device=0):
    """The synthetic found-injection set ``[first, first + count)`` generated on the device (gwi_synth_injections):
    {column name: DeviceArray}.  Bit-identical to ``synthetic.make_injections_philox(seed, first, count)``."""
    cols = {n: DeviceArray.empty((int(count),), device) for n in INJ_COLUMNS}
    ptrs = (C.c_void_p * 9)(*[C.c_void_p(cols[n]._buf.ptr) for n in INJ_COLUMNS])
    _check(load_library().gwi_synth_injections(int(device), int(seed), int(first), int(count), ptrs, None))
    return cols


# ---- description marshalling -----------------------------------------------------------------
class _Desc:
    """Keeps the ctypes structures and every NumPy array they point to alive."""

    def __init__(self, spec, col_index, need_neff_grad=False, chunk_steps=0, n_deep=-1, batch_hint=0, keep_sample_index=False):
        self.keep = []
        nt = len(spec.terms)
        self.terms = (gwi_term * max(1, nt))()
        for i, t in enumerate(spec.terms):
            ct = self.terms[i]
            ct.kind = t.kind
            ct.feature = t.feature
            ct.outside = t.outside
            ct.logx = int(bool(t.logx))
            cols = [col_index[c] for c in t.cols] + [-1, -1]
            ct.col[0], ct.col[1] = cols[0], cols[1]
            slots = list(t.slots) + [-1] * 6
            for k in range(6):
                ct.slot[k] = int(slots[k])
            cst = list(t.cst) + [0.0] * 4
            for k in range(4):
                ct.cst[k] = float(cst[k])
            ct.n_splines = int(t.n_splines)
            ct.norm_group = int(t.norm_group)
            ct.x_lo, ct.x_hi = float(t.xrange[0]), float(t.xrange[1])
            if t.xi_range is not None:
                ct.xi_lo, ct.xi_hi = float(t.xi_range[0]), float(t.xi_range[1])
            else:
                ct.xi_lo, ct.xi_hi = ct.x_lo, ct.x_hi
            grid = t.grid_xi if t.grid_xi is not None else t.grid_feat
            if grid is not None and t.norm_group >= 0:
                g = np.ascontiguousarray(grid, dtype=np.float64)
                if g.size != np.size(spec.groups[t.norm_group].log_w):
                    raise ValueError(f"term {t.name}: grid length does not match its norm group")
                self.keep.append(g)
                ct.grid = _dptr(g)
            if getattr(t, "knots", None) is not None:  # explicit knot vector / order (interpolation.py:72-106)
                kn = np.ascontiguousarray(t.knots, dtype=np.float64)
                self.keep.append(kn)
                ct.knots, ct.n_knots, ct.order = _dptr(kn), kn.size, int(t.order)
        ng = len(spec.groups)
        self.groups = (gwi_norm_group * max(1, ng))()
        for i, g in enumerate(spec.groups):
            lw = np.ascontiguousarray(g.log_w, dtype=np.float64)
            self.keep.append(lw)
            self.groups[i].n_grid = lw.size
            self.groups[i].log_w = _dptr(lw)
        nc = len(spec.cuts)
        self.cuts = (gwi_cut * max(1, nc))()
        for i, c in enumerate(spec.cuts):
            cols = [col_index[x] for x in c.cols] + [-1, -1]
            self.cuts[i].kind = c.kind
            self.cuts[i].col[0], self.cuts[i].col[1] = cols[0], cols[1]
            self.cuts[i].lo, self.cuts[i].hi = float(c.lo), float(c.hi)
        d = gwi_model_desc()
        d.n_terms, d.terms = nt, self.terms
        d.n_groups, d.groups = ng, self.groups
        d.n_cuts, d.cuts = nc, self.cuts
        d.n_params = int(spec.n_params)
        d.need_neff_grad = int(bool(need_neff_grad))
        d.chunk_steps = int(chunk_steps)
        d.n_deep = int(n_deep)
        d.batch_hint = int(batch_hint)
        d.keep_sample_index = int(bool(keep_sample_index))
        self.desc = d


class Catalog:
    """gwi_catalog over NumPy columns.  PE columns: dict name -> (E, S) array (or a ragged list of
    per-event 1-D arrays); injection columns: dict name -> (I,) array."""

    def __init__(self, pe_cols, inj_cols, total_inj, device=0, on_device=False):
        """on_device=True: the columns are copied into device memory HERE (once) and the catalog hands the library device
        pointers (gwi_catalog_desc.columns_on_device) -- the situation of a caller whose sample arrays already live on the
        GPU (jax / torch arrays): gwi_model_create then builds the plan without any host <-> device traffic."""
        lib = load_library()
        self.names = list(pe_cols.keys())
        if list(inj_cols.keys()) != self.names:
            raise ValueError("PE and injection column names must match")
        self.col_index = {n: i for i, n in enumerate(self.names)}
        first = pe_cols[self.names[0]]
        dev = [_is_device_array(v) for v in list(pe_cols.values()) + list(inj_cols.values())]
        if any(dev):
            # device-resident columns (jax / torch / cupy arrays, DeviceArray): borrowed as device pointers
            if not all(dev):
                raise ValueError("the sample columns of one catalog must be all host arrays or all device arrays")
            self._init_from_device_arrays(lib, pe_cols, inj_cols, total_inj, device)
            return
        if isinstance(first, np.ndarray) and first.ndim == 2:
            E, S_ = first.shape
            self.offsets = np.arange(E + 1, dtype=np.int64) * S_
            self.pe = [np.ascontiguousarray(pe_cols[n], dtype=np.float64).reshape(-1) for n in self.names]
        else:  # ragged: list of 1-D arrays per event
            E = len(first)
            sizes = [len(x) for x in first]
            self.offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
            self.pe = [np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=np.float64) for x in pe_cols[n]]) if E else np.zeros(0)) for n in self.names]
        self.inj = [np.ascontiguousarray(inj_cols[n], dtype=np.float64).reshape(-1) for n in self.names]
        self.n_events = int(E)
        self.n_inj = int(self.inj[0].size)
        self.total_inj = float(total_inj)
        ncol = len(self.names)
        self.on_device = bool(on_device)
        if self.on_device:
            self._dev = []
            ptrs = []
            for cols in (self.pe, self.inj):
                row = []
                for a in cols:
                    b = DeviceBuffer(a.size, device)
                    if a.size:
                        b.upload(a)
                    self._dev.append(b)
                    row.append(C.cast(C.c_void_p(b.ptr), C.POINTER(C.c_double)))
                ptrs.append(row)
            self._pe_ptrs = (C.POINTER(C.c_double) * ncol)(*ptrs[0])
            self._inj_ptrs = (C.POINTER(C.c_double) * ncol)(*ptrs[1])
        else:
            self._pe_ptrs = (C.POINTER(C.c_double) * ncol)(*[_dptr(a) for a in self.pe])
            self._inj_ptrs = (C.POINTER(C.c_double) * ncol)(*[_dptr(a) for a in self.inj])
        d = gwi_catalog_desc()
        d.n_columns = ncol
        d.n_events = self.n_events
        d.pe_offsets = self.offsets.ctypes.data_as(C.POINTER(C.c_int64))
        d.pe_columns = self._pe_ptrs
        d.n_inj = self.n_inj
        d.inj_columns = self._inj_ptrs
        d.total_inj = self.total_inj
        d.device = int(device)
        d.columns_on_device = 1 if self.on_device else 0
        self.device = int(device)
        self._desc = d
        h = C.c_void_p()
        _check(lib.gwi_catalog_create(C.byref(d), C.byref(h)))
        self.handle = h
        self._owner = lib  # a handle is destroyed by the library that created it

    def _init_from_device_arrays(self, lib, pe_cols, inj_cols, total_inj, device):
        def ptr(a, ndim):
            ci = a.__cuda_array_interface__
            if ci.get("typestr") != "<f8" or ci.get("strides") is not None or len(ci["shape"]) != ndim:
                raise ValueError("device-resident sample arrays must be C-contiguous float64, (E, S) for PE samples and (I,) for injections")
            return C.cast(C.c_void_p(int(ci["data"][0])), C.POINTER(C.c_double)), tuple(int(x) for x in ci["shape"])

        pe = [ptr(pe_cols[n], 2) for n in self.names]
        inj = [ptr(inj_cols[n], 1) for n in self.names]
        if len({s for _, s in pe}) != 1 or len({s for _, s in inj}) != 1:
            raise ValueError("inconsistent column shapes")
        E, S_ = pe[0][1]
        self._keep = (list(pe_cols.values()), list(inj_cols.values()))  # the arrays own the device memory
        self.pe = self.inj = None
        self.offsets = np.arange(E + 1, dtype=np.int64) * S_
        self.n_events, self.n_inj, self.total_inj = int(E), int(inj[0][1][0]), float(total_inj)
        ncol = len(self.names)
        self.on_device = True
        self._pe_ptrs = (C.POINTER(C.c_double) * ncol)(*[p for p, _ in pe])
        self._inj_ptrs = (C.POINTER(C.c_double) * ncol)(*[p for p, _ in inj])
        d = gwi_catalog_desc()
        d.n_columns, d.n_events = ncol, self.n_events
        d.pe_offsets = self.offsets.ctypes.data_as(C.POINTER(C.c_int64))
        d.pe_columns, d.n_inj, d.inj_columns = self._pe_ptrs, self.n_inj, self._inj_ptrs
        d.total_inj, d.device, d.columns_on_device = self.total_inj, int(device), 1
        self.device = int(device)
        self._desc = d
        h = C.c_void_p()
        _check(lib.gwi_catalog_create(C.byref(d), C.byref(h)))
        self.handle = h
        self._owner = lib

    def close(self):
        if getattr(self, "handle", None):
            self._owner.gwi_catalog_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HostPlan:
    """Test hook: the static plan built on the host (no CUDA needed)."""

    def __init__(self, catalog, spec, need_neff_grad=False, chunk_steps=0, n_deep=-1, n_workers=0, batch_hint=0, keep_sample_index=False):
        lib = load_library()
        self._d = _Desc(spec, catalog.col_index, need_neff_grad, chunk_steps, n_deep, batch_hint, keep_sample_index)
        h = C.c_void_p()
        _check(lib.gwi_debug_plan_build(catalog.handle, C.byref(self._d.desc), int(n_workers), C.byref(h)))
        self.handle = h
        self._owner = lib

    def read(self, what, dtype=np.int64):
        lib = load_library()
        n = lib.gwi_debug_plan_read(self.handle, what, None, 0)
        if n < 0:
            raise GwiError(n, "gwi_debug_plan_read")
        out = np.empty(n, dtype=dtype)
        lib.gwi_debug_plan_read(self.handle, what, out.ctypes.data, n)
        return out

    def close(self):
        if getattr(self, "handle", None):
            self._owner.gwi_debug_plan_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Model:
    """gwi_model: the device-resident evaluation plan of one (catalog, model description)."""

    def __init__(self, catalog, spec, need_neff_grad=False, chunk_steps=0, n_deep=-1, batch_hint=0, keep_sample_index=False):
        """keep_sample_index=True: the model also keeps the catalog position of every stream position (4 bytes per padded
        sample of device memory), which :meth:`sample_log_weights` and :meth:`draw_samples` need."""
        lib = load_library()
        self.catalog = catalog
        self.keep_sample_index = bool(keep_sample_index)
        self.n_params = int(spec.n_params)
        self.n_events = catalog.n_events
        self.n_groups = len(spec.groups)
        self.need_neff_grad = bool(need_neff_grad)
        self._d = _Desc(spec, catalog.col_index, need_neff_grad, chunk_steps, n_deep, batch_hint, keep_sample_index)
        h = C.c_void_p()
        _check(lib.gwi_model_create(catalog.handle, C.byref(self._d.desc), C.byref(h)))
        self.handle = h
        self._owner = lib
        self._bufs = None

    # -- introspection ---------------------------------------------------------------------
    def info(self):
        i = gwi_model_info()
        _check(load_library().gwi_model_get_info(self.handle, C.byref(i)))
        d = {n: getattr(i, n) for n, _ in gwi_model_info._fields_ if not n.startswith("reserved")}
        d["plan_seconds"] = dict(zip(("total", "columns_upload", "keys_sort_bounds", "geometry_host", "fill"), [float(x) for x in i.plan_seconds]))
        return d

    def read_plan(self, what, dtype=np.int64):
        """Test hook (gwi_debug_model_read): the plan of the live model; what = 1 copies the stream columns back from the device."""
        lib = load_library()
        n = lib.gwi_debug_model_read(self.handle, what, None, 0)
        if n < 0:
            raise GwiError(n, "gwi_debug_model_read")
        out = np.empty(n, dtype=dtype)
        lib.gwi_debug_model_read(self.handle, what, out.ctypes.data, n)
        return out

    # -- library-owned multi-GPU exchange (include/gwi.h: gwi_comm_*) -------------------------
    def comm_local_handle(self, n_ranks):
        """This rank's exchange-buffer handle (80 bytes) to be all-gathered by any host-side means."""
        buf = C.create_string_buffer(80)
        _check(load_library().gwi_comm_local_handle(self.handle, int(n_ranks), buf))
        return buf.raw

    def comm_connect(self, handles, rank):
        """``handles``: the 80-byte handles of ALL ranks in rank order.  Follow with a host barrier."""
        blob = C.create_string_buffer(b"".join(handles), 80 * len(handles))
        _check(load_library().gwi_comm_connect(self.handle, blob, int(rank), len(handles)))

    def loglike_sharded(self, lam_ptr, out_ptr, Nobs, marginalize_selection=False, min_neff_cut=True, max_variance_cut=False, stream=None):
        o = gwi_like_opts(int(Nobs), int(marginalize_selection), int(min_neff_cut), int(max_variance_cut))
        _check(load_library().gwi_loglike_sharded(self.handle, C.c_void_p(lam_ptr), C.byref(o), C.c_void_p(out_ptr), C.c_void_p(stream)))

    def sharded_push(self, lam_ptr, stream=None):
        _check(load_library().gwi_sharded_push(self.handle, C.c_void_p(lam_ptr), C.c_void_p(stream)))

    def sharded_combine(self, out_ptr, Nobs, marginalize_selection=False, min_neff_cut=True, max_variance_cut=False, stream=None):
        o = gwi_like_opts(int(Nobs), int(marginalize_selection), int(min_neff_cut), int(max_variance_cut))
        _check(load_library().gwi_sharded_combine(self.handle, C.byref(o), C.c_void_p(out_ptr), C.c_void_p(stream)))

    def last_sites(self):
        """``[E + 1, 4]`` {log mean weight, log N_eff, variance, status} of the last evaluation; row 0 = injections."""
        lib = load_library()
        n = lib.gwi_model_last_sites(self.handle, None, 0)
        if n < 0:
            _check(int(n))
        out = np.zeros(int(n))
        got = lib.gwi_model_last_sites(self.handle, _dptr(out), int(n))
        if got < 0:
            _check(int(got))
        return out.reshape(-1, 4)

    def set_exact_shift(self, on=True):
        _check(load_library().gwi_model_set_exact_shift(self.handle, int(on)))

    def set_timing(self, on=True):
        _check(load_library().gwi_model_set_timing(self.handle, int(on)))

    def stream_times_ms(self, cap=64):
        buf = (C.c_float * cap)()
        n = load_library().gwi_model_stream_times(self.handle, buf, cap)
        if n < 0:
            _check(n)
        return np.array(buf[:n], dtype=np.float64)

    def partial_size(self):
        return int(load_library().gwi_partial_size(self.handle))

    # -- host-buffer calls -----------------------------------------------------------------
    def loglike_host(self, lam, Nobs, marginalize_selection=False, min_neff_cut=True, max_variance_cut=False):
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        if lam.size != self.n_params:
            raise ValueError(f"expected {self.n_params} hyper-parameters, got {lam.size}")
        o = gwi_like_opts(int(Nobs), int(marginalize_selection), int(min_neff_cut), int(max_variance_cut))
        out = np.empty(GWI_LIKE_HEADER + self.n_params, dtype=np.float64)
        rc = load_library().gwi_loglike_host(self.handle, _dptr(lam), C.byref(o), _dptr(out))
        if rc not in (0, -5):
            _check(rc)
        head = dict(zip(LIKE_FIELDS, out[:GWI_LIKE_HEADER]))
        return head, out[GWI_LIKE_HEADER:].copy()

    def evaluate(self, lam, jacobians=True):
        """gwi_eval with temporary device buffers; returns NumPy arrays."""
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        if lam.size != self.n_params:
            raise ValueError(f"expected {self.n_params} hyper-parameters, got {lam.size}")
        E, P, G = self.n_events, self.n_params, self.n_groups
        dev = self.catalog.device
        sizes = dict(logBF=E, logNeff=E, log_mu=1, logNeff_inj=1, logZ=G)
        if jacobians:
            sizes.update(J_logBF=E * P, J_log_mu=P)
            if self.need_neff_grad:
                sizes.update(J_logNeff=E * P, J_logNeff_inj=P)
        bufs = {k: DeviceBuffer(n, dev) for k, n in sizes.items()}
        lam_d = DeviceBuffer(P, dev)
        lam_d.upload(lam)
        outs = gwi_outputs()
        for k, b in bufs.items():
            setattr(outs, k, b.ptr)
        _check(load_library().gwi_eval(self.handle, lam_d.ptr, C.byref(outs), None))
        synchronize()
        res = {k: b.download() for k, b in bufs.items()}
        for k in ("J_logBF", "J_logNeff"):
            if k in res:
                res[k] = res[k].reshape(E, P)
        res["log_mu"] = float(res["log_mu"][0])
        res["logNeff_inj"] = float(res["logNeff_inj"][0])
        for b in bufs.values():
            b.free()
        lam_d.free()
        return res

    def _n_catalog(self):
        return int(self.catalog.offsets[-1]) + int(self.catalog.n_inj)

    def sample_log_weights(self, lam):
        """gwi_sample_log_weights: log w of every catalog sample (``-inf`` where the weight is 0), PE samples in event order
        followed by the injections, as one NumPy array.  Needs ``keep_sample_index=True``."""
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        if lam.size != self.n_params:
            raise ValueError(f"expected {self.n_params} hyper-parameters, got {lam.size}")
        dev = self.catalog.device
        lam_d, out_d = DeviceBuffer(self.n_params, dev), DeviceBuffer(self._n_catalog(), dev)
        try:
            lam_d.upload(lam)
            _check(load_library().gwi_sample_log_weights(self.handle, C.c_void_p(lam_d.ptr), C.c_void_p(out_d.ptr), None))
            synchronize()
            return out_d.download()
        finally:
            lam_d.free()
            out_d.free()

    def draw_samples(self, lam, seed, draws_per_event, draws_inj):
        """gwi_draw_samples: ``(pe[E, draws_per_event], inj[draws_inj])`` int64 local indices drawn with probability
        proportional to the weight (-1 for an event / injection set without weight).  Needs ``keep_sample_index=True``."""
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        if lam.size != self.n_params:
            raise ValueError(f"expected {self.n_params} hyper-parameters, got {lam.size}")
        E, dpe, dinj = self.n_events, int(draws_per_event), int(draws_inj)
        n = E * dpe + dinj
        dev = self.catalog.device
        lam_d, out_d = DeviceBuffer(self.n_params, dev), DeviceBuffer(n, dev)  # (8-byte items: int64 read back as bits)
        try:
            lam_d.upload(lam)
            _check(load_library().gwi_draw_samples(self.handle, C.c_void_p(lam_d.ptr), int(seed) & 0xFFFFFFFFFFFFFFFF, dpe, dinj, C.c_void_p(out_d.ptr), None))
            synchronize()
            out = out_d.download().view(np.int64)[:n]
        finally:
            lam_d.free()
            out_d.free()
        return out[: E * dpe].reshape(E, dpe).copy(), out[E * dpe :].copy()

    # -- device-pointer calls (multi-GPU plumbing) --------------------------------------------
    def partial(self, lam_ptr, record_ptr, stream=None):
        _check(load_library().gwi_partial(self.handle, lam_ptr, record_ptr, stream))

    def combine(self, records_ptr, n_ranks, out_ptr, Nobs, marginalize_selection=False, min_neff_cut=True, max_variance_cut=False, stream=None):
        o = gwi_like_opts(int(Nobs), int(marginalize_selection), int(min_neff_cut), int(max_variance_cut))
        _check(load_library().gwi_combine(self.handle, records_ptr, int(n_ranks), C.byref(o), out_ptr, stream))

    def loglike(self, lam_ptr, out_ptr, Nobs, marginalize_selection=False, min_neff_cut=True, max_variance_cut=False, stream=None):
        o = gwi_like_opts(int(Nobs), int(marginalize_selection), int(min_neff_cut), int(max_variance_cut))
        _check(load_library().gwi_loglike(self.handle, lam_ptr, C.byref(o), out_ptr, stream))

    def loglike_batch_ptr(self, lam_ptr, n_chains, out_ptr, Nobs, marginalize_selection=False, min_neff_cut=True, max_variance_cut=False, stream=None):
        o = gwi_like_opts(int(Nobs), int(marginalize_selection), int(min_neff_cut), int(max_variance_cut))
        _check(load_library().gwi_loglike_batch(self.handle, lam_ptr, int(n_chains), C.byref(o), out_ptr, stream))

    def loglike_batch(self, lams, Nobs, marginalize_selection=False, min_neff_cut=True, max_variance_cut=False):
        """gwi_loglike_batch over ``lams[n_chains, P]`` (host array in, host arrays out)."""
        lams = np.ascontiguousarray(lams, dtype=np.float64)
        n, P = lams.shape
        if P != self.n_params:
            raise ValueError(f"expected {self.n_params} hyper-parameters per chain, got {P}")
        dev = self.catalog.device
        lam_d, out_d = DeviceBuffer(n * P, dev), DeviceBuffer(n * (GWI_LIKE_HEADER + P), dev)
        lam_d.upload(lams)
        o = gwi_like_opts(int(Nobs), int(marginalize_selection), int(min_neff_cut), int(max_variance_cut))
        _check(load_library().gwi_loglike_batch(self.handle, lam_d.ptr, n, C.byref(o), out_d.ptr, None))
        synchronize()
        out = out_d.download().reshape(n, GWI_LIKE_HEADER + P)
        lam_d.free()
        out_d.free()
        return out[:, 0].copy(), out[:, GWI_LIKE_HEADER:].copy(), out[:, :GWI_LIKE_HEADER].copy()

    def loglike_batch_host(self, lams, Nobs, marginalize_selection=False, min_neff_cut=True, max_variance_cut=False):
        """gwi_loglike_batch_host over ``lams[n_chains, P]``: one call, host buffers in and out (graph-replayed per batch
        size).  Returns ``(log_l[n], grad[n, P], header[n, GWI_LIKE_HEADER])``."""
        lams = np.ascontiguousarray(lams, dtype=np.float64)
        n, P = lams.shape
        if P != self.n_params:
            raise ValueError(f"expected {self.n_params} hyper-parameters per chain, got {P}")
        out = np.empty((n, GWI_LIKE_HEADER + P), dtype=np.float64)
        o = gwi_like_opts(int(Nobs), int(marginalize_selection), int(min_neff_cut), int(max_variance_cut))
        _check(load_library().gwi_loglike_batch_host(self.handle, _dptr(lams), n, C.byref(o), _dptr(out)))
        return out[:, 0].copy(), out[:, GWI_LIKE_HEADER:].copy(), out[:, :GWI_LIKE_HEADER].copy()

    def close(self):
        if getattr(self, "handle", None):
            self._owner.gwi_model_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- native NUTS driver (csrc/nuts.cpp) ----------------------------------------------------------
NUTS_MULTINOMIAL, NUTS_WINDOWED_ADAPT, NUTS_DENSE_MASS = 1, 2, 4  # include/gwi.h: GWI_NUTS_*


def _nuts_opts(n_warmup, n_samples, max_depth, seed, target_accept, flags=0):
    return gwi_nuts_opts(int(n_warmup), int(n_samples), int(max_depth), int(flags), int(seed), float(target_accept))


def _nuts_info(i):
    return {n: getattr(i, n) for n, _ in gwi_nuts_info._fields_}


def nuts_sample(potential, theta0, n_warmup, n_samples, seed=0, target_accept=0.8, max_depth=8, flags=0):
    """gwi_nuts_sample on a Python potential ``theta -> (U, dU/dtheta)`` (tests, small problems: the
    callback re-enters the interpreter once per leapfrog step).  Returns ``(samples, info)``."""
    lib = load_library()
    theta0 = np.ascontiguousarray(theta0, dtype=np.float64)
    dim = theta0.size

    def _cb(_ctx, th, g):
        u, grad = potential(np.ctypeslib.as_array(th, shape=(dim,)).copy())
        np.ctypeslib.as_array(g, shape=(dim,))[:] = grad
        return float(u)

    cb = POTENTIAL_FN(_cb)
    samples = np.empty((int(n_samples), dim), dtype=np.float64)
    info = gwi_nuts_info()
    o = _nuts_opts(n_warmup, n_samples, max_depth, seed, target_accept, flags)
    _check(lib.gwi_nuts_sample(C.cast(cb, C.c_void_p), None, dim, _dptr(theta0), C.byref(o), _dptr(samples), C.byref(info)))
    return samples, _nuts_info(info)


class Posterior:
    """gwi_posterior: U(theta) = -(log L + log prior) of one Model, evaluated and sampled natively.
    ``blocks``: iterable of ``(lambda_slice, prior_sigma, smoothing_tau or None, difference_degree,
    fix_first_zero)`` -- the format of ``pipeline.bspline_prior_blocks`` / ``nuts.BSplinePosterior``."""

    def __init__(self, model, blocks, Nobs, marginalize_selection=False, min_neff_cut=True, max_variance_cut=False):
        lib = load_library()
        self.model = model
        blocks = list(blocks)
        arr = (gwi_prior_block * max(1, len(blocks)))()
        for i, (sl, sig, tau, deg, fix0) in enumerate(blocks):
            arr[i] = gwi_prior_block(int(sl.start), int(sl.stop - sl.start), float(sig), -1.0 if tau is None else float(tau), int(deg), int(bool(fix0)))
        o = gwi_like_opts(int(Nobs), int(marginalize_selection), int(min_neff_cut), int(max_variance_cut))
        h = C.c_void_p()
        _check(lib.gwi_posterior_create(model.handle, C.byref(o), arr, len(blocks), C.byref(h)))
        self.handle = h
        self._owner = lib
        self.dim = int(lib.gwi_posterior_dim(h))

    def potential(self, theta):
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        assert theta.size == self.dim
        grad = np.empty(self.dim, dtype=np.float64)
        u = self._owner.gwi_posterior_potential(self.handle, _dptr(theta), _dptr(grad))
        return float(u), grad

    def sample(self, theta0, n_warmup, n_samples, seed=0, target_accept=0.8, max_depth=8, flags=0):
        theta0 = np.ascontiguousarray(theta0, dtype=np.float64)
        assert theta0.size == self.dim
        samples = np.empty((int(n_samples), self.dim), dtype=np.float64)
        info = gwi_nuts_info()
        o = _nuts_opts(n_warmup, n_samples, max_depth, seed, target_accept, flags)
        _check(self._owner.gwi_nuts_sample_posterior(self.handle, _dptr(theta0), C.byref(o), _dptr(samples), C.byref(info)))
        return samples, _nuts_info(info)

    def sample_chains(self, theta0, n_warmup, n_samples, seed=0, target_accept=0.8, max_depth=8, flags=0):
        """``theta0[n_chains, dim]`` -> ``(samples[n_chains, n_samples, dim], [info per chain])``: the chains advance together,
        one batched likelihood call per round of leapfrog steps (gwi_nuts_sample_posterior_chains; chain c = ``sample`` with
        ``seed + c``).  Build the model with ``batch_hint = n_chains``."""
        theta0 = np.ascontiguousarray(theta0, dtype=np.float64)
        assert theta0.ndim == 2 and theta0.shape[1] == self.dim
        K = theta0.shape[0]
        samples = np.empty((K, int(n_samples), self.dim), dtype=np.float64)
        infos = (gwi_nuts_info * K)()
        o = _nuts_opts(n_warmup, n_samples, max_depth, seed, target_accept, flags)
        _check(self._owner.gwi_nuts_sample_posterior_chains(self.handle, K, _dptr(theta0), C.byref(o), _dptr(samples), infos))
        return samples, [_nuts_info(infos[c]) for c in range(K)]

    def close(self):
        if getattr(self, "handle", None):
            self._owner.gwi_posterior_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
