"""Host-side mirror of the reference's plugin interface on top of the C-ABI (include/spectral.h).

* ``SpectralPlanner``       one handle per GPU around ``libspectral.so`` -- batch entry points
  (host buffers = the end-to-end path; device tensors = the resident path; argmin, top-k).
* ``Params`` / ``find_traj`` / ``run_btrapz``  the same names, argument meaning and return values as
  the reference's ``src/trp_wrapper.py:19-32,56-121`` (``cub_wrapper.py`` likewise), bound to OUR
  ``libtrp.so`` / ``libcub.so``.

There is no CPU path: importing works anywhere, but creating a planner or calling ``find_traj``
without the built libraries or without a CUDA device raises.  PyTorch is used only for device
memory / streams by ``solve_device``; it is imported lazily.
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from .wire import ScenarioBatch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.environ.get("SPECTRAL_LIB_DIR") or os.path.join(_HERE, "lib")  # override: kernel experiments built out of tree

TRP, CUB = 0, 1
VARIANT_ID = {"trp": TRP, "cub": CUB, TRP: TRP, CUB: CUB}

SOLVED, SOLVED_INACCURATE, FAIL_NO_CORRIDOR, FAIL_SOLVER, FAIL_POINTS_CHECK, FAIL_TOO_MANY = range(6)
FLAG_POLISHED_S, FLAG_POLISHED_L, FLAG_VERIFIED_S, FLAG_VERIFIED_L = 1, 2, 4, 8
FLAG_VERIFIED = FLAG_VERIFIED_S | FLAG_VERIFIED_L
FAIL_COST = 100000000000.0
NUM_KERNELS = 6
NUM_CLASSES = 5
NUM_WORK = 12
TOPK_MAX = 1024   # SPECTRAL_TOPK_MAX
CERT_FAMILIES = ("position", "velocity", "acceleration", "jerk")   # SPECTRAL_CERT_FAMILIES, the last axis of certify_device's viol
KERNEL_NAMES = ("tables", "corridor", "classify", "qp", "finalize", "argmin")

CUBE_DTYPE = np.dtype([
    ("beg_t", np.int32), ("end_t", np.int32), ("t", np.float64), ("t_dif", np.float64),
    ("beg_l", np.float64), ("end_l", np.float64), ("upp_skew", np.float64), ("upp_bias", np.float64),
    ("down_skew", np.float64), ("down_bias", np.float64), ("l_upp_skew", np.float64),
    ("l_upp_bias", np.float64), ("l_down_skew", np.float64), ("l_down_bias", np.float64),
    ("merge", np.uint8), ("split", np.uint8), ("_pad", np.uint8, (2,)), ("count", np.int32)])
assert CUBE_DTYPE.itemsize == 112  # struct Cube, include/btrapz/cube_type.h:2-24

_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)


class SpectralInputs(ctypes.Structure):
    _fields_ = [(n, _dp) for n in ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref", "init",
                                   "scalars", "weights")] + [("weights_stride", ctypes.c_int)]


class SpectralOutputs(ctypes.Structure):
    _fields_ = [("K", _ip), ("segs", ctypes.c_void_p), ("ctrl", _dp), ("obj", _dp), ("a_cost", _dp), ("status", _ip),
                ("iters", _ip), ("flags", _ip), ("npts", _ip), ("samples", _dp), ("samples_cap", ctypes.c_int),
                ("lu", _dp)]


class SpectralOptions(ctypes.Structure):
    _fields_ = [("max_iter", ctypes.c_int), ("eps_abs", ctypes.c_double), ("eps_rel", ctypes.c_double),
                ("eps_prim_inf", ctypes.c_double), ("rho", ctypes.c_double), ("sigma", ctypes.c_double),
                ("alpha", ctypes.c_double), ("scaling", ctypes.c_int), ("check_termination", ctypes.c_int),
                ("adaptive_rho_interval", ctypes.c_int), ("adaptive_rho_tolerance", ctypes.c_double),
                ("polish", ctypes.c_int), ("polish_delta", ctypes.c_double), ("polish_refine_iter", ctypes.c_int),
                ("polish_rounds", ctypes.c_int), ("infeasibility_precheck", ctypes.c_int),
                ("precheck_margin", ctypes.c_double), ("shared_kkt", ctypes.c_int)]


class SpectralWinner(ctypes.Structure):
    """SpectralWinner of include/spectral.h: the best trajectory of a (multi-GPU) sweep."""
    _fields_ = [("cost", ctypes.c_double), ("index", ctypes.c_longlong), ("rank", ctypes.c_int), ("K", ctypes.c_int),
                ("segs", ctypes.c_ubyte * (32 * 112)), ("ctrl", ctypes.c_double * (12 * 32))]


WINNER_DTYPE = np.dtype([("cost", np.float64), ("index", np.int64), ("rank", np.int32), ("K", np.int32),
                         ("segs", CUBE_DTYPE, (32,)), ("ctrl", np.float64, (12 * 32,))])
assert WINNER_DTYPE.itemsize == ctypes.sizeof(SpectralWinner)


class Params(ctypes.Structure):
    """struct Params of include/btrapz/py_cpp_.h:6-21 == class Params of src/trp_wrapper.py:19-32."""
    _fields_ = [("s_acc_weight", ctypes.c_double), ("s_jerk_weight", ctypes.c_double),
                ("l_acc_weight", ctypes.c_double), ("l_jerk_weight", ctypes.c_double),
                ("weight_s_ref", ctypes.c_double), ("weight_ds_ref", ctypes.c_double),
                ("weight_l_ref", ctypes.c_double), ("weight_dl_ref", ctypes.c_double),
                ("weight_end_s", ctypes.c_double), ("weight_end_l", ctypes.c_double), ("iteration", ctypes.c_int)]


_lib = None


ROAD = (0.0, 50.0, -2.0, 8.0)   # s_l_l, s_u_l, d_l_l, d_u_l of the reference's road (src/cart_frenet.py:54-58)


def lib_path(name: str = "libspectral.so") -> str:
    return os.path.join(LIB_DIR, name)


def load_library() -> ctypes.CDLL:
    """Load libspectral.so; raises if it has not been built (there is no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` or "
                           "`make -C spectral_b200/csrc` (there is no CPU fallback)" % path)
    lib = ctypes.CDLL(path)
    lib.spectral_create.argtypes = [ctypes.c_int] * 5 + [ctypes.POINTER(ctypes.c_void_p)]
    lib.spectral_destroy.argtypes = [ctypes.c_void_p]
    lib.spectral_last_error.argtypes = [ctypes.c_void_p]
    lib.spectral_last_error.restype = ctypes.c_char_p
    lib.spectral_default_options.argtypes = [ctypes.POINTER(SpectralOptions)]
    lib.spectral_wait.argtypes = [ctypes.c_void_p]
    lib.spectral_host_alloc.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_size_t]
    lib.spectral_host_free.argtypes = [ctypes.c_void_p]
    for fn in (lib.spectral_solve_batch, lib.spectral_solve_batch_async):
        fn.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                       ctypes.POINTER(SpectralInputs), ctypes.POINTER(SpectralOptions), ctypes.POINTER(SpectralOutputs)]
    lib.spectral_solve_batch_device.argtypes = lib.spectral_solve_batch.argtypes + [ctypes.c_void_p]
    lib.spectral_solve_weights.argtypes = lib.spectral_solve_batch.argtypes
    lib.spectral_solve_weights_device.argtypes = lib.spectral_solve_batch_device.argtypes
    lib.spectral_argmin_device.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong,
                                           ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    lib.spectral_launch_count.argtypes = [ctypes.c_void_p]
    lib.spectral_launch_count.restype = ctypes.c_longlong
    lib.spectral_measure_fp64_peak.argtypes = [ctypes.c_void_p, _dp]
    lib.spectral_set_timing.argtypes = [ctypes.c_void_p, ctypes.c_int]
    lib.spectral_get_timing.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_float), _ip]
    lib.spectral_get_work.argtypes = [ctypes.c_void_p, _dp, ctypes.c_int]
    lib.spectral_get_class_timing.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_float)]
    lib.spectral_comm_init.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_ubyte)]
    lib.spectral_bounds_device.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, _dp,
                                           ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    lib.spectral_ego_states_device.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                               ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    lib.spectral_frenet_to_cartesian_device.argtypes = [ctypes.c_void_p, ctypes.c_longlong] + [ctypes.c_void_p] * 5
    lib.spectral_comm_unique_id.argtypes = [ctypes.POINTER(ctypes.c_ubyte)]
    lib.spectral_sweep_argmin.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p]
    lib.spectral_topk_device.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int,
                                         ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    lib.spectral_sweep_topk.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int,
                                        ctypes.c_void_p, ctypes.POINTER(ctypes.c_int), ctypes.c_void_p]
    lib.spectral_eval_device.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(SpectralOutputs), ctypes.c_int, ctypes.c_void_p,
                                         ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    lib.spectral_certify_device.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(SpectralInputs),
                                            ctypes.c_int, ctypes.POINTER(SpectralOutputs), _dp, ctypes.c_void_p, ctypes.c_void_p,
                                            ctypes.c_void_p]
    _lib = lib
    return lib


def default_options(**overrides) -> SpectralOptions:
    o = SpectralOptions()
    load_library().spectral_default_options(ctypes.byref(o))
    for k, v in overrides.items():
        if not hasattr(o, k):
            raise AttributeError("unknown option %r" % k)
        setattr(o, k, v)
    return o


@dataclass
class BatchResult:
    K: np.ndarray        # [B] segment counts
    segs: np.ndarray     # [B, k_max] CUBE_DTYPE, the selected corridor sequence (new_corridor)
    ctrl: np.ndarray     # [B, 12*k_max] control points, s-axis [0,6K) then l-axis [6K,12K)
    obj: np.ndarray      # [B] QP objective
    a_cost: np.ndarray   # [B] wrapper cost (1e11 on failure)
    status: np.ndarray   # [B]
    iters: np.ndarray    # [B] ADMM iterations
    flags: np.ndarray    # [B]
    npts: np.ndarray     # [B]
    samples: Optional[np.ndarray] = None  # [B, samples_cap, 6]
    lu: Optional[np.ndarray] = None       # [B, 2, k_max, 21, 2]

    def ok(self) -> np.ndarray:
        return self.status <= SOLVED_INACCURATE

    def verified(self) -> np.ndarray:
        return self.ok() & ((self.flags & FLAG_VERIFIED) == FLAG_VERIFIED)


def _d(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def _i(a):
    return a.ctypes.data_as(_ip) if a is not None else None


class SpectralPlanner:
    """One handle per GPU (spectral_create / spectral_destroy)."""

    def __init__(self, device: int = 0, max_batch: int = 1024, n_max: int = 128, r_max: int = 8, k_max: int = 32):
        self._lib = load_library()
        self._h = ctypes.c_void_p()
        self.device, self.max_batch, self.n_max, self.r_max, self.k_max = device, max_batch, n_max, r_max, k_max
        rc = self._lib.spectral_create(device, max_batch, n_max, r_max, k_max, ctypes.byref(self._h))
        if rc != 0:
            msg = self._lib.spectral_last_error(self._h).decode() if self._h else "no CUDA device"
            if self._h:
                self._lib.spectral_destroy(self._h)
            self._h = ctypes.c_void_p()
            raise RuntimeError("spectral_create failed (rc=%d): %s -- libspectral has no CPU path" % (rc, msg))

    def close(self):
        if getattr(self, "_h", None):
            if getattr(self, "_pending", None) is not None:
                self._lib.spectral_wait(self._h)
                self._pending = None
            for _, ptr in self.__dict__.pop("_pin", {}).values():
                self._lib.spectral_host_free(ptr)
            self._lib.spectral_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError("libspectral error %d: %s" % (rc, self._lib.spectral_last_error(self._h).decode()))

    # ---- end-to-end path: host (numpy) buffers, H2D + kernels + D2H inside the call
    def solve(self, variant, batch: ScenarioBatch, weights: Sequence[float], options: Optional[SpectralOptions] = None,
              samples_cap: int = 0, want_lu: bool = False) -> BatchResult:
        B = batch.batch
        w = np.ascontiguousarray(np.asarray(weights, dtype=np.float64))
        if w.shape not in ((10,), (B, 10)):
            raise ValueError("weights must have shape (10,) or (B, 10)")
        arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in batch.arrays()]
        inp = SpectralInputs(*[_d(a) for a in arrs], _d(w), 0 if w.ndim == 1 else 1)
        km = self.k_max
        res = BatchResult(np.zeros(B, np.int32), np.zeros((B, km), CUBE_DTYPE), np.zeros((B, 12 * km)), np.zeros(B),
                          np.zeros(B), np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32),
                          np.zeros(B, np.int32),
                          np.zeros((B, samples_cap, 6)) if samples_cap > 0 else None,
                          np.zeros((B, 2, km, 21, 2)) if want_lu else None)
        out = SpectralOutputs(_i(res.K), res.segs.ctypes.data_as(ctypes.c_void_p), _d(res.ctrl), _d(res.obj),
                              _d(res.a_cost), _i(res.status), _i(res.iters), _i(res.flags), _i(res.npts),
                              _d(res.samples), samples_cap, _d(res.lu))
        self._check(self._lib.spectral_solve_batch(self._h, VARIANT_ID[variant], B, batch.n_knots, batch.n_regions,
                                                   float(batch.delta_t), ctypes.byref(inp),
                                                   ctypes.byref(options) if options is not None else None,
                                                   ctypes.byref(out)))
        return res

    def solve_weights(self, variant, scenario: ScenarioBatch, weights, options: Optional[SpectralOptions] = None,
                      samples_cap: int = 0) -> BatchResult:
        """Weight sweep (the batch form of trp_wrapper.py:56-97 run_btrapz): ONE scenario (a ScenarioBatch of 1) against
        B weight vectors [B, 10]; the corridor stage runs once on the device and is shared by all lanes."""
        if scenario.batch != 1:
            raise ValueError("solve_weights takes exactly one scenario")
        w = np.ascontiguousarray(np.asarray(weights, dtype=np.float64))
        if w.ndim != 2 or w.shape[1] != 10:
            raise ValueError("weights must have shape (B, 10)")
        B = w.shape[0]
        arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in scenario.arrays()]
        inp = SpectralInputs(*[_d(a) for a in arrs], _d(w), 1)
        km = self.k_max
        res = BatchResult(np.zeros(B, np.int32), np.zeros((B, km), CUBE_DTYPE), np.zeros((B, 12 * km)), np.zeros(B),
                          np.zeros(B), np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32),
                          np.zeros(B, np.int32), np.zeros((B, samples_cap, 6)) if samples_cap > 0 else None, None)
        out = SpectralOutputs(_i(res.K), res.segs.ctypes.data_as(ctypes.c_void_p), _d(res.ctrl), _d(res.obj),
                              _d(res.a_cost), _i(res.status), _i(res.iters), _i(res.flags), _i(res.npts),
                              _d(res.samples), samples_cap, None)
        self._check(self._lib.spectral_solve_weights(self._h, VARIANT_ID[variant], B, scenario.n_knots, scenario.n_regions,
                                                     float(scenario.delta_t), ctypes.byref(inp),
                                                     ctypes.byref(options) if options is not None else None, ctypes.byref(out)))
        return res

    # ---- pipelined host path: page-locked buffers owned by the planner, one batch in flight per planner
    def _pinned(self, key, shape, dtype):
        """A page-locked numpy array (cudaHostAlloc through the C-ABI), cached per (name, shape)."""
        cache = self.__dict__.setdefault("_pin", {})
        k = (key, tuple(shape), np.dtype(dtype).str)
        if k not in cache:
            nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
            ptr = ctypes.c_void_p()
            self._check(self._lib.spectral_host_alloc(ctypes.byref(ptr), max(nbytes, 1)))
            buf = (ctypes.c_char * max(nbytes, 1)).from_address(ptr.value)
            cache[k] = (np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape), ptr)
        return cache[k][0]

    def solve_async(self, variant, batch: ScenarioBatch, weights: Sequence[float],
                    options: Optional[SpectralOptions] = None) -> None:
        """Enqueue one batch (H2D copies, kernels, D2H copies) on this planner's stream and return; `wait()` returns the
        result.  Inputs are staged into page-locked buffers unless they already are this planner's (see `pinned_inputs`).
        A caller keeps the GPU full by cycling over a few planners."""
        if getattr(self, "_pending", None) is not None:
            raise RuntimeError("a batch is already in flight on this planner: call wait() first")
        B, km = batch.batch, self.k_max
        w = np.ascontiguousarray(np.asarray(weights, dtype=np.float64))
        if w.shape not in ((10,), (B, 10)):
            raise ValueError("weights must have shape (10,) or (B, 10)")
        names = ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref", "init", "scalars")
        staged = []
        for name, a in zip(names, batch.arrays()):
            pin = self._pinned("in_" + name, a.shape, np.float64)
            if a is not pin:
                np.copyto(pin, a)
            staged.append(pin)
        wp = self._pinned("in_w", w.shape, np.float64)
        np.copyto(wp, w)
        inp = SpectralInputs(*[_d(a) for a in staged], _d(wp), 0 if w.ndim == 1 else 1)
        res = BatchResult(self._pinned("K", (B,), np.int32), self._pinned("segs", (B, km), CUBE_DTYPE),
                          self._pinned("ctrl", (B, 12 * km), np.float64), self._pinned("obj", (B,), np.float64),
                          self._pinned("a_cost", (B,), np.float64), self._pinned("status", (B,), np.int32),
                          self._pinned("iters", (B,), np.int32), self._pinned("flags", (B,), np.int32),
                          self._pinned("npts", (B,), np.int32), None, None)
        out = SpectralOutputs(_i(res.K), res.segs.ctypes.data_as(ctypes.c_void_p), _d(res.ctrl), _d(res.obj),
                              _d(res.a_cost), _i(res.status), _i(res.iters), _i(res.flags), _i(res.npts), None, 0, None)
        self._check(self._lib.spectral_solve_batch_async(self._h, VARIANT_ID[variant], B, batch.n_knots, batch.n_regions,
                                                         float(batch.delta_t), ctypes.byref(inp),
                                                         ctypes.byref(options) if options is not None else None,
                                                         ctypes.byref(out)))
        self._pending = (res, inp, out, staged, wp)  # keeps the argument structs alive

    def pinned_inputs(self, batch: ScenarioBatch) -> ScenarioBatch:
        """Copy of `batch` living in this planner's page-locked input buffers: passing it to solve_async skips the staging copy."""
        names = ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref", "init", "scalars")
        arrs = []
        for name, a in zip(names, batch.arrays()):
            pin = self._pinned("in_" + name, a.shape, np.float64)
            np.copyto(pin, a)
            arrs.append(pin)
        return ScenarioBatch(batch.n_knots, batch.n_regions, batch.delta_t, *arrs)

    def wait(self) -> BatchResult:
        """Block until the batch enqueued by solve_async has landed; the arrays are views of the planner's page-locked
        output buffers and are overwritten by the next solve_async on this planner."""
        if getattr(self, "_pending", None) is None:
            raise RuntimeError("nothing in flight")
        self._check(self._lib.spectral_wait(self._h))
        res = self._pending[0]
        self._pending = None
        return res

    # ---- resident path: torch CUDA tensors (float64 / int32), enqueued on the current stream
    def solve_device(self, variant, n_knots: int, n_regions: int, delta_t: float, inputs: dict, outputs: dict,
                     options: Optional[SpectralOptions] = None, stream: Optional[int] = None):
        """inputs: s_bounds,l_bounds,ds_bounds,dl_bounds,s_ref,l_ref,init,scalars,weights (CUDA float64 tensors);
        outputs: K,segs(uint8 [B,k_max*112]),ctrl,obj,a_cost,status,iters,flags,npts (CUDA tensors)."""
        import torch
        B = int(inputs["s_ref"].shape[0])
        ptr = lambda t: ctypes.cast(ctypes.c_void_p(t.data_ptr()), _dp) if t is not None else None  # noqa: E731
        iptr = lambda t: ctypes.cast(ctypes.c_void_p(t.data_ptr()), _ip) if t is not None else None  # noqa: E731
        w = inputs["weights"]
        inp = SpectralInputs(*[ptr(inputs[k]) for k in ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref",
                                                        "l_ref", "init", "scalars")], ptr(w), 0 if w.dim() == 1 else 1)
        g = outputs.get
        out = SpectralOutputs(iptr(outputs["K"]), ctypes.c_void_p(outputs["segs"].data_ptr()), ptr(outputs["ctrl"]),
                              ptr(g("obj")), ptr(g("a_cost")), iptr(outputs["status"]), iptr(g("iters")),
                              iptr(g("flags")), iptr(g("npts")), ptr(g("samples")),
                              int(g("samples").shape[1]) if g("samples") is not None else 0, ptr(g("lu")))
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        self._check(self._lib.spectral_solve_batch_device(self._h, VARIANT_ID[variant], B, n_knots, n_regions,
                                                          float(delta_t), ctypes.byref(inp),
                                                          ctypes.byref(options) if options is not None else None,
                                                          ctypes.byref(out), ctypes.c_void_p(stream)))

    def alloc_device_outputs(self, B: int, samples_cap: int = 0):
        import torch
        dev = torch.device("cuda", self.device)
        o = dict(K=torch.zeros(B, dtype=torch.int32, device=dev),
                 segs=torch.zeros(B, self.k_max * 112, dtype=torch.uint8, device=dev),
                 ctrl=torch.zeros(B, 12 * self.k_max, dtype=torch.float64, device=dev),
                 obj=torch.zeros(B, dtype=torch.float64, device=dev),
                 a_cost=torch.zeros(B, dtype=torch.float64, device=dev),
                 status=torch.zeros(B, dtype=torch.int32, device=dev),
                 iters=torch.zeros(B, dtype=torch.int32, device=dev),
                 flags=torch.zeros(B, dtype=torch.int32, device=dev),
                 npts=torch.zeros(B, dtype=torch.int32, device=dev))
        if samples_cap:
            o["samples"] = torch.zeros(B, samples_cap, 6, dtype=torch.float64, device=dev)
        return o

    def argmin_device(self, a_cost, index_offset: int, out_cost, out_index, stream: Optional[int] = None):
        """(min cost, lowest index) of a CUDA float64 tensor -> out_cost (float64[1]), out_index (int64[1])."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        self._check(self._lib.spectral_argmin_device(self._h, int(a_cost.numel()), ctypes.c_void_p(a_cost.data_ptr()),
                                                     int(index_offset), ctypes.c_void_p(out_cost.data_ptr()),
                                                     ctypes.c_void_p(out_index.data_ptr()), ctypes.c_void_p(stream)))

    @staticmethod
    def _check_k(k) -> int:
        k = int(k)
        if not 1 <= k <= TOPK_MAX:
            raise ValueError("k must be in [1, %d], got %d" % (TOPK_MAX, k))
        return k

    def _check_tensor(self, t, name: str, dtype, rows: int, row_elems: Optional[int] = None):
        """`t` must be a contiguous tensor of `dtype` on this planner's GPU with at least `rows` rows (of `row_elems`
        elements each, when given): the kernels read it through a raw pointer."""
        import torch
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.device.index != self.device:
            raise ValueError("%s must be a CUDA tensor on cuda:%d" % (name, self.device))
        if t.dtype != dtype or not t.is_contiguous():
            raise ValueError("%s must be a contiguous %s tensor" % (name, dtype))
        if row_elems is None:
            if t.numel() < rows:
                raise ValueError("%s holds %d elements, %d are needed" % (name, t.numel(), rows))
        elif t.dim() == 0 or t.shape[0] < rows or t[0].numel() != row_elems:
            raise ValueError("%s must have shape [>= %d, %d elements per row], got %s" % (name, rows, row_elems, tuple(t.shape)))

    def topk_device(self, a_cost, k: int, index_offset: int = 0, out_cost=None, out_index=None, stream: Optional[int] = None):
        """The k best entries of a CUDA float64 tensor, ascending on (cost, index_offset + i) (spectral_topk_device: -0.0 equals
        +0.0, NaN last, costs returned as stored; slots beyond the number of entries are (+inf, -1)).  Returns
        (cost float64[k], index int64[k]) on the device, enqueued on `stream` (default: the current torch stream)."""
        import torch
        k = self._check_k(k)
        if index_offset < 0:
            raise ValueError("index_offset must be non-negative")
        self._check_tensor(a_cost, "a_cost", torch.float64, 1)
        if out_cost is None:
            out_cost = torch.empty(k, dtype=torch.float64, device=a_cost.device)
        if out_index is None:
            out_index = torch.empty(k, dtype=torch.int64, device=a_cost.device)
        self._check_tensor(out_cost, "out_cost", torch.float64, k)
        self._check_tensor(out_index, "out_index", torch.int64, k)
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        self._check(self._lib.spectral_topk_device(self._h, int(a_cost.numel()), ctypes.c_void_p(a_cost.data_ptr()), int(index_offset),
                                                   k, ctypes.c_void_p(out_cost.data_ptr()), ctypes.c_void_p(out_index.data_ptr()),
                                                   ctypes.c_void_p(stream)))
        return out_cost, out_index

    # ---- multi-GPU exchange through the C-ABI (NCCL inside libspectral.so)
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = (ctypes.c_ubyte * 128)()
        if load_library().spectral_comm_unique_id(buf) != 0:
            raise RuntimeError("spectral_comm_unique_id failed (libnccl.so.2 not loadable?)")
        return bytes(buf)

    def comm_init(self, nranks: int, rank: int, unique_id: Optional[bytes]) -> None:
        buf = (ctypes.c_ubyte * 128)(*unique_id) if unique_id is not None else None
        self._check(self._lib.spectral_comm_init(self._h, int(nranks), int(rank), buf))

    def sweep_argmin(self, outputs: dict, index_offset: int, B: Optional[int] = None, stream: Optional[int] = None) -> dict:
        """Collective over all ranks of the communicator: this rank's shard results (device outputs of solve_device)
        -> the sweep's best trajectory on every rank (spectral_sweep_argmin)."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        B = int(outputs["a_cost"].numel()) if B is None else int(B)
        out = SpectralOutputs()
        out.K = ctypes.cast(ctypes.c_void_p(outputs["K"].data_ptr()), _ip)
        out.segs = outputs["segs"].data_ptr()
        out.ctrl = ctypes.cast(ctypes.c_void_p(outputs["ctrl"].data_ptr()), _dp)
        out.a_cost = ctypes.cast(ctypes.c_void_p(outputs["a_cost"].data_ptr()), _dp)
        w = SpectralWinner()
        self._check(self._lib.spectral_sweep_argmin(self._h, B, ctypes.byref(out), int(index_offset), ctypes.byref(w),
                                                    ctypes.c_void_p(stream)))
        K = int(w.K)
        segs = np.frombuffer(bytes(w.segs), dtype=CUBE_DTYPE)[:max(K, 0)].copy()
        return dict(cost=float(w.cost), index=int(w.index), rank=int(w.rank), K=K, segs=segs,
                    ctrl=np.array(w.ctrl[:12 * max(K, 0)], dtype=np.float64))

    def sweep_topk(self, outputs: dict, index_offset: int, k: int, B: Optional[int] = None, stream: Optional[int] = None) -> list:
        """Collective over all ranks of the communicator (spectral_sweep_topk): this rank's shard results -> the sweep's k best
        trajectories on every rank, as a list of min(k, total scenarios) dicts shaped like sweep_argmin's.  B = 0: this rank
        takes part without scenarios."""
        import torch
        k = self._check_k(k)
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        B = int(outputs["a_cost"].numel()) if B is None else int(B)
        if B < 0:
            raise ValueError("B must be non-negative")
        if index_offset < 0:
            raise ValueError("index_offset must be non-negative")
        out = SpectralOutputs()
        if B > 0:
            self._check_tensor(outputs["a_cost"], "a_cost", torch.float64, B)
            self._check_tensor(outputs["K"], "K", torch.int32, B)
            self._check_tensor(outputs["segs"], "segs", torch.uint8, B, self.k_max * 112)
            self._check_tensor(outputs["ctrl"], "ctrl", torch.float64, B, 12 * self.k_max)
            out.K = ctypes.cast(ctypes.c_void_p(outputs["K"].data_ptr()), _ip)
            out.segs = outputs["segs"].data_ptr()
            out.ctrl = ctypes.cast(ctypes.c_void_p(outputs["ctrl"].data_ptr()), _dp)
            out.a_cost = ctypes.cast(ctypes.c_void_p(outputs["a_cost"].data_ptr()), _dp)
        ws = (SpectralWinner * k)()
        n = ctypes.c_int()
        self._check(self._lib.spectral_sweep_topk(self._h, B, ctypes.byref(out), int(index_offset), k, ws, ctypes.byref(n),
                                                  ctypes.c_void_p(stream)))
        arr = np.frombuffer(ws, dtype=WINNER_DTYPE, count=n.value)
        res = []
        for w in arr:
            K = max(int(w["K"]), 0)
            res.append(dict(cost=float(w["cost"]), index=int(w["index"]), rank=int(w["rank"]), K=int(w["K"]),
                            segs=w["segs"][:K].copy(), ctrl=w["ctrl"][:12 * K].copy()))
        return res

    # ---- upstream of the path (Car.getCar / get_bounds of src/cart_frenet.py:644-1026), CUDA tensors in and out
    def bounds_device(self, obstacles, n_knots: int, r_cap: int, n_obs=None, road=ROAD, stream: Optional[int] = None):
        """obstacles: float64 [B, M, 6] = (s, l, t0, vel_s, vel_l, horizon) per obstacle, creation order; n_obs: int32 [B] or None.
        Returns (s_bounds [B, r_cap, N, 2], l_bounds [B, r_cap, N, 2], n_lanes int32 [B]); lanes >= n_lanes[b] are empty lanes
        (never selected by the corridor stage), so the pair feeds solve_device with n_regions = r_cap."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        B, M = int(obstacles.shape[0]), int(obstacles.shape[1])
        sb = torch.empty(B, r_cap, n_knots, 2, dtype=torch.float64, device=obstacles.device)
        lb = torch.empty(B, r_cap, n_knots, 2, dtype=torch.float64, device=obstacles.device)
        nl = torch.empty(B, dtype=torch.int32, device=obstacles.device)
        rd = (ctypes.c_double * 4)(*[float(v) for v in road])
        self._check(self._lib.spectral_bounds_device(self._h, B, n_knots, M, ctypes.c_void_p(obstacles.data_ptr()),
                                                     ctypes.c_void_p(n_obs.data_ptr()) if n_obs is not None else None, rd, r_cap,
                                                     ctypes.c_void_p(sb.data_ptr()), ctypes.c_void_p(lb.data_ptr()),
                                                     ctypes.c_void_p(nl.data_ptr()), ctypes.c_void_p(stream)))
        return sb, lb, nl

    # ---- downstream of the path (run_ego / frenet_to_cartesian3D of src/cart_frenet.py), CUDA tensors in and out
    def ego_states_device(self, samples, npts, s_offset, stream: Optional[int] = None):
        """samples: float64 [B, cap, 6] (the `samples` output), npts: int32 [B], s_offset: float64 [B] or [1] -> float64 [B, cap, 4]."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        B, cap = int(samples.shape[0]), int(samples.shape[1])
        states = torch.zeros(B, cap, 4, dtype=torch.float64, device=samples.device)
        self._check(self._lib.spectral_ego_states_device(self._h, B, ctypes.c_void_p(samples.data_ptr()), ctypes.c_void_p(npts.data_ptr()), cap,
                                                         ctypes.c_void_p(s_offset.data_ptr()), 1 if s_offset.numel() > 1 else 0,
                                                         ctypes.c_void_p(states.data_ptr()), ctypes.c_void_p(stream)))
        return states

    def frenet_to_cartesian_device(self, ref, s_cond, d_cond, stream: Optional[int] = None):
        """ref: float64 [n, 6], s_cond / d_cond: float64 [n, 3] -> float64 [n, 6] = (x, y, v, a, theta, kappa)."""
        import torch
        if stream is None:
            stream = torch.cuda.current_stream().cuda_stream
        n = int(ref.shape[0])
        out = torch.empty(n, 6, dtype=torch.float64, device=ref.device)
        self._check(self._lib.spectral_frenet_to_cartesian_device(self._h, n, ctypes.c_void_p(ref.data_ptr()), ctypes.c_void_p(s_cond.data_ptr()),
                                                                  ctypes.c_void_p(d_cond.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                                                  ctypes.c_void_p(stream)))
        return out

    # ---- solved trajectories at caller-chosen times (spectral_eval_device)
    def eval_device(self, outputs: dict, times, B: Optional[int] = None, jerk: bool = False, stream: Optional[int] = None):
        """The trajectories of `outputs` (alloc_device_outputs / solve_device: K, segs, ctrl, status) at `times`, a CUDA
        float64 tensor [T] (every scenario) or [B, T] (per scenario).  Returns (states float64 [B, T, 6] = (s, ds, dds, l, dl,
        ddl), jerk float64 [B, T, 2] = (ddds, dddl) or None, horizon float64 [B]), enqueued on `stream` (default: the
        current torch stream).  NaN rows for times outside [-1e-9, H + 1e-9] and for failed scenarios (include/spectral.h)."""
        import torch
        B = int(outputs["K"].numel()) if B is None else int(B)
        if B < 1:
            raise ValueError("B must be positive")
        self._check_tensor(outputs["K"], "K", torch.int32, B)
        self._check_tensor(outputs["status"], "status", torch.int32, B)
        self._check_tensor(outputs["segs"], "segs", torch.uint8, B, self.k_max * 112)
        self._check_tensor(outputs["ctrl"], "ctrl", torch.float64, B, 12 * self.k_max)
        if not isinstance(times, torch.Tensor) or times.dim() not in (1, 2):
            raise ValueError("times must be a tensor of shape [T] or [B, T]")
        T = int(times.shape[-1])
        if T < 1:
            raise ValueError("times is empty")
        if times.dim() == 2:
            self._check_tensor(times, "times", torch.float64, B, T)
        else:
            self._check_tensor(times, "times", torch.float64, T)
        dev = times.device
        states = torch.empty(B, T, 6, dtype=torch.float64, device=dev)
        jk = torch.empty(B, T, 2, dtype=torch.float64, device=dev) if jerk else None
        horizon = torch.empty(B, dtype=torch.float64, device=dev)
        out = SpectralOutputs()
        out.K = ctypes.cast(ctypes.c_void_p(outputs["K"].data_ptr()), _ip)
        out.status = ctypes.cast(ctypes.c_void_p(outputs["status"].data_ptr()), _ip)
        out.segs = outputs["segs"].data_ptr()
        out.ctrl = ctypes.cast(ctypes.c_void_p(outputs["ctrl"].data_ptr()), _dp)
        if stream is None:
            stream = torch.cuda.current_stream(dev).cuda_stream
        self._check(self._lib.spectral_eval_device(self._h, B, ctypes.byref(out), T, ctypes.c_void_p(times.data_ptr()),
                                                   1 if times.dim() == 2 else 0, ctypes.c_void_p(states.data_ptr()),
                                                   ctypes.c_void_p(jk.data_ptr()) if jk is not None else None,
                                                   ctypes.c_void_p(horizon.data_ptr()), ctypes.c_void_p(stream)))
        return states, jk, horizon

    # ---- feasibility certificate of solved trajectories (spectral_certify_device)
    def certify_device(self, variant, n_knots: int, inputs: dict, outputs: dict, tol, shared_inputs: bool = False,
                       B: Optional[int] = None, stream: Optional[int] = None):
        """How far each trajectory of `outputs` (K, segs, ctrl, status, a_cost) is from satisfying the constraint rows of the
        QP it was solved for, from `inputs` (ds_bounds, dl_bounds, init, scalars: the solve's inputs; shared_inputs=True: the
        one scenario of a solve_weights run).  `tol`: the acceptable violation, one float or one per row family (CERT_FAMILIES),
        in the QP's row units (include/spectral.h); there is no default.  Returns (viol float64 [B, 2, 4]: the largest violation
        per axis (s, l) and family, NaN for scenarios that cannot be certified; cost float64 [B]: a_cost where every entry is
        <= tol, FAIL_COST elsewhere), enqueued on `stream` (default: the current torch stream).  Primal feasibility only, not
        optimality.  `cost` feeds topk_device / argmin_device, or sweep_topk / sweep_argmin as outputs["a_cost"]."""
        import torch
        B = int(outputs["K"].numel()) if B is None else int(B)
        if B < 1:
            raise ValueError("B must be positive")
        n_knots = int(n_knots)
        if not 3 <= n_knots <= self.n_max:
            raise ValueError("n_knots must be in [3, %d]" % self.n_max)
        tol = np.broadcast_to(np.asarray(tol, dtype=np.float64), (len(CERT_FAMILIES),)).copy()
        if not (tol >= 0.0).all():
            raise ValueError("tol must be non-negative, got %s" % tol)
        self._check_tensor(outputs["K"], "K", torch.int32, B)
        self._check_tensor(outputs["status"], "status", torch.int32, B)
        self._check_tensor(outputs["segs"], "segs", torch.uint8, B, self.k_max * 112)
        self._check_tensor(outputs["ctrl"], "ctrl", torch.float64, B, 12 * self.k_max)
        self._check_tensor(outputs["a_cost"], "a_cost", torch.float64, B)
        Bi = 1 if shared_inputs else B
        for name, row in (("ds_bounds", 2 * n_knots), ("dl_bounds", 2 * n_knots), ("init", 6), ("scalars", 10)):
            self._check_tensor(inputs[name], name, torch.float64, Bi, row)
        dev = outputs["ctrl"].device
        viol = torch.empty(B, 2, len(CERT_FAMILIES), dtype=torch.float64, device=dev)
        cost = torch.empty(B, dtype=torch.float64, device=dev)
        inp = SpectralInputs()
        for name in ("ds_bounds", "dl_bounds", "init", "scalars"):
            setattr(inp, name, ctypes.cast(ctypes.c_void_p(inputs[name].data_ptr()), _dp))
        out = SpectralOutputs()
        out.K = ctypes.cast(ctypes.c_void_p(outputs["K"].data_ptr()), _ip)
        out.status = ctypes.cast(ctypes.c_void_p(outputs["status"].data_ptr()), _ip)
        out.segs = outputs["segs"].data_ptr()
        out.ctrl = ctypes.cast(ctypes.c_void_p(outputs["ctrl"].data_ptr()), _dp)
        out.a_cost = ctypes.cast(ctypes.c_void_p(outputs["a_cost"].data_ptr()), _dp)
        if stream is None:
            stream = torch.cuda.current_stream(dev).cuda_stream
        self._check(self._lib.spectral_certify_device(self._h, VARIANT_ID[variant], B, n_knots, ctypes.byref(inp),
                                                      0 if shared_inputs else 1, ctypes.byref(out), _d(tol),
                                                      ctypes.c_void_p(viol.data_ptr()), ctypes.c_void_p(cost.data_ptr()),
                                                      ctypes.c_void_p(stream)))
        return viol, cost

    def launch_count(self) -> int:
        return int(self._lib.spectral_launch_count(self._h))

    def measure_fp64_peak(self) -> float:
        v = ctypes.c_double()
        self._check(self._lib.spectral_measure_fp64_peak(self._h, ctypes.byref(v)))
        return v.value

    def set_timing(self, on: bool):
        self._check(self._lib.spectral_set_timing(self._h, 1 if on else 0))

    def get_timing(self) -> dict:
        """Summed device ms per kernel class over the calls recorded since set_timing(True), plus 'calls'."""
        ms = (ctypes.c_float * NUM_KERNELS)()
        calls = ctypes.c_int()
        self._check(self._lib.spectral_get_timing(self._h, ms, ctypes.byref(calls)))
        out = {k: float(ms[i]) for i, k in enumerate(KERNEL_NAMES)}
        out["calls"] = calls.value
        return out

    def get_work(self, reset: bool = False) -> dict:
        w = (ctypes.c_double * NUM_WORK)()
        self._check(self._lib.spectral_get_work(self._h, w, 1 if reset else 0))
        return dict(admm_iters=w[0], admm_flops=w[1], scenarios=w[2], solved=w[3], sum_K=w[4], admm_flops_variable=w[5],
                    **{"admm_flops_class%d" % c: w[6 + c] for c in range(NUM_CLASSES)})

    def get_class_timing(self) -> list:
        """Summed device ms per solver class (K <= 8, 10, 12, 16, 32) since set_timing(True)."""
        ms = (ctypes.c_float * NUM_CLASSES)()
        self._check(self._lib.spectral_get_class_timing(self._h, ms))
        return [float(x) for x in ms]


# ------------------------------------------------------------------ the reference's plugin surface
_plugins = {}


def _plugin(variant: str) -> ctypes.CDLL:
    """Our libtrp.so / libcub.so (trp_wrapper.py:45-54: CDLL + argtypes + restype)."""
    if variant not in _plugins:
        path = lib_path("lib%s.so" % variant)
        if not os.path.exists(path):
            raise RuntimeError(path + " is missing (build with `make -C spectral_b200/csrc`)")
        cdll = ctypes.CDLL(path)
        cdll.find_traj.argtypes = (ctypes.POINTER(Params),)
        cdll.find_traj.restype = ctypes.c_double
        _plugins[variant] = cdll
    return _plugins[variant]


def _run_btrapz(params: Params, variant: str = "trp") -> float:
    """`_run_btrapz = cdll.find_traj` of trp_wrapper.py:49: returns a_cost or 100000000000."""
    return float(_plugin(variant).find_traj(ctypes.byref(params)))


def find_traj(weights_file: Optional[str] = None, variant: str = "trp", iteration: int = 3) -> bool:
    """trp_wrapper.py:99-121: read the tab-separated 10 weights, run find_traj, False iff it failed."""
    if weights_file is None:
        weights_file = os.path.join(os.environ.get("SPECTRAL_IO_DIR", "/home/srujan_d/RISS/code/btrapz/src"),
                                    "weights.txt")
    with open(weights_file) as f:
        vals = [float(v) for v in f.readlines()[0].split("\t")[:10]]
    return _run_btrapz(Params(*vals, iteration), variant) != FAIL_COST


def run_btrapz(trial, variant: str = "trp") -> float:
    """trp_wrapper.py:56-97: the Optuna objective -- 10 weights suggested in [0, 50], iteration = 1."""
    names = ("s_acc_weight", "s_jerk_weight", "l_acc_weight", "l_jerk_weight", "weight_s_ref", "weight_ds_ref",
             "weight_l_ref", "weight_dl_ref", "weight_end_s", "weight_end_l")
    vals = [trial.suggest_float(n, 0, 50) for n in names]
    return _run_btrapz(Params(*vals, 1), variant)
