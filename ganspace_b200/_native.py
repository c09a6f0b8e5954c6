"""ctypes binding of the C-ABI shared library (include/ganspace_b200.h).

There is no CPU fallback: if the library is missing, or a compute entry point is called without a CUDA
device, this module raises.  torch is used only for device memory and streams.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os
from pathlib import Path

import torch

_LIB_PATH = Path(__file__).resolve().parent / "libganspace_b200.so"
_lib = None

# name -> (restype, argtypes); mirrors include/ganspace_b200.h one to one
_P, _I, _L, _Z, _D, _F = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_double, C.c_float
SIGNATURES = {
    "gsb_abi_version": (_I, []),
    "gsb_last_error": (C.c_char_p, []),
    "gsb_legacy_normal_f32": (_I, [_P, _I, _L, _P, _L, _P]),
    "gsb_legacy_truncnorm_f32": (_I, [_P, _I, _L, _D, _D, _F, _P, _L, _P]),
    "gsb_mt19937_raw_u32": (_I, [_P, _I, _L, _P, _L, _P]),
    "gsb_mt19937_jump_polys": (_I, [_L, _I, _P]),
    "gsb_mt19937_jump_state_host": (_I, [C.c_uint32, _P, _P]),
    "gsb_legacy_normal_split_step_words": (_L, [_L, _I]),
    "gsb_legacy_normal_split_workspace_bytes": (_Z, [_I, _L, _I]),
    "gsb_legacy_normal_f32_split": (_I, [_P, _I, _L, _P, _L, _I, _P, _P, _Z, _P]),
    "gsb_legacy_normal_split_status": (_I, [_P, _I, _L, _I, _P, _P]),
    "gsb_mapping_packed_bytes": (_Z, [_I, _I]),
    "gsb_mapping_pack": (_I, [_P, _P, _I, _I, _F, _P, _P]),
    "gsb_mapping_workspace_bytes": (_Z, [_L, _I]),
    "gsb_mapping_forward": (_I, [_P, _I, _I, _P, _P, _L, _I, _P, _Z, _P]),
    "gsb_mapping_status": (_I, [_P, _I, _I, _P]),
    "gsb_linear_forward": (_I, [_P, _P, _P, _P, _L, _I, _I, _I, _P, _Z, _P]),
    "gsb_linear_workspace_bytes": (_Z, [_L, _I, _I, _I]),
    "gsb_leaky_relu": (_I, [_P, _P, _L, _F, _P]),
    "gsb_sg1_packed_bytes": (_Z, [_P, _I, _I]),
    "gsb_sg1_pack": (_I, [_P, _I, _I, _P, _P, _P, _Z, _P]),
    "gsb_sg1_workspace_bytes": (_Z, [_P, _I, _I, _I, _L]),
    "gsb_sg1_forward": (_I, [_P, _P, _I, _I, _I, _I, _P, _I, _L, _P, _L, _P, _Z, _P]),
    "gsb_sg1_status": (_I, [_P, _P, _I, _I, _P]),
    "gsb_batch_stats_workspace_bytes": (_Z, [_L, _I]),
    "gsb_batch_stats": (_I, [_P, _L, _I, _L, _P, _P, _P, _Z, _P]),
    "gsb_batch_stats_multi_workspace_bytes": (_Z, [_I, _L, _I]),
    "gsb_batch_stats_multi": (_I, [_P, _I, _L, _I, _L, _P, _P, _P, _Z, _P]),
    "gsb_ipca_state_bytes": (_Z, [_I, _I]),
    "gsb_ipca_workspace_bytes": (_Z, [_I, _I]),
    "gsb_ipca_reset": (_I, [_P, _I, _I, _P]),
    "gsb_ipca_chain_step": (_I, [_P, _I, _I, _L, _L, _P, _P, _P, _Z, _P]),
    "gsb_ipca_export": (_I, [_P, _I, _I, _L, _P, _P, _P, _P, _P, _P, _P]),
    "gsb_ipca_chain_persistent_supported": (_I, [_I, _I]),
    "gsb_ipca_queue_bytes": (_Z, [_I]),
    "gsb_ipca_queue_reset": (_I, [_P, _I, _P]),
    "gsb_ipca_queue_publish": (_I, [_P, _I, _I, _I, _P, _P, _I, _I, _I, _I, _I, _P]),
    "gsb_ipca_chain_run": (_I, [_P, _I, _I, _L, _P, _I, _I, _I, _P, _Z, _P]),
    "gsb_sym_eig_top": (_I, [_P, _I, _I, _P, _P, _P, _Z, _P]),
    "gsb_eig_status": (_I, [_P, _P]),
    "gsb_project_std_workspace_bytes": (_Z, [_I]),
    "gsb_project_std": (_I, [_P, _L, _I, _L, _P, _I, _P, _P, _P, _Z, _P]),
    "gsb_linreg_state_bytes": (_Z, [_I, _I]),
    "gsb_linreg_reset": (_I, [_P, _I, _I, _P]),
    "gsb_linreg_workspace_bytes": (_Z, [_L, _I]),
    "gsb_linreg_accumulate": (_I, [_P, _I, _I, _P, _L, _I, _P, _P, _P, _P, _P, _Z, _P]),
    "gsb_linreg_solve": (_I, [_P, _I, _I, _L, _P, _P, _P]),
    "gsb_linreg_solve_status": (_I, [_P, _I, _I, _P, _P]),
    "gsb_linreg_normal_matrix": (_P, [_P, _I, _I]),
    "gsb_linreg_solve_pinv": (_I, [_P, _I, _I, _P, _P, _D, _P, _P]),
    "gsb_ipca_set_chain_mode": (_I, [_I]),
    "gsb_synthesis_packed_bytes": (_Z, [_P, _I, _I]),
    "gsb_synthesis_pack": (_I, [_P, _I, _I, _P, _P, _Z, _P]),
    "gsb_synthesis_workspace_bytes": (_Z, [_P, _I, _L]),
    "gsb_synthesis_forward": (_I, [_P, _P, _I, _I, _I, _P, _L, _P, _L, _P, _Z, _P]),
    "gsb_synthesis_status": (_I, [_P, _P, _I, _I, _P]),
    "gsb_synthesis_render_workspace_bytes": (_Z, [_P, _I, _L, _I]),
    "gsb_synthesis_render": (_I, [_P, _P, _I, _I, _I, _P, _I, _P, _I, _L, _P, _L, _P, _P, _Z, _P]),
    "gsb_bigd_rows": (_I, [_I, _I]),
    "gsb_bigd_state_bytes": (_Z, [_L, _I]),
    "gsb_bigd_workspace_bytes": (_Z, [_L, _I, _I, _I]),
    "gsb_bigd_reset": (_I, [_P, _P, _L, _I, _I, _P]),
    "gsb_bigd_chain_step": (_I, [_P, _P, _L, _I, _I, _L, _I, _I, _P, _P, _Z, _P]),
    "gsb_bigd_export": (_I, [_P, _P, _L, _I, _L, _P, _P, _P, _P, _P, _P, _P]),
    "gsb_bigd_gram_matrix": (_P, [_P, _L, _I, _I]),
    "gsb_bigd_step_gram": (_I, [_P, _P, _L, _I, _I, _L, _I, _I, _P, _P, _Z, _P]),
    "gsb_bigd_step_solve": (_I, [_P, _P, _L, _I, _I, _L, _I, _I, _P, _P, _Z, _P]),
    "gsb_bigd_step_commit": (_I, [_P, _P, _L, _I, _I, _L, _I, _I, _P, _P, _Z, _P]),
}


class StyledConvDesc(C.Structure):
    """``gsb_styled_conv`` of include/ganspace_b200.h (device pointers to the module's fp32 parameters)."""
    _fields_ = [("conv_weight", C.c_void_p), ("mod_weight", C.c_void_p), ("mod_bias", C.c_void_p),
                ("act_bias", C.c_void_p), ("noise", C.c_void_p), ("noise_weight", C.c_void_p),
                ("cin", C.c_int), ("cout", C.c_int), ("upsample", C.c_int), ("res_in", C.c_int)]


class ToRGBDesc(C.Structure):
    """``gsb_to_rgb`` of include/ganspace_b200.h."""
    _fields_ = [("conv_weight", C.c_void_p), ("mod_weight", C.c_void_p), ("mod_bias", C.c_void_p), ("bias", C.c_void_p),
                ("cin", C.c_int)]


class SG1LayerDesc(C.Structure):
    """``gsb_sg1_layer`` of include/ganspace_b200.h."""
    _fields_ = [("kind", C.c_int), ("cin", C.c_int), ("cout", C.c_int), ("res_out", C.c_int), ("weight", C.c_void_p),
                ("bias", C.c_void_p), ("noise_weight", C.c_void_p), ("noise", C.c_void_p), ("style_weight", C.c_void_p),
                ("style_bias", C.c_void_p)]


class NativeError(RuntimeError):
    pass


def lib_path() -> Path:
    return _LIB_PATH


def load():
    """Load libganspace_b200.so (built in-tree by ``__graft_entry__.build()`` / csrc/Makefile)."""
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise NativeError(
                f"{_LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). ganspace_b200 has no CPU fallback.")
        lib = C.CDLL(str(_LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the header and the library drift apart
            fn.restype, fn.argtypes = res, args
        if lib.gsb_abi_version() != 1:
            raise NativeError("ABI version mismatch between ganspace_b200/_native.py and the library")
        _lib = lib
    return _lib


def require_cuda(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise NativeError("ganspace_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    dev = torch.device(device if device is not None else "cuda")
    if dev.type != "cuda":
        raise NativeError(f"ganspace_b200 runs on CUDA devices only, got {dev}")
    return dev


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    if t is None:
        return C.c_void_p(0)
    assert t.is_cuda and t.is_contiguous(), "device-contiguous tensor expected"
    return C.c_void_p(t.data_ptr())


def _check(rc: int, what: str):
    if rc != 0:
        raise NativeError(f"{what} failed ({rc}): {load().gsb_last_error().decode()}")


class _Instrument:
    """Launch counter and optional per-section CUDA-event timers (used by bench.py for the roofline).

    ``launches`` counts the kernels this library enqueued (each C-ABI call launches a fixed number).
    When ``timing`` is on, sections wrap their C call in a pair of events recorded on the launching
    stream; ``section_ms()`` sums them after a synchronize."""

    def __init__(self):
        self.launches = 0
        self.timing = False
        self._events = {}
        self.rows = {}
        self.timeline = [] if os.environ.get("GANSPACE_B200_TIMELINE") == "1" else None

    def reset(self):
        self.launches = 0
        self._events = {}
        self.rows = {}

    def mark(self, name):
        """GANSPACE_B200_TIMELINE=1: a timed event on the current stream (tools/phase_probe.py prints them)."""
        if self.timeline is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(torch.cuda.current_stream())
            self.timeline.append((name, ev))

    def timeline_ms(self):
        torch.cuda.synchronize()
        t0 = self.timeline[0][1]
        return [(n, t0.elapsed_time(e)) for n, e in self.timeline]

    def add_rows(self, name, n):
        """rows (samples) a section's kernels processed -- the roofline's unit count (bench.py)."""
        self.rows[name] = self.rows.get(name, 0) + int(n)

    def count(self, n):
        self.launches += n

    class _Sec:
        def __init__(self, outer, name):
            self.o, self.name = outer, name

        def __enter__(self):
            if self.o.timing:
                self.e0 = torch.cuda.Event(enable_timing=True)
                self.e1 = torch.cuda.Event(enable_timing=True)
                self.e0.record(torch.cuda.current_stream())

        def __exit__(self, *a):
            if self.o.timing:
                self.e1.record(torch.cuda.current_stream())
                self.o._events.setdefault(self.name, []).append((self.e0, self.e1))
            self.o.mark(self.name + " done")

    def section(self, name):
        return self._Sec(self, name)

    def section_ms(self):
        torch.cuda.synchronize()
        return {k: (sum(a.elapsed_time(b) for a, b in v), len(v)) for k, v in self._events.items()}


instrument = _Instrument()

# the kernels behind each timed section (bench.py's roofline names the one it reports)
SECTION_KERNELS = {
    "mapping": "mapping MLP: pixelnorm_split + 8 x mapping_layer_tc_kernel (tcgen05, fp16 hi/lo x3)",
    "linear": "gen_z linear: mapping_layer_tc_kernel (tcgen05, fp16 hi/lo x3, bias epilogue, TMA store) for n >= 128",
    "synthesis": "StyledConv chain: tap-GEMM tc_gemm_plain (tcgen05) + gather/scatter/blur epilogues",
}


def kernel_name(section: str) -> str:
    if section == "mapping" and os.environ.get("GANSPACE_B200_MAPPING", MAPPING_DEFAULT) == "simt":
        return "mapping MLP: pixelnorm + 8 x sgemm_tn_bias_act_kernel (fp32 FMA)"
    return SECTION_KERNELS.get(section, section)


class _Scratch:
    """Grow-only per-device scratch buffers keyed by purpose (the C ABI never allocates)."""

    def __init__(self):
        self._bufs = {}

    def get(self, key, nbytes: int, device) -> torch.Tensor:
        k = (key, str(device))
        buf = self._bufs.get(k)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
            self._bufs[k] = buf
        return buf

    def clear(self):
        self._bufs.clear()


scratch = _Scratch()


# ------------------------------------------------------------------------------------------------
# thin tensor-level wrappers
# ------------------------------------------------------------------------------------------------
_jump_polys = {}        # (step_words, count) -> host table; (step_words, count, device) -> device copy


def jump_polys(n_per_stream: int, parts: int, device) -> torch.Tensor:
    """Device copy of the MT19937 jump polynomials for streams of n_per_stream normals split into `parts` sub-streams
    (computed once per process on the host, ~0.1 s; csrc/rng_jump.cu)."""
    import numpy as np
    lib = load()
    step = int(lib.gsb_legacy_normal_split_step_words(int(n_per_stream), int(parts)))
    key = (step, parts - 1)
    if key not in _jump_polys:
        table = np.zeros((parts - 1, 624), np.uint32)
        _check(lib.gsb_mt19937_jump_polys(step, parts - 1, table.ctypes.data_as(C.c_void_p)), "gsb_mt19937_jump_polys")
        _jump_polys[key] = table
    dkey = key + (str(device),)
    if dkey not in _jump_polys:
        _jump_polys[dkey] = torch.from_numpy(_jump_polys[key].view(np.int32)).to(device)
    return _jump_polys[dkey]


def split_parts(n_per_stream: int) -> int:
    """CTAs per stream: long streams (a 10k-row batch = 5.12M normals = 8.6 ms on one SM) are generated by up to 8 CTAs."""
    env = os.environ.get("GANSPACE_B200_RNG_PARTS")
    if env:
        return max(1, min(16, int(env)))
    if n_per_stream % 2:
        return 1
    return max(1, min(8, n_per_stream // 600_000))


def legacy_normal(seeds, n_per_stream: int, device, out=None, parts: int = 1, scratch_key: str = "rng_split") -> torch.Tensor:
    """RandomState(seed).standard_normal(n_per_stream).astype(float32) for every seed -> [S, n].
    ``parts`` > 1: every stream is generated by that many CTAs (MT19937 jump-ahead), bit-identical output."""
    lib = load()
    dev = require_cuda(device)
    # ``seeds``: a list of ints, or an int32 device tensor from seeds_tensor() (no host->device copy on this call: a copy
    # issued behind a long kernel would block the host until that kernel has finished)
    seeds_dev = seeds if isinstance(seeds, torch.Tensor) else _seeds_tensor(seeds, dev)
    assert seeds_dev.is_cuda and seeds_dev.dtype == torch.int32 and seeds_dev.is_contiguous()
    S = seeds_dev.numel()
    if out is None:
        out = torch.empty((S, n_per_stream), dtype=torch.float32, device=dev)
    assert out.is_cuda and out.is_contiguous() and out.numel() >= S * n_per_stream
    if parts > 1 and S > 0 and n_per_stream >= 2 and n_per_stream % 2 == 0:
        polys = jump_polys(n_per_stream, parts, dev)
        ws = scratch.get(scratch_key, lib.gsb_legacy_normal_split_workspace_bytes(S, n_per_stream, parts), dev)
        with torch.cuda.device(dev), instrument.section("rng"):
            _check(lib.gsb_legacy_normal_f32_split(_ptr(seeds_dev), S, n_per_stream, _ptr(out), n_per_stream, parts, _ptr(polys),
                                                   _ptr(ws), ws.numel(), _stream()), "gsb_legacy_normal_f32_split")
        instrument.count(2)
        return out
    with torch.cuda.device(dev), instrument.section("rng"):
        _check(lib.gsb_legacy_normal_f32(_ptr(seeds_dev), S, n_per_stream, _ptr(out), n_per_stream, _stream()),
               "gsb_legacy_normal_f32")
    instrument.count(1)
    return out


def seeds_tensor(seeds, dev):
    return _seeds_tensor(seeds, dev)


def rng_split_status(n_streams: int, n_per_stream: int, parts: int, device) -> int:
    """Status word of the last split launch of this shape on ``device`` (0 = fine; synchronises)."""
    lib = load()
    dev = require_cuda(device)
    ws = scratch.get("rng_split", lib.gsb_legacy_normal_split_workspace_bytes(n_streams, n_per_stream, parts), dev)
    flags = C.c_uint(0)
    with torch.cuda.device(dev):
        _check(lib.gsb_legacy_normal_split_status(_ptr(ws), n_streams, n_per_stream, parts, C.byref(flags), _stream()),
               "gsb_legacy_normal_split_status")
    return int(flags.value)


def _seeds_tensor(seeds, dev):
    """uint32 seeds carried in an int32 tensor (two's-complement reinterpretation)."""
    vals = [(int(s) & 0xFFFFFFFF) for s in seeds]
    vals = [v - (1 << 32) if v >= (1 << 31) else v for v in vals]
    return torch.tensor(vals, dtype=torch.int32, device=dev)


def legacy_truncnorm(seeds, n_per_stream: int, lo: float, hi: float, scale: float, device) -> torch.Tensor:
    lib = load()
    dev = require_cuda(device)
    sd = _seeds_tensor(seeds, dev)
    out = torch.empty((sd.numel(), n_per_stream), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _check(lib.gsb_legacy_truncnorm_f32(_ptr(sd), sd.numel(), n_per_stream, lo, hi, scale, _ptr(out),
                                            n_per_stream, _stream()), "gsb_legacy_truncnorm_f32")
    return out


def mt19937_raw(seeds, n_per_stream: int, device) -> torch.Tensor:
    lib = load()
    dev = require_cuda(device)
    sd = _seeds_tensor(seeds, dev)
    out = torch.empty((sd.numel(), n_per_stream), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _check(lib.gsb_mt19937_raw_u32(_ptr(sd), sd.numel(), n_per_stream, _ptr(out), n_per_stream, _stream()),
               "gsb_mt19937_raw_u32")
    return out


# default mapping-network path: "tc" = tcgen05 fp16x3 split (fp32-grade), "simt" = fp32 FMA kernels
MAPPING_DEFAULT = "tc"


class PackedMapping:
    """Pre-scaled mapping-network weights in the layout the kernels read (gsb_mapping_pack)."""

    def __init__(self, weight: torch.Tensor, bias: torch.Tensor, lr_mul: float):
        lib = load()
        dev = require_cuda(weight.device)
        self.n_layers, self.dim = int(weight.shape[0]), int(weight.shape[1])
        assert weight.shape == (self.n_layers, self.dim, self.dim) and bias.shape == (self.n_layers, self.dim)
        self.device = dev
        self.packed = torch.empty(lib.gsb_mapping_packed_bytes(self.n_layers, self.dim), dtype=torch.uint8, device=dev)
        w = weight.detach().to(dev, torch.float32).contiguous()
        b = bias.detach().to(dev, torch.float32).contiguous()
        with torch.cuda.device(dev):
            _check(lib.gsb_mapping_pack(_ptr(w), _ptr(b), self.n_layers, self.dim, float(lr_mul),
                                        _ptr(self.packed), _stream()), "gsb_mapping_pack")

    def check(self):
        """Raise if the tensor-core path saw an activation outside fp16's range (synchronises)."""
        flags = C.c_uint(0)
        with torch.cuda.device(self.device):
            _check(load().gsb_mapping_status(_ptr(self.packed), self.n_layers, self.dim, C.byref(flags)),
                   "gsb_mapping_status")
        if flags.value & 1:
            raise NativeError("mapping network: an activation exceeded fp16 range in the tensor-core path; "
                              "results are invalid (set GANSPACE_B200_MAPPING=simt)")

    def forward(self, z: torch.Tensor, out: torch.Tensor = None, pixelnorm: bool = True,
                force_simt: bool = None, leave_free_sms: int = 0) -> torch.Tensor:
        lib = load()
        if force_simt is None:
            force_simt = os.environ.get("GANSPACE_B200_MAPPING", MAPPING_DEFAULT) == "simt"
        assert z.is_cuda and z.dtype == torch.float32 and z.shape[-1] == self.dim
        z2 = z.reshape(-1, self.dim)
        if not z2.is_contiguous():
            z2 = z2.contiguous()
        n = z2.shape[0]
        if out is None:
            out = torch.empty_like(z2)
        ws_bytes = lib.gsb_mapping_workspace_bytes(n, self.dim)
        ws = scratch.get("mapping", ws_bytes, z.device)
        flags = (1 if pixelnorm else 0) | (2 if force_simt else 0) | ((int(leave_free_sms) & 0xff) << 8)
        with torch.cuda.device(z.device), instrument.section("mapping"):
            _check(lib.gsb_mapping_forward(_ptr(self.packed), self.n_layers, self.dim, _ptr(z2), _ptr(out), n,
                                           flags, _ptr(ws), ws.numel(), _stream()), "gsb_mapping_forward")
        instrument.count(self.n_layers + (1 if pixelnorm else 0))
        instrument.add_rows("mapping", n)
        return out.reshape(z.shape)


def linear(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor = None, lrelu: bool = False, bounded: bool = False) -> torch.Tensor:
    """y = x @ w.T (+ bias); x [n,K], w [N,K] (N % 128 == 0, K % 16 == 0).  ``bounded`` (|x| < 6e4 guaranteed by the caller)
    lets n >= 128, N % 256 == 0, K % 64 == 0 run on the tensor cores (fp32-grade); otherwise the fp32 FMA GEMM kernel."""
    lib = load()
    assert x.is_cuda and x.dtype == torch.float32 and w.dtype == torch.float32 and x.shape[-1] == w.shape[1]
    x2 = x.reshape(-1, x.shape[-1]).contiguous()
    w = w.contiguous()
    n, K = x2.shape
    N = w.shape[0]
    y = torch.empty((n, N), dtype=torch.float32, device=x.device)
    flags = (1 if lrelu else 0) | (2 if bounded else 0)
    ws = scratch.get("linear", lib.gsb_linear_workspace_bytes(n, N, K, flags), x.device)
    with torch.cuda.device(x.device), instrument.section("linear"):
        _check(lib.gsb_linear_forward(_ptr(x2), _ptr(w), _ptr(bias.contiguous() if bias is not None else None), _ptr(y),
                                      n, N, K, flags, _ptr(ws), ws.numel(), _stream()), "gsb_linear_forward")
    instrument.count(5 if (bounded and n >= 128 and N % 256 == 0 and K % 64 == 0) else 1)
    instrument.add_rows("linear", n)
    return y.reshape(*x.shape[:-1], N)


def leaky_relu(x: torch.Tensor, slope: float = 0.2) -> torch.Tensor:
    """leaky_relu(x, slope) without gain (StyleGAN's G_mapping activation)."""
    lib = load()
    assert x.is_cuda and x.dtype == torch.float32
    x2 = x.contiguous()
    y = torch.empty_like(x2)
    with torch.cuda.device(x.device):
        _check(lib.gsb_leaky_relu(_ptr(x2), _ptr(y), x2.numel(), float(slope), _stream()), "gsb_leaky_relu")
    instrument.count(1)
    return y.reshape(x.shape)


def mapping_pixelnorm(z: torch.Tensor) -> torch.Tensor:
    """PixelNorm alone (stylegan2-pytorch/model.py:14-19)."""
    lib = load()
    assert z.is_cuda and z.dtype == torch.float32
    dim = z.shape[-1]
    z2 = z.reshape(-1, dim).contiguous()
    out = torch.empty_like(z2)
    ws = scratch.get("mapping", lib.gsb_mapping_workspace_bytes(z2.shape[0], dim), z.device)
    with torch.cuda.device(z.device):
        _check(lib.gsb_mapping_forward(C.c_void_p(0), 0, dim, _ptr(z2), _ptr(out), z2.shape[0], 1, _ptr(ws),
                                       ws.numel(), _stream()), "gsb_mapping_forward")
    return out.reshape(z.shape)


def batch_stats(x: torch.Tensor, mean_out: torch.Tensor = None, gram_out: torch.Tensor = None):
    """(mean[d] fp64, centred Gram[d,d] fp64) of x[n,d] fp32."""
    lib = load()
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    n, d = x.shape
    ld = x.stride(0)
    if mean_out is None:
        mean_out = torch.empty(d, dtype=torch.float64, device=x.device)
    if gram_out is None:
        gram_out = torch.empty((d, d), dtype=torch.float64, device=x.device)
    ws_bytes = lib.gsb_batch_stats_workspace_bytes(n, d)
    ws = scratch.get("stats", ws_bytes, x.device)
    with torch.cuda.device(x.device), instrument.section("stats"):
        _check(lib.gsb_batch_stats(C.c_void_p(x.data_ptr()), n, d, ld, _ptr(mean_out), _ptr(gram_out), _ptr(ws),
                                   ws.numel(), _stream()), "gsb_batch_stats")
    instrument.count(3)
    return mean_out, gram_out


def batch_stats_multi(x: torch.Tensor, n_groups: int, rows_per_group: int, mean_out: torch.Tensor = None,
                      gram_out: torch.Tensor = None):
    """(mean[G,d] fp64, centred Gram[G,d,d] fp64) of G consecutive groups of rows of x[G*rows, d] fp32, one set of launches."""
    lib = load()
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    assert x.shape[0] >= n_groups * rows_per_group
    d, ld = x.shape[1], x.stride(0)
    mean = mean_out if mean_out is not None else torch.empty((n_groups, d), dtype=torch.float64, device=x.device)
    gram = gram_out if gram_out is not None else torch.empty((n_groups, d, d), dtype=torch.float64, device=x.device)
    assert mean.shape == (n_groups, d) and gram.shape == (n_groups, d, d) and mean.dtype == gram.dtype == torch.float64
    ws_bytes = lib.gsb_batch_stats_multi_workspace_bytes(n_groups, rows_per_group, d)
    ws = scratch.get("stats", ws_bytes, x.device)
    with torch.cuda.device(x.device), instrument.section("stats"):
        _check(lib.gsb_batch_stats_multi(C.c_void_p(x.data_ptr()), n_groups, rows_per_group, d, ld, _ptr(mean), _ptr(gram),
                                         _ptr(ws), ws.numel(), _stream()), "gsb_batch_stats_multi")
    instrument.count(4 if (d % 128 == 0 and d <= 1024) else 3 * n_groups)
    return mean, gram


class IPCAChain:
    """Device-resident IncrementalPCA state + the Gram-form chain step (small-d engine).

    The chain is the sequential part of a run (K dependent eigensolves), so its steps are enqueued on a
    dedicated high-priority stream: step k waits only for the statistics of group k (an event on the
    producing stream) and runs while the main stream already generates / reduces the next groups."""

    def __init__(self, d: int, c: int, device, side_stream: bool = True):
        lib = load()
        self.dev = require_cuda(device)
        self.d, self.c = int(d), int(c)
        self.state = torch.empty(lib.gsb_ipca_state_bytes(self.d, self.c), dtype=torch.uint8, device=self.dev)
        self.ws = torch.empty(lib.gsb_ipca_workspace_bytes(self.d, self.c), dtype=torch.uint8, device=self.dev)
        self.n_seen = 0
        self.stream = None
        if side_stream and os.environ.get("GANSPACE_B200_CHAIN_STREAM", "1") != "0":
            with torch.cuda.device(self.dev):
                self.stream = torch.cuda.Stream(device=self.dev, priority=-1)
        with torch.cuda.device(self.dev):
            _check(lib.gsb_ipca_reset(_ptr(self.state), self.d, self.c, _stream()), "gsb_ipca_reset")
            if self.stream is not None:
                self.stream.wait_stream(torch.cuda.current_stream())

    def step(self, n_batch: int, mean_b: torch.Tensor, gram_b: torch.Tensor):
        lib = load()
        assert mean_b.dtype == torch.float64 and gram_b.dtype == torch.float64
        with torch.cuda.device(self.dev):
            if self.stream is not None:
                self.stream.wait_stream(torch.cuda.current_stream())      # statistics of this group are ready
                mean_b.record_stream(self.stream)
                gram_b.record_stream(self.stream)
                ctx = torch.cuda.stream(self.stream)
            else:
                ctx = contextlib.nullcontext()
            with ctx, instrument.section("chain"):
                _check(lib.gsb_ipca_chain_step(_ptr(self.state), self.d, self.c, self.n_seen, int(n_batch),
                                               _ptr(mean_b), _ptr(gram_b), _ptr(self.ws), self.ws.numel(), _stream()),
                       "gsb_ipca_chain_step")
        # kernels per step: first step = direct solve (8) + seeding of the subspace form (1); later steps = one cluster
        # launch (orthogonal iteration, csrc/subspace.cu).  Shapes outside the subspace kernel's range: direct solve (8).
        subspace = (self.d % 128 == 0 and 128 <= self.d <= 512 and self.c % 8 == 0 and 8 <= self.c <= 128
                    and os.environ.get("GANSPACE_B200_CHAIN", "") not in ("direct", "lanczos") and not _chain_forced_direct)
        instrument.count((1 if self.n_seen > 0 else 9) if subspace else 8)
        self.n_seen += int(n_batch)

    # ---- persistent run: ONE resident cluster kernel for steps 1 .. K-1, fed through a device queue (csrc/subspace.cu) --------
    def begin_run(self, n_groups: int, n_batch: int) -> bool:
        """Declare a run of ``n_groups`` equal batches.  Returns False (and changes nothing) when the shape has no persistent
        kernel or GANSPACE_B200_CHAIN_PERSISTENT=0; then every step() is its own launch."""
        lib = load()
        # Opt-in (GANSPACE_B200_CHAIN_PERSISTENT=1).  Measured on config 2: no gain over one launch per step once the producers
        # leave SMs free, and a hazard: with CUDA's lazy module loading the first launch of any not-yet-loaded kernel blocks until
        # the resident kernel exits (it then gives up after its timeout).  Use with CUDA_MODULE_LOADING=EAGER or after a warm-up.
        if (n_groups < 2 or self.n_seen != 0 or os.environ.get("GANSPACE_B200_CHAIN_PERSISTENT", "0") != "1"
                or not lib.gsb_ipca_chain_persistent_supported(self.d, self.c)):
            return False
        self._run = {"K": int(n_groups), "nb": int(n_batch), "next": 0, "keep": [], "closed": False}
        self._queue = torch.empty(lib.gsb_ipca_queue_bytes(n_groups), dtype=torch.uint8, device=self.dev)
        with torch.cuda.device(self.dev):
            _check(lib.gsb_ipca_queue_reset(_ptr(self._queue), n_groups, _stream()), "gsb_ipca_queue_reset")
        return True

    def _publish(self, k0, count, mean_base, gram_base, flag, round_first=0, world=1, per_rank=1):
        with torch.cuda.device(self.dev):
            _check(load().gsb_ipca_queue_publish(_ptr(self._queue), self._run["K"], int(k0), int(count), _ptr(mean_base), _ptr(gram_base),
                                                 self.d, int(round_first), int(world), int(per_rank), int(flag), _stream()),
                   "gsb_ipca_queue_publish")
        instrument.count(1)

    def run_step(self, n_batch: int, mean_b: torch.Tensor, gram_b: torch.Tensor):
        """step() inside a declared run: group 0 is solved directly and followed by the launch of the resident kernel; later
        groups are handed to it through the queue (the tensors are kept alive until the run ends)."""
        run = self._run
        k = run["next"]
        assert not run["closed"] and k < run["K"] and int(n_batch) == run["nb"], "persistent chain: unexpected batch"
        if k == 0:
            self.step(n_batch, mean_b, gram_b)
            lib = load()
            with torch.cuda.device(self.dev):
                stream = self.stream if self.stream is not None else torch.cuda.current_stream()
                if self.stream is not None:
                    self.stream.wait_stream(torch.cuda.current_stream())       # the queue has been reset
                with torch.cuda.stream(stream):
                    _check(lib.gsb_ipca_chain_run(_ptr(self.state), self.d, self.c, run["nb"], _ptr(self._queue), run["K"], 1, run["K"],
                                                  _ptr(self.ws), self.ws.numel(), _stream()), "gsb_ipca_chain_run")
            instrument.count(1)
        else:
            assert mean_b.dtype == torch.float64 and gram_b.dtype == torch.float64 and mean_b.is_contiguous() and gram_b.is_contiguous()
            run["keep"].append((mean_b, gram_b))
            self._publish(k, 1, mean_b, gram_b, 1)
            self.n_seen += int(n_batch)
        run["next"] = k + 1

    def end_run(self):
        """Close a declared run: if fewer than K groups were published (interrupt, early stop) tell the kernel to stop there."""
        run = getattr(self, "_run", None)
        if run is None or run["closed"]:
            return
        run["closed"] = True
        if 1 <= run["next"] < run["K"]:
            self._publish(run["next"], 1, None, None, 2)

    def join(self):
        """Make the current stream wait for every chain step enqueued so far."""
        self.end_run()
        if self.stream is not None:
            with torch.cuda.device(self.dev):
                torch.cuda.current_stream().wait_stream(self.stream)

    def export(self):
        lib = load()
        self.join()
        f64 = dict(dtype=torch.float64, device=self.dev)
        out = {
            "components": torch.empty((self.c, self.d), **f64), "singular_values": torch.empty(self.c, **f64),
            "mean": torch.empty(self.d, **f64), "var": torch.empty(self.d, **f64),
            "explained_variance": torch.empty(self.c, **f64),
            "explained_variance_ratio": torch.empty(self.c, **f64),
        }
        with torch.cuda.device(self.dev):
            _check(lib.gsb_ipca_export(_ptr(self.state), self.d, self.c, self.n_seen, _ptr(out["components"]),
                                       _ptr(out["singular_values"]), _ptr(out["mean"]), _ptr(out["var"]),
                                       _ptr(out["explained_variance"]), _ptr(out["explained_variance_ratio"]),
                                       _stream()), "gsb_ipca_export")
            check_eig_status("IPCAChain.export")
        instrument.count(1)
        return out


class ChainNotConverged(NativeError):
    """A chain step reached its iteration cap before its residual tolerance (no spectral gap after component c)."""


_chain_forced_direct = False


def set_chain_mode(direct: bool):
    """Every chain step enqueued from now on is the exact direct eigen-solve (True) / the default solver (False)."""
    global _chain_forced_direct
    _check(load().gsb_ipca_set_chain_mode(1 if direct else 0), "gsb_ipca_set_chain_mode")
    _chain_forced_direct = bool(direct)


def check_eig_status(what: str):
    """Raise if a chain kernel reported a failure since the last check (synchronises the current stream)."""
    flags = C.c_uint(0)
    _check(load().gsb_eig_status(C.byref(flags), _stream()), "gsb_eig_status")
    if flags.value:
        if flags.value & 8:
            raise NativeError(f"{what}: the resident chain kernel waited longer than GANSPACE_B200_CHAIN_TIMEOUT_S for a group's "
                              f"statistics and gave up (status {flags.value})")
        raise ChainNotConverged(f"{what}: a chain step hit its iteration cap without reaching the residual tolerance "
                                f"(status {flags.value}): the spectrum has no gap after component c (numerical rank below "
                                "n_components?); the exact route is GANSPACE_B200_CHAIN=direct (decomposition.compute re-runs "
                                "through it by itself)")


def sym_eig_top(a: torch.Tensor, c: int):
    lib = load()
    assert a.is_cuda and a.dtype == torch.float64 and a.dim() == 2 and a.shape[0] == a.shape[1]
    d = a.shape[0]
    a = a.contiguous().clone()
    evals = torch.empty(c, dtype=torch.float64, device=a.device)
    evecs = torch.empty((c, d), dtype=torch.float64, device=a.device)
    ws = torch.empty(lib.gsb_ipca_workspace_bytes(d, c), dtype=torch.uint8, device=a.device)
    with torch.cuda.device(a.device):
        _check(lib.gsb_sym_eig_top(_ptr(a), d, c, _ptr(evals), _ptr(evecs), _ptr(ws), ws.numel(), _stream()),
               "gsb_sym_eig_top")
        check_eig_status("sym_eig_top")
    return evals, evecs


def project_std(x: torch.Tensor, dirs: torch.Tensor, sub: torch.Tensor = None) -> torch.Tensor:
    lib = load()
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    n, d = x.shape
    dirs = dirs.to(x.device, torch.float32).contiguous()
    c = dirs.shape[0]
    assert dirs.shape[1] == d
    if sub is not None:
        sub = sub.to(x.device, torch.float64).contiguous()
    out = torch.empty(c, dtype=torch.float32, device=x.device)
    ws = scratch.get("projstd", lib.gsb_project_std_workspace_bytes(c), x.device)
    with torch.cuda.device(x.device):
        _check(lib.gsb_project_std(C.c_void_p(x.data_ptr()), n, d, x.stride(0), _ptr(dirs), c, _ptr(sub), _ptr(out),
                                   _ptr(ws), ws.numel(), _stream()), "gsb_project_std")
    instrument.count(2)
    return out


class LinregAccumulator:
    """Normal-equation accumulators of the latent regression (decomposition.py:77-139)."""

    def __init__(self, c: int, latent_dim: int, device):
        lib = load()
        self.dev = require_cuda(device)
        self.c, self.L = int(c), int(latent_dim)
        self.state = torch.empty(lib.gsb_linreg_state_bytes(self.c, self.L), dtype=torch.uint8, device=self.dev)
        self.n_total = 0
        with torch.cuda.device(self.dev):
            _check(lib.gsb_linreg_reset(_ptr(self.state), self.c, self.L, _stream()), "gsb_linreg_reset")

    def accumulate(self, act, comp32, mean32, stdev32, z):
        lib = load()
        n, d = act.shape
        act, comp32, mean32, stdev32, z = (t.contiguous() for t in (act, comp32, mean32, stdev32, z))
        assert z.shape == (n, self.L) and comp32.shape == (self.c, d)
        ws = scratch.get("linreg", lib.gsb_linreg_workspace_bytes(n, self.c), self.dev)
        with torch.cuda.device(self.dev):
            _check(lib.gsb_linreg_accumulate(_ptr(self.state), self.c, self.L, _ptr(act), n, d, _ptr(comp32),
                                             _ptr(mean32), _ptr(stdev32), _ptr(z), _ptr(ws), ws.numel(), _stream()),
                   "gsb_linreg_accumulate")
        instrument.count(2)
        self.n_total += n

    RCOND = 1e-6        # eigenvalues of A^T A below RCOND * largest count as zero in the minimum-norm fallback

    def solve(self):
        """(M_t [c, L], Z_mean [L]) fp64.  Well-conditioned normal equations (the usual case: the columns of A are unit-variance
        PC coordinates) are solved by Cholesky; if a pivot fails, the minimum-norm least-squares solution is formed from the
        eigen-decomposition of A^T A -- what scipy's gelsd (decomposition.py:133) returns for a rank-deficient A."""
        lib = load()
        M = torch.zeros((self.c, self.L), dtype=torch.float64, device=self.dev)
        zmean = torch.empty(self.L, dtype=torch.float64, device=self.dev)
        info = C.c_int(0)
        with torch.cuda.device(self.dev):
            _check(lib.gsb_linreg_solve(_ptr(self.state), self.c, self.L, self.n_total, _ptr(M), _ptr(zmean), _stream()),
                   "gsb_linreg_solve")
            _check(lib.gsb_linreg_solve_status(_ptr(self.state), self.c, self.L, C.byref(info), _stream()), "gsb_linreg_solve_status")
        instrument.count(1)
        self.rank_deficient_at = int(info.value)
        if info.value != 0:
            n = (self.c + 31) // 32 * 32                      # the eigensolver wants a multiple of 32: pad with a -1 diagonal
            off = int(lib.gsb_linreg_normal_matrix(_ptr(self.state), self.c, self.L)) - self.state.data_ptr()
            ata = self.state[off:off + self.c * self.c * 8].view(torch.float64).view(self.c, self.c)
            if not bool(torch.isfinite(ata).all()):
                raise NativeError("latent regression: the normal equations contain non-finite entries (a zero or NaN stdev "
                                  "column?); scipy's lstsq raises on such input as well")
            pad = torch.zeros((n, n), dtype=torch.float64, device=self.dev)
            pad[:self.c, :self.c] = ata
            if n > self.c:
                pad[self.c:, self.c:] = -torch.eye(n - self.c, dtype=torch.float64, device=self.dev)
            evals, evecs = sym_eig_top(pad, self.c)           # padding eigenvalues (-1) sort last and are not returned
            evecs = evecs[:, :self.c].contiguous()
            with torch.cuda.device(self.dev):
                _check(lib.gsb_linreg_solve_pinv(_ptr(self.state), self.c, self.L, _ptr(evals), _ptr(evecs), self.RCOND, _ptr(M),
                                                 _stream()), "gsb_linreg_solve_pinv")
            instrument.count(9)
        return M, zmean


class PackedSG1:
    """StyleGAN (v1) synthesis network packed for csrc/synthesis_sg1.cu (gsb_sg1_pack).

    ``layers``: dicts with kind ('const' | 'same' | 'nearest' | 'fused'), weight (const [c,4,4] or conv weight [co,ci,3,3]),
    bias [co], noise_weight [co], noise [r,r], style_weight [2co, dlatent], style_bias [2co] (fp32 tensors), cin, cout, res_out;
    ``rgb_weight`` [3, c_last] and ``rgb_bias`` [3] of torgb."""
    KINDS = {"const": 0, "same": 1, "nearest": 2, "fused": 3}
    STOPS = {"epi": 0, "conv": 1, "style": 2, "image": 3}

    def __init__(self, layers, rgb_weight: torch.Tensor, rgb_bias: torch.Tensor, dlatent: int = 512):
        lib = load()
        self.device = require_cuda(rgb_weight.device)
        self.dlatent = int(dlatent)
        self.n_layers = len(layers)
        self.desc = (SG1LayerDesc * self.n_layers)()
        self.shapes = []                        # (res_out, cout) per layer
        f32 = lambda t: t.detach().to(self.device, torch.float32).contiguous()
        keep = []
        for i, L in enumerate(layers):
            ts = {k: f32(L[k]) for k in ("weight", "bias", "noise_weight", "noise", "style_weight", "style_bias")}
            keep.append(ts)
            d = self.desc[i]
            for k, t in ts.items():
                setattr(d, k, t.data_ptr())
            d.kind, d.cin, d.cout, d.res_out = self.KINDS[L["kind"]], int(L["cin"]), int(L["cout"]), int(L["res_out"])
            assert ts["noise"].numel() == d.res_out ** 2 and ts["style_weight"].shape == (2 * d.cout, self.dlatent)
            self.shapes.append((d.res_out, d.cout))
        rw, rb = f32(rgb_weight).reshape(3, -1), f32(rgb_bias).reshape(3)
        nbytes = lib.gsb_sg1_packed_bytes(self.desc, self.n_layers, self.dlatent)
        if nbytes == 0:
            raise NativeError(f"gsb_sg1_packed_bytes: {lib.gsb_last_error().decode()}")
        self.packed = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _check(lib.gsb_sg1_pack(self.desc, self.n_layers, self.dlatent, _ptr(rw), _ptr(rb), _ptr(self.packed),
                                    self.packed.numel(), _stream()), "gsb_sg1_pack")
            torch.cuda.current_stream().synchronize()      # the temporaries above may be freed after this returns

    def out_dims(self, n_run: int, stop: str) -> int:
        r, co = self.shapes[n_run - 1]
        return {"epi": r * r * co, "conv": r * r * co, "style": 2 * co, "image": 3 * r * r}[stop]

    def forward(self, w_layers: torch.Tensor, n_run: int, stop: str = "epi", out: torch.Tensor = None) -> torch.Tensor:
        """Result ``stop`` of layer ``n_run - 1`` for per-layer latents w_layers [Lw, n, dlatent] (layer j reads entry
        min(j, Lw - 1); Lw = 1: one latent for all layers): fp32 rows [n, out_dims] (NHWC for 'epi' / 'conv', NCHW for
        'image'); ``out`` may be a row-strided 2-D view (e.g. the batch rows of the large-d IPCA buffer)."""
        lib = load()
        assert w_layers.is_cuda and w_layers.dtype == torch.float32 and w_layers.dim() == 3 and w_layers.shape[2] == self.dlatent
        w_layers = w_layers.contiguous()
        n, d, code = w_layers.shape[1], self.out_dims(n_run, stop), self.STOPS[stop]
        if out is None:
            out = torch.empty((n, d), dtype=torch.float32, device=w_layers.device)
        assert out.is_cuda and out.dtype == torch.float32 and out.shape == (n, d) and out.stride(1) == 1
        ws_bytes = lib.gsb_sg1_workspace_bytes(self.desc, self.n_layers, n_run, code, n)
        ws = scratch.get("synthesis_sg1", ws_bytes, w_layers.device)
        with torch.cuda.device(w_layers.device), instrument.section("synthesis_sg1"):
            _check(lib.gsb_sg1_forward(_ptr(self.packed), self.desc, self.n_layers, self.dlatent, n_run, code, _ptr(w_layers),
                                       w_layers.shape[0], n, C.c_void_p(out.data_ptr()), out.stride(0), _ptr(ws), ws.numel(),
                                       _stream()), "gsb_sg1_forward")
        # per layer: 1 style launch; per chunk of samples: GEMM + gather (not on the constant layer), epilogue, stats, norm
        launches = 1 if stop == "style" else n_run + (1 if stop == "image" else 0)
        if stop != "style":
            for i in range(n_run):
                L = self.desc[i]
                hw_in = (L.res_out // (2 if L.kind >= 2 else 1)) ** 2
                chunks = -(-n // max(1, 4096 // hw_in))
                launches += chunks * ((2 if L.kind else 0) + (1 if (stop == "conv" and i == n_run - 1) else 3))
        instrument.count(launches)
        instrument.add_rows("synthesis_sg1", n)
        return out

    def check(self):
        """Raise if an operand left fp16's range since the pack (synchronises)."""
        flags = C.c_uint(0)
        with torch.cuda.device(self.device):
            _check(load().gsb_sg1_status(_ptr(self.packed), self.desc, self.n_layers, self.dlatent, C.byref(flags)),
                   "gsb_sg1_status")
        if flags.value & 1:
            raise NativeError("StyleGAN synthesis: an activation exceeded fp16 range in the tap-GEMM operands; results are invalid")


class PackedSynthesis:
    """StyleGAN2 synthesis layers conv1, convs.0 .. convs.k packed for the tap-GEMM kernels (gsb_synthesis_pack).

    ``layers``: dicts with conv_weight [co,ci,3,3], mod_weight [ci,S], mod_bias [ci], act_bias [co], noise [r,r],
    noise_weight [1] (fp32 CUDA tensors) and upsample (bool), res_in (int), in execution order."""

    def __init__(self, const_input: torch.Tensor, layers, style_dim: int):
        lib = load()
        self.device = require_cuda(const_input.device)
        self.style_dim = int(style_dim)
        self.n_layers = len(layers)
        self._keep = []
        self.desc = (StyledConvDesc * self.n_layers)()
        self.shapes = []                        # (res_out, cout) per layer
        f32 = lambda t: t.detach().to(self.device, torch.float32).contiguous()
        for i, L in enumerate(layers):
            ts = {k: f32(L[k]) for k in ("conv_weight", "mod_weight", "mod_bias", "act_bias", "noise", "noise_weight")}
            self._keep.append(ts)
            co, ci = ts["conv_weight"].shape[0], ts["conv_weight"].shape[1]
            assert ts["conv_weight"].shape == (co, ci, 3, 3) and ts["mod_weight"].shape == (ci, self.style_dim)
            res_in, up = int(L["res_in"]), bool(L["upsample"])
            res_out = 2 * res_in if up else res_in
            assert ts["noise"].numel() == res_out * res_out and ts["noise_weight"].numel() == 1
            d = self.desc[i]
            for k, t in ts.items():
                setattr(d, k, t.data_ptr())
            d.cin, d.cout, d.upsample, d.res_in = ci, co, int(up), res_in
            self.shapes.append((res_out, co))
        cst = f32(const_input).reshape(-1, 4, 4)
        nbytes = lib.gsb_synthesis_packed_bytes(self.desc, self.n_layers, self.style_dim)
        if nbytes == 0:
            raise NativeError(f"gsb_synthesis_packed_bytes: {lib.gsb_last_error().decode()}")
        self.packed = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _check(lib.gsb_synthesis_pack(self.desc, self.n_layers, self.style_dim, _ptr(cst), _ptr(self.packed),
                                          self.packed.numel(), _stream()), "gsb_synthesis_pack")
            torch.cuda.current_stream().synchronize()      # the temporaries above may be freed after this returns

    def out_dims(self, n_run: int) -> int:
        r, co = self.shapes[n_run - 1]
        return r * r * co

    def forward(self, w: torch.Tensor, n_run: int, out: torch.Tensor = None) -> torch.Tensor:
        """Activation of layer ``n_run - 1`` for w[n, style_dim]: fp32 NHWC rows [n, res*res*cout] (``out`` may be a
        row-strided 2-D view, e.g. the batch rows of the large-d IPCA buffer)."""
        lib = load()
        assert w.is_cuda and w.dtype == torch.float32 and w.dim() == 2 and w.shape[1] == self.style_dim
        w = w.contiguous()
        n, d = w.shape[0], self.out_dims(n_run)
        if out is None:
            out = torch.empty((n, d), dtype=torch.float32, device=w.device)
        assert out.is_cuda and out.dtype == torch.float32 and out.shape == (n, d) and out.stride(1) == 1
        ws_bytes = lib.gsb_synthesis_workspace_bytes(self.desc, n_run, n)
        ws = scratch.get("synthesis", ws_bytes, w.device)
        with torch.cuda.device(w.device), instrument.section("synthesis"):
            _check(lib.gsb_synthesis_forward(_ptr(self.packed), self.desc, self.n_layers, n_run, self.style_dim, _ptr(w), n,
                                             C.c_void_p(out.data_ptr()), out.stride(0), _ptr(ws), ws.numel(), _stream()),
                   "gsb_synthesis_forward")
        # per layer: 4 style/demod launches; per chunk of samples: 1 GEMM + 1 (stride-1) or 2 (upsample) epilogue launches
        launches = 1
        for i in range(n_run):
            res_in = self.desc[i].res_in
            chunks = -(-n // max(1, 4096 // (res_in * res_in)))
            launches += 4 + chunks * (3 if self.desc[i].upsample else 2)
        instrument.count(launches)
        instrument.add_rows("synthesis", n)
        return out

    def render(self, w_layers: torch.Tensor, n_run: int, rgbs, want_act: bool = False):
        """Generator.forward on the fused chain (gsb_synthesis_render): ``w_layers`` [Lw, n, style_dim] per-layer latents (Lw = 1:
        one global latent), ``rgbs``: list of dicts (conv_weight [3,cin], mod_weight, mod_bias, bias [3]) for to_rgb1,
        to_rgbs.0, ... up to the one that follows layer n_run-1 or earlier.  Returns (activation of layer n_run-1 as fp32 NHWC
        rows or None, skip image after the last ToRGB as fp32 NHWC [n, res, res, 3] or None)."""
        lib = load()
        assert w_layers.is_cuda and w_layers.dtype == torch.float32 and w_layers.dim() == 3 and w_layers.shape[2] == self.style_dim
        w_layers = w_layers.contiguous()
        Lw, n = int(w_layers.shape[0]), int(w_layers.shape[1])
        keep = []
        descs = (ToRGBDesc * max(1, len(rgbs)))()
        for j, r in enumerate(rgbs):
            ts = {k: r[k].detach().to(self.device, torch.float32).contiguous() for k in ("conv_weight", "mod_weight", "mod_bias", "bias")}
            keep.append(ts)
            cin = ts["conv_weight"].shape[-1]
            assert ts["conv_weight"].numel() == 3 * cin and ts["bias"].numel() == 3
            for k, t in ts.items():
                setattr(descs[j], k, t.data_ptr())
            descs[j].cin = int(cin)
        act = rgb = None
        if want_act:
            act = torch.empty((n, self.out_dims(n_run)), dtype=torch.float32, device=self.device)
        if rgbs:
            res = self.shapes[2 * (len(rgbs) - 1)][0]
            rgb = torch.empty((n, res, res, 3), dtype=torch.float32, device=self.device)
        ws_bytes = lib.gsb_synthesis_render_workspace_bytes(self.desc, n_run, n, self.style_dim)
        ws = scratch.get("synthesis", ws_bytes, self.device)
        with torch.cuda.device(self.device), instrument.section("synthesis"):
            _check(lib.gsb_synthesis_render(_ptr(self.packed), self.desc, self.n_layers, n_run, self.style_dim, descs, len(rgbs),
                                            _ptr(w_layers), Lw, n, _ptr(act), act.stride(0) if act is not None else 0, _ptr(rgb),
                                            _ptr(ws), ws.numel(), _stream()), "gsb_synthesis_render")
            if keep:
                torch.cuda.current_stream().synchronize()      # the temporary parameter copies may be freed after this
        instrument.count(1)
        instrument.add_rows("synthesis", n)
        return act, rgb

    def check(self):
        flags = C.c_uint(0)
        with torch.cuda.device(self.device):
            _check(load().gsb_synthesis_status(_ptr(self.packed), self.desc, self.n_layers, self.style_dim, C.byref(flags)),
                   "gsb_synthesis_status")
        if flags.value & 1:
            raise NativeError("synthesis: an operand exceeded fp16 range in the tensor-core path; results are invalid")


def pick_global_signs(rowmax_all: torch.Tensor) -> torch.Tensor:
    """svd_flip across feature shards: rowmax_all [W, c, 2] = per shard (max |.|, its signed value); the sign of the
    global maximum wins, ties go to the lowest shard (= lowest feature index, np.argmax's first-occurrence rule)."""
    idx = torch.argmax(rowmax_all[:, :, 0], dim=0)                      # first maximal shard per row
    val = rowmax_all[idx, torch.arange(rowmax_all.shape[1], device=rowmax_all.device), 1]
    return torch.where(val < 0, -torch.ones_like(val), torch.ones_like(val)).contiguous()


def exchange_rows(stage: torch.Tensor, out: torch.Tensor, world: int, group=None):
    """Row-parallel -> feature-sharded exchange of one IPCA batch (SURVEY.md section 8e).  ``stage`` [q, d]: the q rows
    this rank produced, all d features; ``out`` [world*q, d/world]: every rank's rows for THIS rank's feature block,
    in rank (= sample) order.  One all-to-all; the send side is packed by a strided copy."""
    import torch.distributed as dist
    q, d = stage.shape
    dl = d // world
    assert d % world == 0 and out.shape == (world * q, dl) and out.is_contiguous()
    send = stage.view(q, world, dl).permute(1, 0, 2).contiguous()       # [world, q, dl]: block s goes to rank s
    dist.all_to_all_single(out.view(world, q, dl), send, group=group)
    return out


class BigIPCA:
    """Large-d IncrementalPCA engine (csrc/bigd.cu): the stacked matrix M = [S*Vt; batch; correction] lives in HBM,
    producers write the batch rows in place (``batch_rows``), ``step`` runs one partial_fit.

    ``shard=(rank, world)``: feature-sharded over a torch.distributed job -- this object holds the column block
    d/world of M; ``step`` all-reduces the small-side Gram (fp64, (c+nb+1)^2) and agrees on the svd_flip signs."""

    def __init__(self, d: int, c: int, nb_max: int, device, shard=None, gram: str = None):
        lib = load()
        self.dev = require_cuda(device)
        # small-side Gram kernel: "tc" = tcgen05 with a promoted accumulator (gram_tc.cu; default -- measured error vs fp64
        # 1.6e-6 against 2.4e-6 for the fp32 FMA kernel, and 2.1x faster per step), "simt" = fp32 FMA kernel (bigd.cu);
        # widths that are not a multiple of 64 fall back to the FMA kernel inside the library
        gram = gram or os.environ.get("GANSPACE_B200_BIGD_GRAM", "tc")
        if gram not in ("simt", "tc"):
            raise NativeError(f"unknown Gram kernel '{gram}' (simt | tc)")
        self.flags = 1 if gram == "tc" else 0
        self.shard = shard if (shard is not None and shard[1] > 1) else None
        self.d_full = int(d)
        if self.shard is not None:
            if d % (16 * self.shard[1]) != 0:
                raise NativeError(f"feature sharding needs d % (16*world) == 0 (d={d}, world={self.shard[1]})")
            d = d // self.shard[1]
        self.d, self.c, self.nb_max = int(d), int(c), int(nb_max)
        ws_bytes = lib.gsb_bigd_workspace_bytes(self.d, self.c, self.nb_max, self.flags)
        if ws_bytes == 0:
            raise NativeError(f"gsb_bigd_workspace_bytes: {lib.gsb_last_error().decode()}")
        self.rows = lib.gsb_bigd_rows(self.c, self.nb_max)
        self.M = torch.empty((self.rows, self.d), dtype=torch.float32, device=self.dev)
        self.state = torch.empty(lib.gsb_bigd_state_bytes(self.d, self.c), dtype=torch.uint8, device=self.dev)
        self.ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.dev)
        self.batch_mean = torch.zeros(self.d, dtype=torch.float64, device=self.dev)
        self.n_seen = 0
        self.last_nb = 0
        with torch.cuda.device(self.dev):
            _check(lib.gsb_bigd_reset(_ptr(self.state), _ptr(self.M), self.d, self.c, self.nb_max, _stream()), "gsb_bigd_reset")
        t_ptr = lib.gsb_bigd_gram_matrix(_ptr(self.ws), self.d, self.c, self.nb_max)
        off = int(t_ptr) - self.ws.data_ptr()
        self._T = self.ws[off:off + self.rows * self.rows * 8].view(torch.float64)      # small-side Gram [rows, rows]
        self._rowmax = torch.empty((self.c, 2), dtype=torch.float32, device=self.dev)

    def batch_rows(self, nb: int) -> torch.Tensor:
        assert 1 <= nb <= self.nb_max
        return self.M[self.c:self.c + nb]

    def _args(self, nb):
        return (_ptr(self.state), _ptr(self.M), self.d, self.c, self.nb_max, self.n_seen, int(nb), self.flags)

    def gram_only(self, nb: int) -> torch.Tensor:
        """Test hook: phase 1 alone (centres the batch rows!); returns the small-side Gram [rows, rows] fp64."""
        with torch.cuda.device(self.dev):
            _check(load().gsb_bigd_step_gram(*self._args(nb), _ptr(self.batch_mean), _ptr(self.ws), self.ws.numel(), _stream()),
                   "gsb_bigd_step_gram")
        return self._T.view(self.rows, self.rows)

    def step(self, nb: int):
        lib = load()
        tail = (_ptr(self.ws), self.ws.numel(), _stream())
        with torch.cuda.device(self.dev), instrument.section("chain"):
            if self.shard is None:
                _check(lib.gsb_bigd_chain_step(*self._args(nb), _ptr(self.batch_mean), *tail), "gsb_bigd_chain_step")
            else:
                import torch.distributed as dist
                _check(lib.gsb_bigd_step_gram(*self._args(nb), _ptr(self.batch_mean), *tail), "gsb_bigd_step_gram")
                dist.all_reduce(self._T)                                   # small-side Gram summed over the feature shards
                _check(lib.gsb_bigd_step_solve(*self._args(nb), _ptr(self._rowmax), *tail), "gsb_bigd_step_solve")
                allmax = torch.empty((self.shard[1] * self.c, 2), dtype=torch.float32, device=self.dev)
                dist.all_gather_into_tensor(allmax, self._rowmax)          # concatenated along dim 0 in rank order
                signs = pick_global_signs(allmax.view(self.shard[1], self.c, 2))
                _check(lib.gsb_bigd_step_commit(*self._args(nb), _ptr(signs), *tail), "gsb_bigd_step_commit")
        lanczos = (os.environ.get("GANSPACE_B200_BIGD_CHAIN") == "lanczos" and self.n_seen > 0 and self.c % 16 == 0
                   and self.c <= 128 and 3 * self.c <= self.rows // 2 + self.rows // 8)
        instrument.count(7 + (37 if lanczos else 5) + (2 if self.flags & 1 else 0))
        self.n_seen += int(nb)
        self.last_nb = int(nb)

    def export(self):
        """sklearn's attributes; under feature sharding every rank returns the full-width arrays (one all-gather)."""
        lib = load()
        f64 = dict(dtype=torch.float64, device=self.dev)
        out = {
            "components": torch.empty((self.c, self.d), dtype=torch.float32, device=self.dev),
            "singular_values": torch.empty(self.c, **f64), "mean": torch.empty(self.d, **f64),
            "var": torch.empty(self.d, **f64), "explained_variance": torch.empty(self.c, **f64),
            "explained_variance_ratio": torch.empty(self.c, **f64),
        }
        with torch.cuda.device(self.dev):
            _check(lib.gsb_bigd_export(_ptr(self.state), _ptr(self.M), self.d, self.c, self.n_seen, _ptr(out["components"]),
                                       _ptr(out["singular_values"]), _ptr(out["mean"]), _ptr(out["var"]),
                                       _ptr(out["explained_variance"]), _ptr(out["explained_variance_ratio"]), _stream()),
                   "gsb_bigd_export")
        instrument.count(3)
        if self.shard is not None:
            import torch.distributed as dist
            W = self.shard[1]
            comp = torch.empty((W * self.c, self.d), dtype=torch.float32, device=self.dev)
            dist.all_gather_into_tensor(comp, out["components"])
            out["components"] = comp.view(W, self.c, self.d).permute(1, 0, 2).reshape(self.c, W * self.d).contiguous()
            for k in ("mean", "var"):
                full = torch.empty(W * self.d, **f64)
                dist.all_gather_into_tensor(full, out[k])
                out[k] = full
            # explained_variance_ratio_ = S^2 / sum(var * n) over ALL features (_incremental_pca.py:366-367)
            out["explained_variance_ratio"] = out["singular_values"] ** 2 / (out["var"].sum() * self.n_seen)
        return out

    def gathered(self, local: torch.Tensor) -> torch.Tensor:
        """[n, d_local] column blocks of every rank -> [n, d_full] (identity without sharding)."""
        if self.shard is None:
            return local
        import torch.distributed as dist
        W = self.shard[1]
        local = local.contiguous()
        n, dl = local.shape
        full = torch.empty((W * n, dl), dtype=local.dtype, device=local.device)
        dist.all_gather_into_tensor(full, local)
        return full.view(W, n, dl).permute(1, 0, 2).reshape(n, W * dl).contiguous()
