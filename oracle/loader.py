"""ctypes bindings for the CPU checkers — TEST INFRASTRUCTURE ONLY.

  RefChain     oracle/_ref/libiqref.so      the reference's own stage sources (compiled in place
                                            from /root/reference/src) on the liquid_compat shim
  OracleChain  oracle/libiqoracle.so        the restated oracle (oracle/iq_oracle.c)

Both expose the same flat API (create / process / reset / captures / info), so the parity tests
can swap one for the other.  Nothing in iq_tool_b200/ may import this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_ROOT = "/root/reference"


class RefInfo(C.Structure):
    _fields_ = [("ratio", C.c_float), ("filter_impl", C.c_int32), ("filter_post_resample", C.c_int32),
                ("filter_block_size", C.c_uint32), ("filter_num_taps", C.c_uint32),
                ("nco_dtheta", C.c_uint32), ("nco_is_post", C.c_int32), ("cap_samples", C.c_uint32),
                ("agc_locked", C.c_uint32), ("agc_gain", C.c_float), ("agc_peak_memory", C.c_float),
                ("agc_samples_seen", C.c_uint64)]


class MsresampInfo(C.Structure):
    _fields_ = [("is_interp", C.c_int), ("num_halfband", C.c_uint), ("m_stage", C.c_uint * 16),
                ("as_stage", C.c_float * 16), ("rate_arbitrary", C.c_float), ("step", C.c_uint32),
                ("npfb", C.c_uint), ("arb_m", C.c_uint), ("arb_fc", C.c_float)]


def build(target: str = "all", quiet: bool = True) -> None:
    """(Re)build the checkers. `ref` is a no-op when /root/reference is absent."""
    subprocess.run(["make", "-C", HERE, target], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


def _load(path: str, prefix: str):
    lib = C.CDLL(path)
    vp, i64, u32p = C.c_void_p, C.c_int64, C.POINTER(C.c_uint32)
    f = lambda n: getattr(lib, prefix + n)  # noqa: E731
    f("create").restype = vp
    f("create").argtypes = [vp]
    f("destroy").argtypes = [vp]
    f("reset").argtypes = [vp]
    f("process").restype = C.c_int
    f("process").argtypes = [vp, vp, i64, vp, i64, C.POINTER(i64)]
    f("set_capture").argtypes = [vp, C.c_int, vp, i64]
    f("get_capture_len").restype = i64
    f("get_capture_len").argtypes = [vp, C.c_int]
    f("set_trace").argtypes = [vp, u32p, i64]
    f("get_trace_len").restype = i64
    f("get_trace_len").argtypes = [vp]
    f("get_info").argtypes = [vp, C.POINTER(RefInfo)]
    f("get_filter_taps").restype = C.c_uint32
    f("get_filter_taps").argtypes = [vp, vp, C.c_uint32]
    f("get_msresamp").restype = vp
    f("get_msresamp").argtypes = [vp]
    f("get_bytes_per_sample").restype = C.c_size_t
    f("get_bytes_per_sample").argtypes = [C.c_int]
    f("convert_block_to_cf32").restype = C.c_int
    f("convert_block_to_cf32").argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_float]
    f("convert_cf32_to_block").restype = C.c_int
    f("convert_cf32_to_block").argtypes = [vp, vp, C.c_size_t, C.c_int]
    f("set_fake_clock").argtypes = [C.c_int, C.c_double]
    f("iq_optimize").restype = C.c_int
    f("iq_optimize").argtypes = [vp, vp, C.c_uint, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                 C.POINTER(C.c_float), C.POINTER(C.c_float)]
    if hasattr(lib, prefix + "process_threaded"):
        f("process_threaded").restype = C.c_int
        f("process_threaded").argtypes = [vp, vp, i64, vp, i64, C.POINTER(i64)]
    if not hasattr(lib, "liquid_compat_msresamp_get_info"):
        return lib   # the GPU drop-in harness carries no liquid layer
    lib.liquid_compat_msresamp_get_info.argtypes = [vp, C.POINTER(MsresampInfo)]
    lib.liquid_compat_msresamp_get_halfband.restype = C.c_uint
    lib.liquid_compat_msresamp_get_halfband.argtypes = [vp, C.c_uint, vp, C.c_uint]
    lib.liquid_compat_msresamp_get_arb_taps.restype = C.c_uint
    lib.liquid_compat_msresamp_get_arb_taps.argtypes = [vp, vp, C.c_uint]
    lib.liquid_compat_nco_constrain.restype = C.c_uint32
    lib.liquid_compat_nco_constrain.argtypes = [C.c_float]
    return lib


_LIBS = {}


def ref_path(fast: bool = False) -> str:
    return os.path.join(HERE, "_ref", "libiqref_fast.so" if fast else "libiqref.so")


def oracle_path() -> str:
    return os.path.join(HERE, "libiqoracle.so")


def have_ref(fast: bool = False) -> bool:
    return os.path.exists(ref_path(fast))


def dropin_path() -> str:
    return os.path.join(os.path.dirname(HERE), "iq_tool_b200", "host", "_build", "libiqdropin_harness.so")


def get_lib(kind: str):
    """kind: 'ref' | 'ref_fast' | 'oracle' | 'dropin' (ref_harness.c driving the GPU drop-in host layer)"""
    if kind not in _LIBS:
        if kind == "dropin":
            if os.path.isdir(REF_ROOT):
                subprocess.run(["make", "-C", os.path.join(os.path.dirname(HERE), "iq_tool_b200", "host"), "harness"],
                               check=True, stdout=subprocess.DEVNULL)
            if not os.path.exists(dropin_path()):
                raise FileNotFoundError(dropin_path())
            _LIBS[kind] = (_load(dropin_path(), "iqref_"), "iqref_")
        elif kind == "oracle":
            build("oracle")  # incremental; plain C, builds anywhere gcc exists
            _LIBS[kind] = (_load(oracle_path(), "iqo_"), "iqo_")
        else:
            fast = kind == "ref_fast"
            if os.path.isdir(REF_ROOT):
                build("ref")  # incremental; only possible where the reference sources exist
            if not have_ref(fast):
                raise FileNotFoundError(ref_path(fast))
            _LIBS[kind] = (_load(ref_path(fast), "iqref_"), "iqref_")
    return _LIBS[kind]


class CpuChain:
    """One chain instance on a CPU checker library."""

    def __init__(self, cfg, kind: str = "oracle"):
        self.lib, self.pfx = get_lib(kind)
        self.kind = kind
        self.cfg = cfg
        self._c = cfg.to_c()
        self.h = self._f("create")(C.byref(self._c))
        if not self.h:
            raise RuntimeError(f"{kind}: chain create failed")
        self._caps = {}
        self._trace = None

    def _f(self, name):
        return getattr(self.lib, self.pfx + name)

    def close(self):
        if self.h:
            self._f("destroy")(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        self._f("reset")(self.h)

    def iq_optimize(self, block1024: np.ndarray, seed: int):
        """One optimiser pass (iq_correct.c:154-235) with rand() seeded by `seed`.
        Returns (mag, phase, avg_power, power_range)."""
        blk = np.ascontiguousarray(block1024, dtype=np.complex64)
        assert blk.size == 1024
        m, p, a, r = C.c_float(0), C.c_float(0), C.c_float(0), C.c_float(0)
        rc = self._f("iq_optimize")(self.h, blk.ctypes.data, seed, C.byref(m), C.byref(p), C.byref(a), C.byref(r))
        if rc != 0:
            raise RuntimeError("iq_optimize failed")
        return m.value, p.value, a.value, r.value

    def info(self) -> RefInfo:
        o = RefInfo()
        self._f("get_info")(self.h, C.byref(o))
        return o

    def filter_taps(self) -> np.ndarray:
        n = self._f("get_filter_taps")(self.h, None, 0)
        out = np.zeros(n, dtype=np.complex64)
        if n:
            self._f("get_filter_taps")(self.h, out.ctypes.data, n)
        return out

    def msresamp_info(self) -> Optional[MsresampInfo]:
        q = self._f("get_msresamp")(self.h)
        if not q:
            return None
        o = MsresampInfo()
        self.lib.liquid_compat_msresamp_get_info(q, C.byref(o))
        return o

    def halfband_taps(self, i: int) -> np.ndarray:
        q = self._f("get_msresamp")(self.h)
        n = self.lib.liquid_compat_msresamp_get_halfband(q, i, None, 0)
        out = np.zeros(n, dtype=np.float32)
        self.lib.liquid_compat_msresamp_get_halfband(q, i, out.ctypes.data, n)
        return out

    def arb_taps(self) -> np.ndarray:
        q = self._f("get_msresamp")(self.h)
        n = self.lib.liquid_compat_msresamp_get_arb_taps(q, None, 0)
        out = np.zeros(n, dtype=np.float32)
        self.lib.liquid_compat_msresamp_get_arb_taps(q, out.ctypes.data, n)
        return out

    def capture(self, stage: int, capacity: int) -> np.ndarray:
        """stage 0: after pre-processor, 1: after resampler (cf32 streams)."""
        buf = np.zeros(capacity, dtype=np.complex64)
        self._caps[stage] = buf
        self._f("set_capture")(self.h, stage, buf.ctypes.data, capacity)
        return buf

    def captured(self, stage: int) -> np.ndarray:
        n = self._f("get_capture_len")(self.h, stage)
        return self._caps[stage][:n]

    def trace(self, capacity: int) -> None:
        self._trace = np.zeros(capacity, dtype=np.uint32)
        self._f("set_trace")(self.h, self._trace.ctypes.data_as(C.POINTER(C.c_uint32)), capacity)

    def traced(self) -> np.ndarray:
        return self._trace[: self._f("get_trace_len")(self.h)]

    def process(self, raw: np.ndarray, threaded: bool = False) -> np.ndarray:
        """raw: interleaved input samples (numpy, any dtype; byte length defines frame count)."""
        raw = np.ascontiguousarray(raw)
        n_frames = raw.nbytes // self.cfg.in_bytes
        ratio = max(1.0, self.cfg.ratio)
        cap_frames = int(n_frames * ratio) + 4 * 16384 + 1024
        out = np.zeros(cap_frames * self.cfg.out_bytes, dtype=np.uint8)
        nout = C.c_int64(0)
        fn = self._f("process_threaded") if threaded else self._f("process")
        rc = fn(self.h, raw.ctypes.data, n_frames, out.ctypes.data, out.nbytes, C.byref(nout))
        if rc != 0:
            raise RuntimeError(f"{self.kind}: process failed rc={rc}")
        from iq_tool_b200.configs import NUMPY_DTYPE
        return out[: nout.value * self.cfg.out_bytes].view(NUMPY_DTYPE[self.cfg.output_format])


def libc_rand_directions(seed: int, n: int = 50) -> np.ndarray:
    """The +-1 sequence `_get_random_direction` (iq_correct.c:391) yields after srand(seed)."""
    libc = C.CDLL(None)
    libc.srand(C.c_uint(seed))
    rand_max = 2147483647
    return np.array([1.0 if libc.rand() > rand_max // 2 else -1.0 for _ in range(n)], dtype=np.float32)


def convert_to_cf32(kind: str, raw: np.ndarray, fmt_code: int, n: int, gain: float) -> np.ndarray:
    lib, pfx = get_lib(kind)
    out = np.zeros(n, dtype=np.complex64)
    raw = np.ascontiguousarray(raw)
    rc = getattr(lib, pfx + "convert_block_to_cf32")(raw.ctypes.data, out.ctypes.data, n, fmt_code, gain)
    if rc != 0:
        raise RuntimeError("convert_block_to_cf32 failed")
    return out


def convert_from_cf32(kind: str, x: np.ndarray, fmt_code: int, out_dtype, bytes_per_sample: int) -> np.ndarray:
    lib, pfx = get_lib(kind)
    x = np.ascontiguousarray(x, dtype=np.complex64)
    out = np.zeros(x.shape[0] * bytes_per_sample, dtype=np.uint8)
    rc = getattr(lib, pfx + "convert_cf32_to_block")(x.ctypes.data, out.ctypes.data, x.shape[0], fmt_code)
    if rc != 0:
        raise RuntimeError("convert_cf32_to_block failed")
    return out.view(out_dtype)
