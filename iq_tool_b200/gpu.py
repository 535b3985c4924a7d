"""ctypes binding of libiqgpu.so (include/iqgpu.h) — the host-side entry to the CUDA chain.

There is no CPU fallback: importing this module fails loudly when the shared library has not
been built (run `python -c "import __graft_entry__ as g; g.build()"` or `make -C
iq_tool_b200/csrc`), and every compute call raises IqGpuError when CUDA is unavailable.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

from .configs import NUMPY_DTYPE, ChainConfig, ChainConfigC

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libiqgpu.so")


class IqGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"iqgpu error {code}: {msg}")
        self.code = code


class ChainInfoC(C.Structure):
    _fields_ = [
        ("ratio", C.c_float), ("is_interp", C.c_int32), ("num_halfband", C.c_uint32),
        ("halfband_m", C.c_uint32 * 16), ("rate_arbitrary", C.c_float), ("arb_step", C.c_uint32),
        ("filter_impl", C.c_int32), ("filter_post_resample", C.c_int32),
        ("filter_block_size", C.c_uint32), ("filter_num_taps", C.c_uint32),
        ("nco_dtheta", C.c_uint32), ("nco_is_post", C.c_int32), ("agc_locked", C.c_uint32),
        ("agc_gain", C.c_float), ("agc_peak_memory", C.c_float), ("agc_samples_seen", C.c_uint64),
        ("frames_in_total", C.c_uint64), ("frames_out_total", C.c_uint64),
        ("fused_front", C.c_uint32), ("kernel_launches", C.c_uint32), ("halo_frames", C.c_uint32),
        ("reserved", C.c_uint32),
    ]


class AgcStateC(C.Structure):
    """iqgpu_agc_state (include/iqgpu.h)."""
    _fields_ = [("locked", C.c_uint32), ("gain", C.c_float), ("peak_memory", C.c_float),
                ("samples_seen", C.c_uint64), ("last_strong_s", C.c_double)]

    def as_tuple(self):
        return (int(self.locked), float(self.gain), float(self.peak_memory), int(self.samples_seen),
                float(self.last_strong_s))


class RawfileStatsC(C.Structure):
    """iqgpu_rawfile_stats (include/iqgpu.h)."""
    _fields_ = [("frames_in", C.c_uint64), ("frames_out", C.c_uint64), ("bytes_written", C.c_uint64),
                ("trains", C.c_uint64)]


class WavInfoC(C.Structure):
    """iqgpu_wav_info (include/iqgpu.h): SF_INFO + SdrMetadata of src/input_wav.c."""
    _fields_ = [("container", C.c_int32), ("sample_format", C.c_int32), ("format_tag", C.c_int32),
                ("channels", C.c_int32), ("bits_per_sample", C.c_int32), ("sample_rate_hz", C.c_int32),
                ("data_offset", C.c_uint64), ("data_bytes", C.c_uint64), ("frames", C.c_uint64),
                ("metadata_present", C.c_int32), ("source_software", C.c_int32),
                ("center_freq_hz_present", C.c_int32), ("timestamp_unix_present", C.c_int32),
                ("center_freq_hz", C.c_double), ("timestamp_unix", C.c_int64),
                ("timestamp_str_present", C.c_int32), ("software_name_present", C.c_int32),
                ("software_version_present", C.c_int32), ("radio_model_present", C.c_int32),
                ("timestamp_str", C.c_char * 64), ("software_name", C.c_char * 64),
                ("software_version", C.c_char * 64), ("radio_model", C.c_char * 128)]

    def as_dict(self) -> dict:
        """The metadata fields that are present, plus the header fields."""
        d = {k: int(getattr(self, k)) for k in ("container", "sample_format", "format_tag", "channels",
                                                "bits_per_sample", "sample_rate_hz", "data_offset", "data_bytes",
                                                "frames", "metadata_present", "source_software")}
        if self.center_freq_hz_present:
            d["center_freq_hz"] = float(self.center_freq_hz)
        if self.timestamp_unix_present:
            d["timestamp_unix"] = int(self.timestamp_unix)
        for k in ("timestamp_str", "software_name", "software_version", "radio_model"):
            if getattr(self, k + "_present"):
                d[k] = bytes(getattr(self, k)).decode("utf-8", "replace")
        return d


CONTAINER_RAW, CONTAINER_WAV, CONTAINER_RF64 = 0, 1, 2


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
            "iq_tool_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, sz, u32p = C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32)
    lib.iqgpu_abi_version.restype = C.c_int
    lib.iqgpu_last_error.restype = C.c_char_p
    lib.iqgpu_device_count.restype = C.c_int
    lib.iqgpu_host_alloc.restype = vp
    lib.iqgpu_host_alloc.argtypes = [sz]
    lib.iqgpu_host_free.argtypes = [vp]
    lib.iqgpu_chain_create.restype = C.c_int
    lib.iqgpu_chain_create.argtypes = [C.POINTER(ChainConfigC), C.c_int, C.POINTER(vp)]
    lib.iqgpu_chain_destroy.argtypes = [vp]
    lib.iqgpu_chain_reset.argtypes = [vp]
    lib.iqgpu_chain_restart.argtypes = [vp]
    lib.iqgpu_chain_get_info.argtypes = [vp, C.POINTER(ChainInfoC)]
    lib.iqgpu_chain_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
    lib.iqgpu_chain_set_iq_factors.argtypes = [vp, C.c_float, C.c_float]
    lib.iqgpu_chain_get_iq_state.restype = C.c_int
    lib.iqgpu_chain_get_iq_state.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.iqgpu_iq_direction.restype = C.c_float
    lib.iqgpu_iq_direction.argtypes = [C.c_uint32, C.c_uint64, C.c_uint32]
    lib.iqgpu_chain_get_kernel_times.restype = C.c_int
    lib.iqgpu_chain_get_kernel_times.argtypes = [vp, C.POINTER(C.c_double), u32p, C.c_int]
    lib.iqgpu_chain_process.argtypes = [vp, vp, sz, u32p, sz, vp, sz, C.POINTER(sz), u32p]
    lib.iqgpu_chain_process_device.argtypes = [vp, vp, sz, u32p, sz, vp, sz, C.POINTER(sz), u32p, vp]
    lib.iqgpu_chain_predict_output.argtypes = [vp, sz, C.POINTER(sz)]
    lib.iqgpu_chain_read_tap.argtypes = [vp, C.c_int, vp, sz, C.POINTER(sz)]
    lib.iqgpu_chain_get_filter_taps.argtypes = [vp, vp, C.c_uint32, u32p]
    lib.iqgpu_chain_get_halfband_taps.argtypes = [vp, C.c_uint32, vp, C.c_uint32, u32p]
    lib.iqgpu_chain_get_arb_taps.argtypes = [vp, vp, C.c_uint32, u32p]
    lib.iqgpu_chain_seek.argtypes = [vp, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.iqgpu_chain_halo_frames.argtypes = [vp, C.POINTER(sz)]
    lib.iqgpu_chain_resampler_outputs_after.argtypes = [vp, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.iqgpu_chain_process_device_begin.argtypes = [vp, vp, sz, u32p, sz, vp]
    lib.iqgpu_chain_pending_chunk_peaks.argtypes = [vp, vp, vp, sz, C.POINTER(sz)]
    lib.iqgpu_chain_process_device_finish.argtypes = [vp, sz, vp, sz, C.POINTER(sz), u32p, vp]
    lib.iqgpu_chain_pending_chunk_peaks_device.argtypes = [vp, sz, vp, sz, C.POINTER(sz), vp]
    lib.iqgpu_chain_agc_advance_device.argtypes = [vp, vp, C.c_uint64, C.c_uint64, vp]
    lib.iqgpu_chain_outputs_after.argtypes = [vp, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.iqgpu_chain_agc_rms_state_device.argtypes = [vp, vp, vp]
    lib.iqgpu_chain_agc_rms_resume_device.argtypes = [vp, sz, vp, vp, sz, vp, vp]
    lib.iqgpu_chain_get_agc_rms_state.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.iqgpu_chain_get_agc_state.argtypes = [vp, C.POINTER(AgcStateC)]
    lib.iqgpu_chain_set_agc_state.argtypes = [vp, C.POINTER(AgcStateC)]
    lib.iqgpu_agc_digital_initial_state.argtypes = [C.POINTER(AgcStateC)]
    lib.iqgpu_agc_digital_initial_state.restype = None
    lib.iqgpu_agc_digital_advance.argtypes = [C.POINTER(AgcStateC), C.c_float, C.c_double, vp, vp, sz, vp]
    lib.iqgpu_rawfile_run.restype = C.c_int
    lib.iqgpu_rawfile_run.argtypes = [C.POINTER(ChainConfigC), C.c_int, C.c_char_p, C.c_char_p, sz, C.POINTER(RawfileStatsC)]
    lib.iqgpu_rawfile_last_error.restype = C.c_char_p
    lib.iqgpu_wav_probe.argtypes = [C.c_char_p, C.POINTER(WavInfoC)]
    lib.iqgpu_wav_parse_auxi.argtypes = [C.c_char_p, sz, C.POINTER(WavInfoC)]
    lib.iqgpu_wav_parse_filename.argtypes = [C.c_char_p, C.POINTER(WavInfoC)]
    lib.iqgpu_wav_center_target_shift.argtypes = [C.POINTER(WavInfoC), C.c_float, C.c_double, C.POINTER(C.c_double)]
    lib.iqgpu_wav_header_bytes.restype = sz
    lib.iqgpu_wav_header_bytes.argtypes = [C.c_int]
    lib.iqgpu_wav_build_header.argtypes = [C.c_int, C.c_int, C.c_int, C.c_uint64, vp, sz]
    lib.iqgpu_wavfile_run.argtypes = [C.POINTER(ChainConfigC), C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_int,
                                      C.c_float, sz, C.POINTER(RawfileStatsC), C.POINTER(WavInfoC)]
    for name in ("iqgpu_wav_probe", "iqgpu_wav_parse_auxi", "iqgpu_wav_parse_filename",
                 "iqgpu_wav_center_target_shift", "iqgpu_wav_build_header", "iqgpu_wavfile_run"):
        getattr(lib, name).restype = C.c_int
    lib.iqgpu_ubench_fp32_peak.restype = C.c_int
    lib.iqgpu_ubench_fp32_peak.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.iqgpu_get_bytes_per_sample.restype = sz
    lib.iqgpu_get_bytes_per_sample.argtypes = [C.c_int]
    lib.iqgpu_convert_block_to_cf32.argtypes = [vp, vp, sz, C.c_int, C.c_float]
    lib.iqgpu_convert_cf32_to_block.argtypes = [vp, vp, sz, C.c_int]
    lib.iqgpu_iq_optimize.argtypes = [vp, vp, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                      C.POINTER(C.c_float), C.POINTER(C.c_float)]
    for name in ("iqgpu_chain_reset", "iqgpu_chain_restart", "iqgpu_chain_get_info", "iqgpu_chain_set_option",
                 "iqgpu_chain_set_iq_factors", "iqgpu_chain_process", "iqgpu_chain_process_device",
                 "iqgpu_chain_predict_output", "iqgpu_chain_read_tap", "iqgpu_chain_get_filter_taps",
                 "iqgpu_chain_get_halfband_taps", "iqgpu_chain_get_arb_taps", "iqgpu_chain_seek",
                 "iqgpu_chain_halo_frames", "iqgpu_chain_resampler_outputs_after",
                 "iqgpu_chain_process_device_begin", "iqgpu_chain_pending_chunk_peaks",
                 "iqgpu_chain_process_device_finish", "iqgpu_chain_get_agc_state", "iqgpu_chain_set_agc_state",
                 "iqgpu_chain_pending_chunk_peaks_device", "iqgpu_chain_agc_advance_device",
                 "iqgpu_agc_digital_advance", "iqgpu_convert_block_to_cf32", "iqgpu_chain_outputs_after",
                 "iqgpu_chain_agc_rms_state_device", "iqgpu_chain_agc_rms_resume_device", "iqgpu_chain_get_agc_rms_state",
                 "iqgpu_convert_cf32_to_block", "iqgpu_iq_optimize"):
        getattr(lib, name).restype = C.c_int
    return lib


lib = _load()


def _check(rc: int) -> None:
    if rc != 0:
        raise IqGpuError(rc, lib.iqgpu_last_error().decode("utf-8", "replace"))


def device_count() -> int:
    return lib.iqgpu_device_count()


def fp32_peak_tflops(device: int = 0) -> float:
    """Measured FP32 FMA peak (packed FFMA2 micro-benchmark inside the library), TFLOP/s."""
    t = C.c_double(0.0)
    _check(lib.iqgpu_ubench_fp32_peak(device, C.byref(t), None))
    return t.value


class Chain:
    """One configured chain (pre-processor + resampler + post-processor) on one GPU.

    device=-1 builds a plan-only chain: design and closed-form bookkeeping work, compute fails.
    """

    def __init__(self, cfg: ChainConfig, device: int = 0, **options):
        self.cfg = cfg
        self._c = cfg.to_c()
        self._h = C.c_void_p()
        _check(lib.iqgpu_chain_create(C.byref(self._c), device, C.byref(self._h)))
        for k, v in options.items():
            self.set_option(k, v)

    def close(self) -> None:
        if getattr(self, "_h", None):
            lib.iqgpu_chain_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, key: str, value: int) -> None:
        _check(lib.iqgpu_chain_set_option(self._h, key.encode(), int(value)))

    def set_iq_factors(self, mag: float, phase: float) -> None:
        _check(lib.iqgpu_chain_set_iq_factors(self._h, mag, phase))

    def iq_state(self):
        """(mag, phase, successful passes, probed blocks) of the in-chain I/Q optimiser."""
        m, p = C.c_float(0), C.c_float(0)
        a, b = C.c_uint64(0), C.c_uint64(0)
        _check(lib.iqgpu_chain_get_iq_state(self._h, C.byref(m), C.byref(p), C.byref(a), C.byref(b)))
        return m.value, p.value, a.value, b.value

    def reset(self) -> None:
        """Stream discontinuity with the reference's semantics (an FFT filter's waiting frames survive, filter.c:417-436)."""
        _check(lib.iqgpu_chain_reset(self._h))

    def restart(self) -> None:
        """Back to the state right after create."""
        _check(lib.iqgpu_chain_restart(self._h))

    def info(self) -> ChainInfoC:
        o = ChainInfoC()
        _check(lib.iqgpu_chain_get_info(self._h, C.byref(o)))
        return o

    KERNEL_CLASSES = ("pre", "dc_scan", "resampler", "filter", "post", "fused_front", "_6", "_7")

    def kernel_times(self, reset: bool = True) -> dict:
        """Accumulated device ms / launch groups per kernel class (needs time_kernels=1)."""
        ms = (C.c_double * 8)()
        cnt = (C.c_uint32 * 8)()
        _check(lib.iqgpu_chain_get_kernel_times(self._h, ms, cnt, int(reset)))
        return {k: (ms[i], cnt[i]) for i, k in enumerate(self.KERNEL_CLASSES) if cnt[i]}

    def predict_output(self, n_frames: int) -> int:
        o = C.c_size_t(0)
        _check(lib.iqgpu_chain_predict_output(self._h, n_frames, C.byref(o)))
        return o.value

    def halo_frames(self) -> int:
        o = C.c_size_t(0)
        _check(lib.iqgpu_chain_halo_frames(self._h, C.byref(o)))
        return o.value

    def seek(self, first_frame: int) -> int:
        o = C.c_uint64(0)
        _check(lib.iqgpu_chain_seek(self._h, first_frame, C.byref(o)))
        return o.value

    def resampler_outputs_after(self, frames_in: int) -> int:
        """Closed form: resampler output frames after `frames_in` input frames since reset."""
        o = C.c_uint64(0)
        _check(lib.iqgpu_chain_resampler_outputs_after(self._h, frames_in, C.byref(o)))
        return o.value

    def outputs_after(self, frames_in: int) -> int:
        """Closed form: chain output frames after `frames_in` input frames since a restart (the resampler's count,
        block-quantised by an FFT filter): the output index of a capture frame."""
        o = C.c_uint64(0)
        _check(lib.iqgpu_chain_outputs_after(self._h, frames_in, C.byref(o)))
        return o.value

    # ---- sharded RMS AGC: end-state hand-over between time shards (include/iqgpu.h) ----
    def agc_rms_state_device(self, dev_state_ptr: int, stream: int = 0) -> None:
        """Copy the RMS AGC's state {g, y2'} (two float32) to device memory, asynchronously on `stream`."""
        _check(lib.iqgpu_chain_agc_rms_state_device(self._h, dev_state_ptr, C.c_void_p(stream) if stream else None))

    def agc_rms_resume_device(self, first_output: int, dev_state_ptr: int, dev_out_ptr: int, out_capacity_bytes: int,
                              dev_changed_ptr: int = 0, stream: int = 0) -> None:
        """Re-run the RMS AGC of the last process_device call from output frame `first_output` with the state at
        `dev_state_ptr` and re-convert the outputs that changed into `dev_out_ptr` (that call's output buffer).
        `dev_changed_ptr` (optional, int32 in device memory) receives whether the end state changed."""
        _check(lib.iqgpu_chain_agc_rms_resume_device(self._h, first_output, dev_state_ptr, dev_out_ptr, out_capacity_bytes,
                                                     dev_changed_ptr or None, C.c_void_p(stream) if stream else None))

    def get_agc_rms_state(self):
        """(g, y2') of the RMS AGC, read to the host."""
        g, y2 = C.c_float(0), C.c_float(0)
        _check(lib.iqgpu_chain_get_agc_rms_state(self._h, C.byref(g), C.byref(y2)))
        return g.value, y2.value

    # ---- sharded digital AGC: process_device split at the peak exchange (include/iqgpu.h) ----
    def process_device_begin(self, dev_in_ptr: int, n_frames: int, stream: int = 0) -> None:
        _check(lib.iqgpu_chain_process_device_begin(self._h, dev_in_ptr, n_frames, None, 0,
                                                    C.c_void_p(stream) if stream else None))

    def pending_chunk_peaks(self):
        """(peaks float32[n_chunks], counts uint32[n_chunks]) of the begun call."""
        n = C.c_size_t(0)
        _check(lib.iqgpu_chain_pending_chunk_peaks(self._h, None, None, 0, C.byref(n)))
        peaks = np.zeros(max(1, n.value), dtype=np.float32)
        counts = np.zeros(max(1, n.value), dtype=np.uint32)
        _check(lib.iqgpu_chain_pending_chunk_peaks(self._h, peaks.ctypes.data, counts.ctypes.data, n.value, C.byref(n)))
        return peaks[: n.value], counts[: n.value]

    def pending_chunk_peaks_device(self, skip_chunks: int, dev_peaks_ptr: int, capacity: int, stream: int = 0) -> int:
        """Copy the begun call's per-chunk peaks [skip_chunks, n_chunks) into device memory (asynchronously); returns
        the number of peaks."""
        n = C.c_size_t(0)
        _check(lib.iqgpu_chain_pending_chunk_peaks_device(self._h, skip_chunks, dev_peaks_ptr, capacity, C.byref(n),
                                                          C.c_void_p(stream) if stream else None))
        return n.value

    def agc_advance_device(self, dev_peaks_ptr: int, first_frame: int, n_frames: int, stream: int = 0) -> None:
        """Advance the device-resident digital-AGC state over the chunks of capture frames
        [first_frame, first_frame + n_frames) whose peaks are in device memory."""
        _check(lib.iqgpu_chain_agc_advance_device(self._h, dev_peaks_ptr, first_frame, n_frames,
                                                  C.c_void_p(stream) if stream else None))

    def process_device_finish(self, skip_chunks: int, dev_out_ptr: int, out_capacity_bytes: int, stream: int = 0) -> int:
        nout = C.c_size_t(0)
        _check(lib.iqgpu_chain_process_device_finish(self._h, skip_chunks, dev_out_ptr, out_capacity_bytes,
                                                     C.byref(nout), None, C.c_void_p(stream) if stream else None))
        return nout.value

    def get_agc_state(self) -> AgcStateC:
        s = AgcStateC()
        _check(lib.iqgpu_chain_get_agc_state(self._h, C.byref(s)))
        return s

    def set_agc_state(self, s: AgcStateC) -> None:
        _check(lib.iqgpu_chain_set_agc_state(self._h, C.byref(s)))

    # ---- design introspection ----
    def filter_taps(self) -> np.ndarray:
        n = C.c_uint32(0)
        _check(lib.iqgpu_chain_get_filter_taps(self._h, None, 0, C.byref(n)))
        out = np.zeros(n.value, dtype=np.complex64)
        if n.value:
            _check(lib.iqgpu_chain_get_filter_taps(self._h, out.ctypes.data, n.value, C.byref(n)))
        return out

    def halfband_taps(self, i: int) -> np.ndarray:
        n = C.c_uint32(0)
        _check(lib.iqgpu_chain_get_halfband_taps(self._h, i, None, 0, C.byref(n)))
        out = np.zeros(n.value, dtype=np.float32)
        _check(lib.iqgpu_chain_get_halfband_taps(self._h, i, out.ctypes.data, n.value, C.byref(n)))
        return out

    def arb_taps(self) -> np.ndarray:
        n = C.c_uint32(0)
        _check(lib.iqgpu_chain_get_arb_taps(self._h, None, 0, C.byref(n)))
        out = np.zeros(n.value, dtype=np.float32)
        if n.value:
            _check(lib.iqgpu_chain_get_arb_taps(self._h, out.ctypes.data, n.value, C.byref(n)))
        return out

    # ---- compute ----
    def _chunks(self, chunk_frames: Optional[Sequence[int]]):
        if chunk_frames is None:
            return None, 0, None
        arr = np.ascontiguousarray(chunk_frames, dtype=np.uint32)
        return arr.ctypes.data_as(C.POINTER(C.c_uint32)), arr.size, arr

    def out_capacity_frames(self, n_frames: int) -> int:
        return int(n_frames * max(1.0, self.cfg.ratio)) + 4 * 16384 + 4096

    def process(self, raw: np.ndarray, chunk_frames: Optional[Sequence[int]] = None,
                return_chunk_counts: bool = False):
        """Host-buffer path (H2D/D2H inside).  raw: interleaved input samples."""
        raw = np.ascontiguousarray(raw)
        n_frames = raw.nbytes // self.cfg.in_bytes
        out = np.zeros(self.out_capacity_frames(n_frames) * self.cfg.out_bytes, dtype=np.uint8)
        nout = C.c_size_t(0)
        cptr, ncz, keep = self._chunks(chunk_frames)
        nchunks = ncz if chunk_frames is not None else (n_frames + 16383) // 16384
        counts = np.zeros(max(1, nchunks), dtype=np.uint32)
        _check(lib.iqgpu_chain_process(self._h, raw.ctypes.data, n_frames, cptr, ncz, out.ctypes.data,
                                       out.nbytes, C.byref(nout),
                                       counts.ctypes.data_as(C.POINTER(C.c_uint32))))
        res = out[: nout.value * self.cfg.out_bytes].view(NUMPY_DTYPE[self.cfg.output_format])
        return (res, counts[:nchunks]) if return_chunk_counts else res

    def process_device(self, dev_in_ptr: int, n_frames: int, dev_out_ptr: int, out_capacity_bytes: int,
                       stream: int = 0, chunk_frames: Optional[Sequence[int]] = None) -> int:
        """Device-resident path; pointers are raw device addresses (e.g. torch data_ptr())."""
        nout = C.c_size_t(0)
        cptr, ncz, keep = self._chunks(chunk_frames)
        _check(lib.iqgpu_chain_process_device(self._h, dev_in_ptr, n_frames, cptr, ncz, dev_out_ptr,
                                              out_capacity_bytes, C.byref(nout), None,
                                              C.c_void_p(stream) if stream else None))
        return nout.value

    def read_tap(self, tap: int) -> np.ndarray:
        n = C.c_size_t(0)
        _check(lib.iqgpu_chain_read_tap(self._h, tap, None, 0, C.byref(n)))
        out = np.zeros(n.value, dtype=np.complex64)
        if n.value:
            _check(lib.iqgpu_chain_read_tap(self._h, tap, out.ctypes.data, n.value, C.byref(n)))
        return out


def convert_block_to_cf32(raw: np.ndarray, fmt_code: int, n_frames: int, gain: float) -> np.ndarray:
    raw = np.ascontiguousarray(raw)
    out = np.zeros(n_frames, dtype=np.complex64)
    _check(lib.iqgpu_convert_block_to_cf32(raw.ctypes.data, out.ctypes.data, n_frames, fmt_code, gain))
    return out


def convert_cf32_to_block(x: np.ndarray, fmt_code: int, out_dtype, bytes_per_sample: int) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.complex64)
    out = np.zeros(x.shape[0] * bytes_per_sample, dtype=np.uint8)
    _check(lib.iqgpu_convert_cf32_to_block(x.ctypes.data, out.ctypes.data, x.shape[0], fmt_code))
    return out.view(out_dtype)


def iq_optimize(block1024: np.ndarray, directions50: np.ndarray, mag: float, phase: float):
    """K6: one I/Q optimiser pass on the GPU.  Returns (mag, phase, avg_power, power_range)."""
    blk = np.ascontiguousarray(block1024, dtype=np.complex64)
    d = np.ascontiguousarray(directions50, dtype=np.float32)
    if blk.size != 1024 or d.size != 50:
        raise ValueError("iq_optimize needs 1024 frames and 50 directions")
    m, p, a, r = C.c_float(mag), C.c_float(phase), C.c_float(0), C.c_float(0)
    _check(lib.iqgpu_iq_optimize(blk.ctypes.data, d.ctypes.data, C.byref(m), C.byref(p), C.byref(a), C.byref(r)))
    return m.value, p.value, a.value, r.value


def agc_initial_state() -> AgcStateC:
    s = AgcStateC()
    lib.iqgpu_agc_digital_initial_state(C.byref(s))
    return s


def agc_digital_advance(state: AgcStateC, target: float, target_rate_hz: float, peaks: np.ndarray,
                        counts: np.ndarray, want_gains: bool = False):
    """Host-only digital-AGC state machine over per-chunk peaks (updates `state` in place)."""
    pk = np.ascontiguousarray(peaks, dtype=np.float32)
    ct = np.ascontiguousarray(counts, dtype=np.uint32)
    assert pk.size == ct.size
    g = np.zeros(max(1, pk.size), dtype=np.float32) if want_gains else None
    _check(lib.iqgpu_agc_digital_advance(C.byref(state), target, target_rate_hz, pk.ctypes.data if pk.size else None,
                                         ct.ctypes.data if ct.size else None, pk.size,
                                         g.ctypes.data if want_gains else None))
    return g[: pk.size] if want_gains else None


def rawfile_run(cfg: ChainConfig, in_path: str, out_path: str, device: int = 0, train_chunks: int = 0) -> RawfileStatsC:
    """Stream a raw I/Q file through the chain into a raw output file (reader / chain / writer overlapped)."""
    st = RawfileStatsC()
    c = cfg.to_c()
    rc = lib.iqgpu_rawfile_run(C.byref(c), device, os.fsencode(in_path), os.fsencode(out_path), train_chunks, C.byref(st))
    if rc != 0:
        raise IqGpuError(rc, lib.iqgpu_rawfile_last_error().decode("utf-8", "replace"))
    return st


def _io_check(rc: int) -> None:
    if rc != 0:
        raise IqGpuError(rc, lib.iqgpu_rawfile_last_error().decode("utf-8", "replace"))


def wav_probe(path: str) -> WavInfoC:
    """wav_initialize's view of a WAV / RF64 capture: header, auxi chunk, file-name metadata (host only)."""
    info = WavInfoC()
    _io_check(lib.iqgpu_wav_probe(os.fsencode(path), C.byref(info)))
    return info


def wav_parse_auxi(chunk: bytes, info: WavInfoC | None = None) -> tuple[bool, WavInfoC]:
    info = info if info is not None else WavInfoC()
    return bool(lib.iqgpu_wav_parse_auxi(chunk, len(chunk), C.byref(info))), info


def wav_parse_filename(base: str, info: WavInfoC | None = None) -> tuple[bool, WavInfoC]:
    info = info if info is not None else WavInfoC()
    return bool(lib.iqgpu_wav_parse_filename(os.fsencode(base), C.byref(info))), info


def wav_center_target_shift(info: WavInfoC, center_target_hz: float, freq_shift_hz_arg: float = 0.0) -> float:
    out = C.c_double()
    _io_check(lib.iqgpu_wav_center_target_shift(C.byref(info), center_target_hz, freq_shift_hz_arg, C.byref(out)))
    return out.value


def wav_build_header(container: int, output_format: int, sample_rate_hz: int, data_bytes: int) -> bytes:
    n = lib.iqgpu_wav_header_bytes(container)
    buf = C.create_string_buffer(max(n, 1))
    _io_check(lib.iqgpu_wav_build_header(container, output_format, sample_rate_hz, data_bytes, buf, n))
    return buf.raw[:n]


def wavfile_run(cfg: ChainConfig, in_path: str, out_path: str, in_container: int = CONTAINER_WAV,
                out_container: int = CONTAINER_WAV, center_target_hz: float = 0.0, device: int = 0,
                train_chunks: int = 0) -> tuple[RawfileStatsC, WavInfoC]:
    """A whole file run with WAV / RF64 containers on either side (format and rate of a WAV input come from its header)."""
    st, info = RawfileStatsC(), WavInfoC()
    c = cfg.to_c()
    rc = lib.iqgpu_wavfile_run(C.byref(c), device, os.fsencode(in_path), in_container, os.fsencode(out_path),
                               out_container, center_target_hz, train_chunks, C.byref(st), C.byref(info))
    _io_check(rc)
    return st, info
