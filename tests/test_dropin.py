"""The drop-in host layer (iq_tool_b200/host/): the reference's stage/module prototypes backed by
libiqgpu.so.  Driven by oracle/ref_harness.c — the SAME driver that walks chunks through the
reference's own stage code — linked against the drop-in objects instead
(iq_tool_b200/host/_build/libiqdropin_harness.so, built by `make -C iq_tool_b200/host harness`).

CPU tests: the library loads, exports the reference's prototypes, designs/validates exactly like
the reference does, and fails loudly without a GPU.  GPU tests: chunk-by-chunk and threaded runs
through the three stage calls reproduce the direct C-ABI result bit for bit and the reference
within the north_star tolerances, in FUSED and EAGER mode."""
import ctypes as C
import os

import numpy as np
import pytest

from helpers import max_lsb, rel_rms_fullscale, snr_db
from iq_tool_b200.synth import synth_numpy
from oracle.loader import CpuChain, dropin_path, have_ref

REFERENCE_PROTOTYPES = [
    # include/pre_processor.h, resampler.h, post_processor.h
    "pre_processor_apply_chain", "pre_processor_reset", "create_resampler", "destroy_resampler",
    "resampler_reset", "resampler_execute", "post_processor_apply_chain", "post_processor_reset",
    # filter.h, frequency_shift.h
    "filter_create", "filter_reset", "filter_destroy", "filter_apply",
    "freq_shift_create", "freq_shift_apply", "freq_shift_reset_nco", "freq_shift_destroy_ncos",
    # sample_convert.h, dc_block.h
    "get_bytes_per_sample", "convert_block_to_cf32", "convert_cf32_to_block",
    "dc_block_create", "dc_block_reset", "dc_block_apply", "dc_block_destroy",
    # iq_correct.h, agc.h
    "iq_correct_init", "iq_correct_apply", "iq_correct_run_optimization", "iq_correct_destroy",
    "iq_correct_run_initial_calibration", "agc_create", "agc_apply", "agc_reset", "agc_destroy",
]


def _have_dropin():
    try:
        from oracle.loader import get_lib
        get_lib("dropin")
        return True
    except (FileNotFoundError, OSError):
        return False


needs_dropin = pytest.mark.skipif(not _have_dropin(), reason="drop-in harness not built (needs the reference headers)")


@needs_dropin
def test_dropin_exports_the_reference_prototypes():
    lib = C.CDLL(dropin_path())
    for name in REFERENCE_PROTOTYPES:
        assert hasattr(lib, name), name


@needs_dropin
@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
def test_dropin_create_resolves_the_filter_like_the_reference(name, workloads):
    """filter_create side effects the host pipeline reads (pipeline.c:232-265): implementation
    type, block size, pre/post placement — no GPU needed (host design only)."""
    cfg = workloads[name].config
    d = CpuChain(cfg, "dropin").info()
    r = CpuChain(cfg, "ref" if have_ref() else "oracle").info()
    assert (d.filter_impl, d.filter_post_resample, d.filter_block_size) == \
           (r.filter_impl, r.filter_post_resample, r.filter_block_size)
    assert d.ratio == r.ratio and d.cap_samples == r.cap_samples


@needs_dropin
def test_dropin_rejects_what_the_reference_rejects(workloads):
    import dataclasses
    from iq_tool_b200.configs import lowpass
    cfg = dataclasses.replace(workloads["cfg2"].config, filters=[lowpass(500e3)])   # beyond the output Nyquist
    with pytest.raises(RuntimeError):
        CpuChain(cfg, "dropin")
    cfg = dataclasses.replace(workloads["cfg1"].config, freq_shift_hz=0.0, shift_after_resample=True)
    with pytest.raises(RuntimeError):
        CpuChain(cfg, "dropin")


@needs_dropin
def test_dropin_fails_loudly_without_a_gpu(workloads):
    from iq_tool_b200 import gpu
    if gpu.device_count() > 0:
        pytest.skip("a GPU is present")
    wl = workloads["cfg1"]
    ch = CpuChain(wl.config, "dropin")
    with pytest.raises(RuntimeError):          # handle_fatal_thread_error path -> process returns -1
        ch.process(synth_numpy(wl, 16384))


# ---------------------------------------------------------------------------------------------
def _tolerance_check(cfg, out, ref):
    assert out.size == ref.size
    if cfg.output_format == "cf32":
        a, b = out.view(np.complex64), ref.view(np.complex64)
        assert rel_rms_fullscale(a, b) <= 1e-5 and snr_db(a, b) >= 100.0
    else:
        assert max_lsb(out, ref) <= 1


@pytest.mark.gpu
@needs_dropin
@pytest.mark.parametrize("name,n", [("cfg1", 40 * 16384 + 777), ("cfg3", 60 * 16384 + 5), ("cfg5", 50 * 16384 + 1)])
def test_dropin_fused_equals_direct_chain_and_reference(name, n, gpu, workloads):
    wl = workloads[name]
    raw = synth_numpy(wl, n)
    direct, counts = gpu.Chain(wl.config, 0).process(raw, return_chunk_counts=True)
    ref = CpuChain(wl.config, "ref" if have_ref() else "oracle").process(raw)
    d = CpuChain(wl.config, "dropin")
    d.trace(n // 16384 + 4)
    out = d.process(raw)                                   # pre -> resample -> post per chunk: 1-chunk trains
    assert np.array_equal(d.traced(), counts)              # per-chunk frames_to_write
    assert np.array_equal(out, direct)                     # same engine, any batching: same bits
    _tolerance_check(wl.config, out, ref)
    d2 = CpuChain(wl.config, "dropin")
    out_t = d2.process(raw, threaded=True)                 # three stage threads, trains of up to 8 chunks
    assert np.array_equal(out_t, direct)
    # stream discontinuity (pre/resampler/post resets as the marker flows through): stream restarts
    d2.reset()
    head = raw[: 2 * 5 * 16384]
    after = d2.process(head)
    if wl.config.filters and wl.config.filter_taps == 4095:
        # FFT filter: the frames that were waiting for a full block survive filter_reset (filter.c:417-436, F5) and lead
        # the new stream — the reference does exactly that, so the reference after the same reset is the yardstick
        r2 = CpuChain(wl.config, "ref" if have_ref() else "oracle")
        r2.process(raw)
        r2.reset()
        _tolerance_check(wl.config, after, r2.process(head))
    else:
        assert np.array_equal(after, gpu.Chain(wl.config, 0).process(head))


@pytest.mark.gpu
@needs_dropin
@pytest.mark.parametrize("name,n", [("cfg1", 6 * 16384 + 777), ("cfg3", 14 * 16384 + 5), ("cfg4", 4 * 16384)])
def test_dropin_eager_module_api_matches_reference(name, n, gpu, workloads, monkeypatch):
    """EAGER mode: every module function (convert, dc_block_apply, iq_correct_apply, freq_shift_apply,
    resampler_execute, filter_apply, agc_apply, convert) does its own work on host buffers."""
    wl = workloads[name]                                   # as specified: cfg4 keeps its DC offset and I/Q imbalance
    raw = synth_numpy(wl, n)                               # (the module-level dc_block_apply reproduces liquid's fp32 rounding)
    monkeypatch.setenv("IQGPU_DROPIN_EAGER", "1")
    d = CpuChain(wl.config, "dropin")
    d.capture(0, n + 16)
    d.capture(1, n + 16)
    out = d.process(raw)
    r = CpuChain(wl.config, "ref" if have_ref() else "oracle")
    r.capture(0, n + 16)
    r.capture(1, n + 16)
    ref = r.process(raw)
    assert rel_rms_fullscale(d.captured(0), r.captured(0)) <= 1e-5     # pre-processor output (buffer A on the host)
    assert rel_rms_fullscale(d.captured(1), r.captured(1)) <= 1e-5     # resampler output
    from helpers import parity_metrics, record_parity
    record_parity(f"dropin_eager/{name}", parity_metrics(wl.config, out, ref))
    _tolerance_check(wl.config, out, ref)


@pytest.mark.gpu
@needs_dropin
def test_dropin_iq_optimizer_runs_on_the_gpu(gpu, workloads, monkeypatch):
    monkeypatch.setenv("IQGPU_IQ_LIBC_RAND", "1")           # the reference's rand() directions; default: seeded generator (B7)
    wl = workloads["cfg4"]
    x = synth_numpy(wl, 4096)
    blk = ((x.astype(np.float32) - 127.5) / 128.0).view(np.complex64)[:1024]
    d = CpuChain(wl.config, "dropin")
    r = CpuChain(wl.config, "ref" if have_ref() else "oracle")
    dm, dp, da, dr = d.iq_optimize(blk, 7)
    rm, rp, ra, rr = r.iq_optimize(blk, 7)
    assert abs(da - ra) <= 1e-3 and abs(dr - rr) <= 1e-3
    assert abs(dm - rm) <= 1.1e-5 and abs(dp - rp) <= 1.1e-5


@pytest.mark.gpu
@needs_dropin
def test_dropin_iq_optimizer_is_repeatable_by_default(gpu, workloads):
    """SURVEY App. B7: the drop-in's optimiser is paced by the sample clock and steps in directions from a seeded
    generator, so the same capture gives the same factors (the reference's depend on time() and on the wall clock)."""
    wl = workloads["cfg4"]
    x = synth_numpy(wl, 4096)
    blk = ((x.astype(np.float32) - 127.5) / 128.0).view(np.complex64)[:1024]
    a = CpuChain(wl.config, "dropin").iq_optimize(blk, 1)
    b = CpuChain(wl.config, "dropin").iq_optimize(blk, 99)      # the libc seed plays no part
    assert a == b and (a[0], a[1]) != (np.float32(wl.config.iq_mag), np.float32(wl.config.iq_phase))
