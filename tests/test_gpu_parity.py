"""GPU parity tests (run on the B200 box: pytest -m gpu).  Everything goes through the C ABI
(libiqgpu.so via iq_tool_b200.gpu); the checker is the CPU oracle / the golden fixtures.

Bars (BASELINE.json north_star):
  * output frame counts and per-chunk frames_to_write: exact
  * int -> cf32 conversion (+ I/Q apply + LUT-NCO mix): bit exact
  * cf32 streams: relative RMS error <= 1e-5 of full scale and SNR >= 100 dB
  * integer outputs: within +-1 LSB
DC-blocker configs carry one documented exception, see test_dc_block_*.
"""
import hashlib

import numpy as np
import pytest

from helpers import max_lsb, rel_rms_fullscale, snr_db
from iq_tool_b200.configs import (AGC_DIGITAL, AGC_LOCAL, BYTES_PER_SAMPLE, FILTER_REQ_FIR, FORMAT_CODES, NUMPY_DTYPE,
                                  ChainConfig, lowpass, stopband)
from iq_tool_b200.synth import synth_numpy
from oracle.loader import CpuChain, have_ref

pytestmark = pytest.mark.gpu

CF32_RMS_TOL = 1e-5     # of full scale (north_star)
CF32_SNR_DB = 100.0
INT_LSB_TOL = 1
# The documented exception (DESIGN.md, DC blocker): measured deviation of the exact-arithmetic DC blocker from the
# reference's fp32 state rounding on the as-specified inputs, plus margin.  Measured values: profiles/r02_parity.md.
CFG2_DC_EXCEPTION_MAX_LSB = 14      # measured 11 (2^24 frames, r2a session)
CFG2_DC_EXCEPTION_RMS_LSB = 2.5     # measured 2.02
CFG4_DC_EXCEPTION_REL_RMS = 3.5e-4  # measured 2.6e-4 (2^22 frames; the LOCAL AGC scales the stream to unit power)
CFG4_DC_EXCEPTION_SNR_DB = 69.0     # measured 71.7 dB


def _oracle_kind():
    return "ref" if have_ref() else "oracle"


def _run_pair(gpu, cfg, raw, taps=2, **opts):
    """taps=2 records all taps (forces the unfused stage-by-stage path); taps=1 records taps 1-2
    and lets the chain use the fused front kernel where it applies."""
    g = gpu.Chain(cfg, 0, record_taps=taps, **opts)
    o = CpuChain(cfg, _oracle_kind())
    n = raw.nbytes // cfg.in_bytes
    o.capture(0, n + 16)
    o.capture(1, n + 16)
    o.trace(n // 16384 + 4)
    ref = o.process(raw)
    out, counts = g.process(raw, return_chunk_counts=True)
    return g, o, out, ref, counts


def _check_final(cfg, out, ref):
    assert out.size == ref.size
    if cfg.output_format == "cf32":
        a, b = out.view(np.complex64), ref.view(np.complex64)
        assert rel_rms_fullscale(a, b) <= CF32_RMS_TOL
        assert snr_db(a, b) >= CF32_SNR_DB
    else:
        assert max_lsb(out, ref) <= INT_LSB_TOL


# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["cfg1", "cfg5"])
def test_golden_fixture_parity(name, gpu, workloads, golden):
    """CUDA chain vs the committed reference outputs (no DC block in these configs)."""
    meta, data = golden
    cfg = workloads[name].config
    g = gpu.Chain(cfg, 0, record_taps=2)
    out, counts = g.process(data[name]["raw"], return_chunk_counts=True)
    assert np.array_equal(counts, data[name]["counts"])
    assert np.array_equal(g.read_tap(0)[:8192].view(np.uint32), data[name]["pre_head"].view(np.uint32))
    rs = g.read_tap(1)
    assert rs.size == data[name]["rs"].size
    assert rel_rms_fullscale(rs, data[name]["rs"]) <= 1e-6 and snr_db(rs, data[name]["rs"]) >= 120.0
    _check_final(cfg, out, data[name]["out"])


@pytest.mark.parametrize("name,n", [("cfg1", (1 << 22) + 4097), ("cfg5", (1 << 23) + 11)])
def test_baseline_config_parity_no_dc(name, n, gpu, workloads):
    wl = workloads[name]
    raw = synth_numpy(wl, n)
    g, o, out, ref, counts = _run_pair(gpu, wl.config, raw)
    assert np.array_equal(counts, o.traced())
    assert np.array_equal(g.read_tap(0).view(np.uint32), o.captured(0).view(np.uint32))   # bit exact
    assert rel_rms_fullscale(g.read_tap(1), o.captured(1)) <= 1e-6
    assert snr_db(g.read_tap(1), o.captured(1)) >= 120.0
    _check_final(wl.config, out, ref)
    gi, oi = g.info(), o.info()
    assert gi.agc_locked == oi.agc_locked and gi.agc_samples_seen == oi.agc_samples_seen
    assert abs(gi.agc_gain - oi.agc_gain) <= 2e-6 * abs(oi.agc_gain)


def test_cfg2_chain_without_dc_offset_meets_the_bar(gpu, workloads):
    """cfg2's chain (DC block + S=4 resampler + 255-tap FIR + cs16) on an input WITHOUT a DC
    offset: the integrator state stays small and the +-1 LSB bar holds end to end."""
    import dataclasses
    wl = dataclasses.replace(workloads["cfg2"], dc=0.0)
    raw = synth_numpy(wl, (1 << 22) + 333)
    g, o, out, ref, counts = _run_pair(gpu, wl.config, raw)
    assert np.array_equal(counts, o.traced())
    assert rel_rms_fullscale(g.read_tap(0), o.captured(0)) <= CF32_RMS_TOL
    assert snr_db(g.read_tap(1), o.captured(1)) >= CF32_SNR_DB
    from helpers import parity_metrics, record_parity
    record_parity("cfg2/dc_offset_removed/dc_mode=0", parity_metrics(wl.config, out, ref))
    _check_final(wl.config, out, ref)


def _dc_reference_f64(x, fs):
    from scipy.signal import lfilter
    alpha = np.float32(2.0 * np.pi * 10.0 / int(fs))
    c = np.float64(-(np.float32(-1.0) + alpha))
    y = lfilter([1.0, -1.0], [1.0, -c], x.astype(np.complex128))
    v = lfilter([1.0], [1.0, -c], x.astype(np.complex128))
    return y, float(np.abs(v).max())


def test_dc_block_is_exact_arithmetic_and_reference_differs_only_by_its_state_rounding(gpu, workloads):
    """DOCUMENTED EXCEPTION.  liquid's DC blocker keeps the integrator state v ~ dc/alpha in fp32
    (direct form II) and forms y = v[n]-v[n-1]; with dc = 0.02 at 20 Msps v reaches ~6.4e3, so
    the reference output carries rounding noise of ~ulp(v) = 4.9e-4 (about -70 dB).  The GPU
    evaluates the same difference equation as y = x - (1-c) v[n-1] with the carry in double.
    Proven here: (1) GPU == float64 recurrence to 1e-6; (2) the oracle deviates from float64
    by ~ulp(v); (3) |GPU - oracle| is bounded by that same ulp(v)."""
    wl = workloads["cfg2"]
    cfg = ChainConfig(input_format="cs16", output_format="cf32", input_rate_hz=wl.config.input_rate_hz,
                      target_rate_hz=wl.config.input_rate_hz, no_resample=True, dc_block=True)
    n = (1 << 21) + 1234
    raw = synth_numpy(wl, n)
    g, o, out, ref, _ = _run_pair(gpu, cfg, raw)
    x = raw.astype(np.float64).view(np.complex128) / 32768.0
    y64, vmax = _dc_reference_f64(x, cfg.input_rate_hz)
    gpu_y, ref_y = out.view(np.complex64), ref.view(np.complex64)
    ulp_v = float(np.spacing(np.float32(vmax)))
    assert rel_rms_fullscale(gpu_y, y64) <= 1e-6           # (1)
    assert rel_rms_fullscale(ref_y, y64) >= 20 * rel_rms_fullscale(gpu_y, y64)   # (2) the oracle is the noisy one
    assert np.abs(gpu_y - ref_y).max() <= 3.0 * ulp_v      # (3)
    # chunk-size invariance of the blocked scan: one call vs ragged calls give the same bits
    g2 = gpu.Chain(cfg, 0)
    parts, pos = [], 0
    for m in (1, 127, 128, 129, 4096, 100000, n):
        m = min(m, n - pos)
        if m <= 0:
            break
        parts.append(g2.process(raw[2 * pos:2 * (pos + m)], chunk_frames=[m]))
        pos += m
    y2 = np.concatenate(parts).view(np.complex64)
    assert rel_rms_fullscale(y2, gpu_y) <= 2e-8


# ---------------------------------------------------------------------------------------------
# cfg2 / cfg4 AS SPECIFIED (BASELINE.json: dc = 0.02 / 0.03, cfg4 with its I/Q imbalance and pinned factors), at
# SURVEY 8(d)'s parity sizes, against the reference's own stage code.  Two evaluations of the DC blocker:
#   dc_mode 1  liquid's fp32 direct-form-II recurrence, literally (serial kernel): the whole chain must meet the
#              north_star bar as written — this pins every other stage of the two configs on their specified inputs;
#   dc_mode 0  the chunk-train default (exact arithmetic, fused front): what it differs by is the reference's own state
#              rounding noise; the deviation is MEASURED, recorded (gpurun_out/parity_r02.jsonl -> profiles/) and bounded
#              by that measurement plus a small margin — the one documented exception (DESIGN.md, DC blocker).
# ---------------------------------------------------------------------------------------------
def _as_specified(gpu, wl, n, **opts):
    raw = synth_numpy(wl, n)
    o = CpuChain(wl.config, _oracle_kind())
    o.trace(n // 16384 + 4)
    ref = o.process(raw)
    g = gpu.Chain(wl.config, 0, **opts)
    out, counts = g.process(raw, return_chunk_counts=True)
    assert np.array_equal(counts, o.traced())               # per-chunk frames_to_write: exact
    assert out.size == ref.size
    return g, out, ref


def test_cfg2_as_specified_with_reference_dc_rounding_meets_the_bar(gpu, workloads):
    from helpers import parity_metrics, record_parity
    wl = workloads["cfg2"]
    g, out, ref = _as_specified(gpu, wl, wl.parity_samples, dc_mode=1)
    m = parity_metrics(wl.config, out, ref)
    record_parity("cfg2/as_specified/dc_mode=1", m)
    assert g.info().fused_front == 0
    assert m["max_lsb"] <= INT_LSB_TOL, m


def test_cfg2_as_specified_default_path_measured_deviation(gpu, workloads):
    """The headline bench configuration on its specified input through the path the bench times (fused front, local DC
    state).  Measured on B200 (profiles/r02_parity.md): see the bound below."""
    from helpers import error_spectrum_db, parity_metrics, record_parity
    wl = workloads["cfg2"]
    g, out, ref = _as_specified(gpu, wl, wl.parity_samples)
    assert g.info().fused_front == 1
    m = parity_metrics(wl.config, out, ref)
    sp = error_spectrum_db(out, ref, wl.config)
    if sp is not None:
        m["err_spectrum_db_fs_per_bin"] = {"min": float(sp.min()), "median": float(np.median(sp)), "max": float(sp.max())}
    record_parity("cfg2/as_specified/dc_mode=0", m)
    # reference integrator noise: ulp(v) = 4.9e-4 at v ~ dc/alpha = 6.4e3, white over 20 MHz, cascade keeps 0.37 MHz of it
    assert m["max_lsb"] <= CFG2_DC_EXCEPTION_MAX_LSB and m["rms_lsb"] <= CFG2_DC_EXCEPTION_RMS_LSB, m


def test_cfg4_as_specified_with_reference_dc_rounding_meets_the_bar(gpu, workloads):
    from helpers import parity_metrics, record_parity
    wl = workloads["cfg4"]
    g, out, ref = _as_specified(gpu, wl, wl.parity_samples, dc_mode=1)
    m = parity_metrics(wl.config, out, ref)
    record_parity("cfg4/as_specified/dc_mode=1", m)
    assert m["rel_rms"] <= CF32_RMS_TOL and m["snr_db"] >= CF32_SNR_DB, m


def test_cfg4_as_specified_default_path_measured_deviation(gpu, workloads):
    from helpers import error_spectrum_db, parity_metrics, record_parity
    wl = workloads["cfg4"]
    g, out, ref = _as_specified(gpu, wl, wl.parity_samples)
    assert g.info().fused_front == 1
    m = parity_metrics(wl.config, out, ref)
    sp = error_spectrum_db(out, ref, wl.config)
    if sp is not None:
        m["err_spectrum_db_fs_per_bin"] = {"min": float(sp.min()), "median": float(np.median(sp)), "max": float(sp.max())}
    record_parity("cfg4/as_specified/dc_mode=0", m)
    assert m["rel_rms"] <= CFG4_DC_EXCEPTION_REL_RMS and m["snr_db"] >= CFG4_DC_EXCEPTION_SNR_DB, m


def test_dc_reference_mode_is_bit_exact_and_call_size_invariant(gpu, workloads):
    """dc_mode 1 at the blocker's output: the same bits as liquid's recurrence in the reference build, however the stream
    is cut into calls (fp32 state carried on the device)."""
    wl = workloads["cfg2"]
    cfg = ChainConfig(input_format="cs16", output_format="cf32", input_rate_hz=wl.config.input_rate_hz,
                      target_rate_hz=wl.config.input_rate_hz, no_resample=True, dc_block=True)
    n = (1 << 20) + 1234
    raw = synth_numpy(wl, n)
    ref = CpuChain(cfg, _oracle_kind()).process(raw)
    one = gpu.Chain(cfg, 0, dc_mode=1).process(raw)
    assert np.array_equal(one.view(np.uint32), ref.view(np.uint32))
    g2 = gpu.Chain(cfg, 0, dc_mode=1)
    parts, pos = [], 0
    for m in (1, 127, 2048, 2049, 100000, n):
        m = min(m, n - pos)
        if m <= 0:
            break
        parts.append(g2.process(raw[2 * pos:2 * (pos + m)], chunk_frames=[m]))
        pos += m
    assert np.array_equal(np.concatenate(parts).view(np.uint32), ref.view(np.uint32))
    g2.reset()
    assert np.array_equal(g2.process(raw[: 2 * 5000]).view(np.uint32), ref[: 2 * 5000].view(np.uint32))


def test_fir_filter_stage_parity(gpu):
    """K3 alone: 255 real taps and a complex band-pass, on cf32 in/out."""
    from iq_tool_b200.configs import pass_range
    rng = np.random.Generator(np.random.PCG64(21))
    n = 3 * 16384 + 77
    x = ((rng.standard_normal(n) + 1j * rng.standard_normal(n)) * 0.2).astype(np.complex64)
    for filt, taps in (([lowpass(100e3)], 255), ([pass_range(102e3, 215e3)], 301), ([stopband(-5e3, 5e3)], 0)):
        cfg = ChainConfig(input_format="cf32", output_format="cf32", input_rate_hz=1e6, target_rate_hz=1e6,
                          no_resample=True, filters=filt, filter_taps=taps, filter_type_request=FILTER_REQ_FIR)
        g, o, out, ref, _ = _run_pair(gpu, cfg, x.view(np.float32))
        _check_final(cfg, out, ref)


def test_rms_agc_parity(gpu):
    """G1 (liquid agc_crcf, LOCAL profile) on a level-stepped tone."""
    n = 6 * 16384
    t = np.arange(n)
    x = (0.2 * np.exp(2j * np.pi * 0.01 * t)).astype(np.complex64)
    x[n // 2:] *= 3.0
    cfg = ChainConfig(input_format="cf32", output_format="cf32", input_rate_hz=1e6, target_rate_hz=1e6,
                      no_resample=True, agc_enable=True, agc_profile=AGC_LOCAL)
    g, o, out, ref, _ = _run_pair(gpu, cfg, x.view(np.float32))
    _check_final(cfg, out, ref)


def test_cfg4_full_chain_without_dc_offset(gpu, workloads):
    """cfg4 (cu8 -> shift, DC block, I/Q apply, S=1 resampler, 1461-tap notch, LOCAL AGC, cf32) on an
    input without DC offset: full north_star bar.  (With dc = 0.03 the DC-blocker exception applies.)"""
    import dataclasses
    wl = dataclasses.replace(workloads["cfg4"], dc=0.0)
    raw = synth_numpy(wl, (1 << 20) + 99)
    g, o, out, ref, counts = _run_pair(gpu, wl.config, raw)
    assert np.array_equal(counts, o.traced())
    assert rel_rms_fullscale(g.read_tap(1), o.captured(1)) <= CF32_RMS_TOL
    from helpers import parity_metrics, record_parity
    m = parity_metrics(wl.config, out, ref)
    record_parity("cfg4/dc_offset_removed/dc_mode=0", m)
    assert m["rel_rms"] <= CF32_RMS_TOL and m["snr_db"] >= CF32_SNR_DB, m


def test_chunk_train_invariance(gpu, workloads):
    """One train == chunk-by-chunk calls == ragged sub-trains, bit for bit (per-chunk semantics
    are closed form, so the GPU result must not depend on how the host batches chunks)."""
    wl = workloads["cfg1"]
    n = 20 * 16384 + 5000
    raw = synth_numpy(wl, n)
    a = gpu.Chain(wl.config, 0).process(raw)
    b_chain = gpu.Chain(wl.config, 0)
    parts = [b_chain.process(raw[2 * s:2 * min(s + 16384, n)]) for s in range(0, n, 16384)]
    assert np.array_equal(a, np.concatenate(parts))
    c_chain = gpu.Chain(wl.config, 0, subtrain_frames=3 * 16384)
    assert np.array_equal(a, c_chain.process(raw))


def test_reset_restarts_the_stream(gpu, workloads):
    wl = workloads["cfg5"]
    raw = synth_numpy(wl, 8 * 16384)
    g = gpu.Chain(wl.config, 0)
    a = g.process(raw)
    g.process(raw[: 2 * 5000])
    g.reset()
    assert np.array_equal(a, g.process(raw))


def test_conversion_kats_on_gpu_are_bit_exact(gpu, golden):
    """sample_convert.h through the C ABI: SHA-256 of the GPU output == the reference's."""
    from test_oracle import _kat_inputs
    meta, _ = golden
    kats = meta["conversion_kats"]
    ins, x = _kat_inputs()
    for fmt, raw in ins.items():
        for gain in (1.0, 0.5, 1.2345):
            y = gpu.convert_block_to_cf32(raw, FORMAT_CODES[fmt], raw.size // 2, gain)
            assert hashlib.sha256(y.tobytes()).hexdigest() == kats[f"to_cf32/{fmt}/gain={gain}"], (fmt, gain)
    for fmt in ("cs8", "cu8", "cs16", "cu16", "sc16q11", "cs24", "cs32", "cu32", "cf32"):
        y = gpu.convert_cf32_to_block(x, FORMAT_CODES[fmt], NUMPY_DTYPE[fmt], BYTES_PER_SAMPLE[fmt])
        assert hashlib.sha256(y.tobytes()).hexdigest() == kats[f"from_cf32/{fmt}"], fmt


def test_all_input_formats_roundtrip_against_oracle(gpu):
    rng = np.random.Generator(np.random.PCG64(31))
    n = 20000
    for fmt in ("cs8", "cu8", "cs16", "cu16", "sc16q11", "cs24", "cs32", "cu32", "cf32"):
        if fmt == "cf32":
            raw = (rng.standard_normal(2 * n) * 0.3).astype(np.float32)
        elif fmt == "cs24":
            raw = rng.integers(0, 256, 6 * n, dtype=np.uint8)
        else:
            info = np.iinfo(NUMPY_DTYPE[fmt])
            raw = rng.integers(info.min, info.max, 2 * n, dtype=NUMPY_DTYPE[fmt], endpoint=True)
        cfg = ChainConfig(input_format=fmt, output_format="cf32", input_rate_hz=1e6, target_rate_hz=1e6,
                          no_resample=True, gain=0.75)
        out = gpu.Chain(cfg, 0).process(raw)
        ref = CpuChain(cfg, "oracle").process(raw)
        assert np.array_equal(out.view(np.uint32), ref.view(np.uint32)), fmt


# ---------------------------------------------------------------------------------------------
# fused front kernel (convert + DC + I/Q + NCO + halfband cascade + polyphase in one HBM pass)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,n", [("cfg1", (1 << 22) + 4097), ("cfg5", (1 << 23) + 11), ("cfg2", (1 << 22) + 333)])
def test_fused_front_equals_stage_by_stage_path(name, n, gpu, workloads):
    wl = workloads[name]
    raw = synth_numpy(wl, n)
    a = gpu.Chain(wl.config, 0, record_taps=1, fused=1)
    b = gpu.Chain(wl.config, 0, record_taps=1, fused=0)
    ya, ca = a.process(raw, return_chunk_counts=True)
    yb, cb = b.process(raw, return_chunk_counts=True)
    assert a.info().fused_front == 1 and b.info().fused_front == 0
    assert np.array_equal(ca, cb)
    ta, tb = a.read_tap(1), b.read_tap(1)
    assert ta.size == tb.size
    if not wl.config.dc_block:
        assert np.array_equal(ta.view(np.uint32), tb.view(np.uint32))    # same FMA order -> same bits
        assert np.array_equal(ya, yb)
    else:
        assert rel_rms_fullscale(ta, tb) <= 1e-7
        assert max_lsb(ya, yb) <= 1


@pytest.mark.parametrize("rate", [744187.5, 2.4e6, 9.0e6])
def test_fused_front_gain_that_is_not_a_power_of_two(rate, gpu):
    """sample_convert.c:136-141 rounds (x / 32768) * gain once per component before anything else sees it.  The packed
    conversion in the fused front feeds packed adds of the first halfband stage; ptxas 12.9 contracts mul.rn.f32x2 +
    add.rn.f32x2 into FFMA2 when it can (it does not for the scalar forms), which would skip that rounding.  With a gain of
    0.7 the product is inexact, so a contraction shows as a bit difference from the stage-by-stage kernels (S = 4, 3, 1)."""
    cfg = ChainConfig(input_format="cs16", output_format="cf32", input_rate_hz=20e6, target_rate_hz=rate, gain=0.7)
    rng = np.random.Generator(np.random.PCG64(5))
    raw = rng.integers(-32768, 32768, size=2 * ((1 << 21) + 777), dtype=np.int16)
    a = gpu.Chain(cfg, 0, fused=1)
    b = gpu.Chain(cfg, 0, fused=0)
    ya, yb = a.process(raw), b.process(raw)
    assert a.info().fused_front == 1 and b.info().fused_front == 0
    assert ya.size == yb.size and np.array_equal(ya.view(np.uint32), yb.view(np.uint32))


@pytest.mark.parametrize("name,n", [("cfg1", (1 << 22) + 4097), ("cfg5", (1 << 23) + 11)])
def test_fused_front_parity_vs_oracle(name, n, gpu, workloads):
    wl = workloads[name]
    raw = synth_numpy(wl, n)
    g, o, out, ref, counts = _run_pair(gpu, wl.config, raw, taps=1)
    assert g.info().fused_front == 1
    assert np.array_equal(counts, o.traced())
    assert rel_rms_fullscale(g.read_tap(1), o.captured(1)) <= 1e-6
    assert snr_db(g.read_tap(1), o.captured(1)) >= 120.0
    _check_final(wl.config, out, ref)


def test_fused_front_is_call_size_invariant(gpu, workloads):
    """Ragged calls (1 frame, odd sizes, sizes straddling block and run boundaries) through the
    fused kernel == one big call, bit for bit: tests the cf32 tail, absolute-index alignment,
    warm-up blocks and the DC table rewind."""
    import dataclasses
    for name in ("cfg5", "cfg2"):
        wl = workloads[name]
        cfg = dataclasses.replace(wl.config, output_format="cf32", agc_enable=False, filters=[], filter_taps=0,
                                  filter_type_request=0)
        n = 300000
        raw = synth_numpy(wl, n)
        one = gpu.Chain(cfg, 0, fused=1).process(raw).view(np.complex64)
        g = gpu.Chain(cfg, 0, fused=1)
        parts, pos = [], 0
        for m in (1, 3, 127, 2048, 5000, 4095, 16384, 100001, 50000, n):
            m = min(m, n - pos)
            if m <= 0:
                break
            parts.append(g.process(raw[2 * pos:2 * (pos + m)], chunk_frames=[m]))
            pos += m
        many = np.concatenate(parts).view(np.complex64)
        assert many.size == one.size
        if cfg.dc_block:
            # the one-call run evaluates the DC blocker per warp stretch (local state + closed-form correction), the
            # ragged calls from the carried state: two fp32 evaluation orders of the same arithmetic
            assert rel_rms_fullscale(many, one) <= 1e-7
        else:
            assert np.array_equal(many.view(np.uint32), one.view(np.uint32))


def test_fused_cu8_and_cf32_inputs(gpu):
    rng = np.random.Generator(np.random.PCG64(41))
    n = 200000
    for fmt, raw in (("cu8", rng.integers(0, 256, 2 * n, dtype=np.uint8)),
                     ("cf32", (rng.standard_normal(2 * n) * 0.3).astype(np.float32)),
                     ("cs8", rng.integers(-128, 128, 2 * n, dtype=np.int8))):
        cfg = ChainConfig(input_format=fmt, output_format="cf32", input_rate_hz=2.4e6, target_rate_hz=250e3,
                          freq_shift_hz=37e3, gain=0.8)
        g, o, out, ref, counts = _run_pair(gpu, cfg, raw, taps=1)
        assert g.info().fused_front == 1 and np.array_equal(counts, o.traced())
        _check_final(cfg, out, ref)


# ---------------------------------------------------------------------------------------------
# K4: FFT block filter (hand-written FFT, overlap-save evaluation of liquid's overlap-add fftfilt)
# ---------------------------------------------------------------------------------------------
def test_cfg3_golden_fixture_parity(gpu, workloads, golden):
    """cfg3 vs the committed reference outputs: 4095 complex taps, block n = 8192 (FFT 16384),
    outputs quantised to whole FFT blocks per chunk, post-resample LUT-NCO shift, cs16."""
    meta, data = golden
    cfg = workloads["cfg3"].config
    g = gpu.Chain(cfg, 0, record_taps=1)
    out, counts = g.process(data["cfg3"]["raw"], return_chunk_counts=True)
    assert np.array_equal(counts, data["cfg3"]["counts"])
    taps = g.filter_taps()
    assert taps.size == 4095 and rel_rms_fullscale(taps, data["cfg3"]["filter_taps"]) <= 1e-9
    rs = g.read_tap(1)
    assert rs.size == data["cfg3"]["rs"].size
    assert rel_rms_fullscale(rs, data["cfg3"]["rs"]) <= 1e-6
    _check_final(cfg, out, data["cfg3"]["out"])


@pytest.mark.parametrize("fused", [0, 1])
def test_cfg3_parity_vs_oracle(fused, gpu, workloads):
    wl = workloads["cfg3"]
    n = (1 << 21) + 4099
    raw = synth_numpy(wl, n)
    g, o, out, ref, counts = _run_pair(gpu, wl.config, raw, taps=1, fused=fused)
    assert g.info().fused_front == fused
    assert np.array_equal(counts, o.traced())           # 0 or 8192 frames per chunk
    assert set(np.unique(counts)) <= {0, 8192}
    assert snr_db(g.read_tap(1), o.captured(1)) >= 120.0
    _check_final(wl.config, out, ref)


def test_fft_filter_equals_fir_filter_and_oracle(gpu):
    """Same master taps through K4 (FFT) and K3 (FIR): identical streams up to fp32 rounding; FFT
    output length is the whole-block prefix.  Covers real (crcf) and complex (cccf) taps, small
    and odd-log2 transform sizes, and ragged chunking of the FFT remainder."""
    from iq_tool_b200.configs import FILTER_REQ_FFT, pass_range
    rng = np.random.Generator(np.random.PCG64(51))
    n = 5 * 16384 + 1234
    x = ((rng.standard_normal(n) + 1j * rng.standard_normal(n)) * 0.2).astype(np.complex64)
    for filt, taps, fftsize in (([lowpass(100e3)], 255, 0), ([pass_range(102e3, 215e3)], 301, 0),
                                ([lowpass(200e3)], 21, 0), ([pass_range(50e3, 90e3)], 1025, 4096),
                                ([lowpass(50e3)], 63, 128)):
        base = dict(input_format="cf32", output_format="cf32", input_rate_hz=1e6, target_rate_hz=1e6,
                    no_resample=True, filters=filt, filter_taps=taps)
        cfg_fft = ChainConfig(filter_type_request=FILTER_REQ_FFT, filter_fft_size=fftsize, **base)
        cfg_fir = ChainConfig(filter_type_request=FILTER_REQ_FIR, **base)
        g, o, out, ref, counts = _run_pair(gpu, cfg_fft, x.view(np.float32), taps=1)
        assert np.array_equal(counts, o.traced())
        _check_final(cfg_fft, out, ref)
        fir = gpu.Chain(cfg_fir, 0).process(x.view(np.float32)).view(np.complex64)
        a = out.view(np.complex64)
        assert a.size % g.info().filter_block_size == 0 and a.size <= fir.size
        assert rel_rms_fullscale(a, fir[: a.size]) <= 2e-6
        # ragged calls carry the remainder exactly like one call
        g2 = gpu.Chain(cfg_fft, 0)
        parts, pos = [], 0
        for m in (1, 100, 16384, 5000, 40000, n):
            m = min(m, n - pos)
            if m <= 0:
                break
            parts.append(g2.process(x.view(np.float32)[2 * pos:2 * (pos + m)], chunk_frames=[m]))
            pos += m
        assert np.array_equal(np.concatenate(parts).view(np.uint32), out.view(np.uint32))


def test_fft_filter_large_transform_split_path(gpu):
    """2n = 65536 > the shared-memory transform: radix-2 global stages + 16384-point sub-blocks.
    Post-resample placement (the reference's pre-resample FFT path corrupts its input when the
    block exceeds the chunk, SURVEY row F4)."""
    from iq_tool_b200.configs import FILTER_REQ_FFT
    rng = np.random.Generator(np.random.PCG64(52))
    n = 20 * 16384
    x = ((rng.standard_normal(n) + 1j * rng.standard_normal(n)) * 0.2).astype(np.complex64)
    cfg = ChainConfig(input_format="cf32", output_format="cf32", input_rate_hz=2e6, target_rate_hz=1e6,
                      filters=[lowpass(20e3)], filter_taps=9001,
                      filter_type_request=FILTER_REQ_FFT, filter_fft_size=65536)
    g, o, out, ref, counts = _run_pair(gpu, cfg, x.view(np.float32), taps=1)
    assert g.info().filter_block_size == 32768 and g.info().filter_post_resample == 1
    assert out.size == 2 * 5 * 32768
    assert np.array_equal(counts, o.traced())
    _check_final(cfg, out, ref)


# ---------------------------------------------------------------------------------------------
# K6: I/Q optimiser pass (iq_correct_run_optimization) — function-level parity with injected RNG
# ---------------------------------------------------------------------------------------------
def test_iq_optimizer_pass_matches_reference(gpu, workloads):
    from oracle.loader import libc_rand_directions
    wl = workloads["cfg4"]
    cfg = wl.config
    x = synth_numpy(wl, 4096)
    blk = ((x.astype(np.float32) - 127.5) / 128.0).view(np.complex64)[:1024]
    kind = _oracle_kind()
    for seed in (1, 7, 12345):
        o = CpuChain(cfg, kind)
        rm, rp, ra, rr = o.iq_optimize(blk, seed)
        gm, gp, ga, gr = gpu.iq_optimize(blk, libc_rand_directions(seed), cfg.iq_mag, cfg.iq_phase)
        assert abs(ga - ra) <= 1e-3 and abs(gr - rr) <= 1e-3          # dB
        # one flipped accept/reject (metric ties at fp32 rounding) moves a factor by 0.05 * 1e-4
        assert abs(gm - rm) <= 1.1e-5 and abs(gp - rp) <= 1.1e-5, (seed, gm, rm, gp, rp)
    # weak signal (peak-to-average < 20 dB): factors untouched, like iq_correct.c:168-171
    rng = np.random.Generator(np.random.PCG64(3))
    noise = ((rng.standard_normal(1024) + 1j * rng.standard_normal(1024)) * 0.1).astype(np.complex64)
    gm, gp, ga, gr = gpu.iq_optimize(noise, libc_rand_directions(1), 0.01, -0.02)
    assert gr < 20.0 and gm == np.float32(0.01) and gp == np.float32(-0.02)


def _digital_agc_schedule(gpu, amps, pieces_list, seed=77):
    """Runs the per-chunk amplitude schedule `amps` through the digital AGC on the GPU (one train and ragged trains) and
    through the oracle chunk by chunk on the sample clock; returns the oracle's per-chunk gains."""
    from oracle import loader
    rate, chunk = 512.0, 64                      # one chunk = 0.125 s: lock after 17 chunks, creep after 32 weak ones
    rng = np.random.Generator(np.random.PCG64(seed))
    amps = np.asarray(amps, dtype=np.float32)
    nchunks = amps.size
    ph = rng.uniform(0, 2 * np.pi, size=nchunks * chunk)
    mag = rng.uniform(0.2, 1.0, size=nchunks * chunk)
    mag[::chunk] = 1.0                                               # every chunk reaches its amplitude
    x = (np.repeat(amps, chunk) * mag * np.exp(1j * ph)).astype(np.complex64)
    cfg = ChainConfig(input_format="cf32", output_format="cf32", input_rate_hz=rate, target_rate_hz=rate,
                      no_resample=True, agc_enable=True, agc_profile=AGC_DIGITAL)
    lib, pfx = loader.get_lib("oracle")
    o = CpuChain(cfg, "oracle")
    ref = np.zeros_like(x)
    try:
        for c in range(nchunks):
            getattr(lib, pfx + "set_fake_clock")(1, c * chunk / rate)
            ref[c * chunk:(c + 1) * chunk] = o.process(x[c * chunk:(c + 1) * chunk].view(np.float32)).view(np.complex64)
    finally:
        getattr(lib, pfx + "set_fake_clock")(0, 0.0)
    oi = o.info()
    sizes = np.full(nchunks, chunk, dtype=np.uint32)
    gain_r = np.abs(ref[::chunk]) / amps
    for pieces in pieces_list:                                       # one train, and ragged trains (state carried)
        g = gpu.Chain(cfg, 0)
        outs, edges = [], np.linspace(0, nchunks, pieces + 1).astype(int)
        for a, b in zip(edges[:-1], edges[1:]):
            outs.append(g.process(x[a * chunk:b * chunk].view(np.float32), chunk_frames=sizes[a:b]).view(np.complex64))
        out = np.concatenate(outs)
        assert out.size == ref.size
        gi = g.info()
        assert (gi.agc_locked, gi.agc_samples_seen) == (oi.agc_locked, oi.agc_samples_seen)
        assert gi.agc_gain == pytest.approx(oi.agc_gain, rel=3e-7) and gi.agc_peak_memory == pytest.approx(oi.agc_peak_memory, rel=3e-7)
        gain_g = np.abs(out[::chunk]) / amps
        assert np.allclose(gain_g, gain_r, rtol=1e-6, atol=0)
        assert np.allclose(out, ref, rtol=1e-6, atol=1e-9)
    return gain_r


def test_digital_agc_chunk_table_scan_equals_the_sequential_state_machine(gpu):
    """G2 (agc.c:105-222) over thousands of chunks in ONE train: the GPU evaluates the per-chunk state
    machine with a parallel scan over the chunk table (event-free stretches in one step, chunks with a lock
    transition / ratchet / creep replayed sequentially); the oracle walks the chunks one by one on the
    sample clock.  The amplitude schedule covers scanning with a rising peak memory, the lock, long
    event-free locked stretches (several scan tiles), isolated and back-to-back ratchets, 'strong'
    refreshes, and long creep phases."""
    rng = np.random.Generator(np.random.PCG64(77))
    amps = [0.05, 0.1, 0.2, 0.15, 0.4] + [0.3] * 30                 # scan, lock at chunk 17
    amps += [0.5, 0.45, 0.44]                                        # ratchet(s)
    amps += [0.42] * 2500                                            # strong, event free: > one 2048-chunk tile
    amps += [0.03] * 300                                             # weak: creep starts after 32 chunks
    amps += [0.9, 0.95, 1.0, 0.2]                                    # ratchets back to back
    amps += list(rng.choice([0.02, 0.3, 0.45, 0.7], size=1500, p=[0.5, 0.3, 0.15, 0.05]))   # mixed
    amps += [0.25] * 2200 + [0.6] + [0.01] * 100
    # a ratchet, then 3000 strong chunks in which nothing happens: with ragged trains two whole trains lie inside that
    # stretch — the grid-wide quiet test answers for them and writes their (single) gain, the scan kernel is skipped
    amps += [0.5] * 40 + [0.45] * 3000
    gain_r = _digital_agc_schedule(gpu, amps, (1, 7))
    # the schedule really exercised every branch
    assert gain_r[40] < gain_r[30] and gain_r[2500 + 38 + 290] > gain_r[2500 + 38 + 10]


@pytest.mark.parametrize("tail", ["quiet", "ratchet_and_creep"])
def test_digital_agc_long_table_is_asked_again_behind_its_head(tail, gpu):
    """A train of more than 3 x 8192 chunks that starts with the scanning phase and the lock is not quiet as a whole; the
    scan kernel then walks only a head of 8192 chunks and the rest of the table is asked again with the state behind the
    head (launch_agc_digital_scan).  `quiet`: nothing happens behind the head — gains come from the quiet test, the scan of
    the rest is skipped.  `ratchet_and_creep`: events behind the head — the scan kernel takes the rest after all.  One
    train (head + rest), and three trains (the later ones are quiet / not quiet as a whole)."""
    amps = [0.05, 0.1, 0.2, 0.15, 0.4] + [0.3] * 30 + [0.5, 0.45, 0.44] + [0.42] * 9000
    if tail == "quiet":
        amps += [0.44] * 17000
    else:
        amps += [0.44] * 6000 + [0.6, 0.55] + [0.5] * 5000 + [0.02] * 200 + [0.5] * 5800
    gain_r = _digital_agc_schedule(gpu, amps, (1, 3), seed=78)
    if tail != "quiet":
        k = 38 + 9000 + 6000
        assert gain_r[k + 3] < gain_r[k - 3] and gain_r[k + 2 + 5000 + 190] > gain_r[k + 2 + 5000 + 10]    # ratchet, creep


@pytest.mark.parametrize("out_fmt", ["cs16", "cu8", "cs8"])
def test_fir_epilogue_conversion_equals_the_post_kernel(out_fmt, gpu, workloads, monkeypatch):
    """When the FIR is the chain's last cf32 stage its epilogue converts to the output format (C2,
    sample_convert.c:213-306) instead of a separate post kernel: same bytes either way, ragged length,
    several sub-trains, and the oracle's +-1 LSB bar."""
    import dataclasses
    wl = dataclasses.replace(workloads["cfg2"], dc=0.0)
    cfg = dataclasses.replace(wl.config, output_format=out_fmt)
    raw = synth_numpy(wl, (1 << 21) + 4321)
    a = gpu.Chain(cfg, 0, subtrain_frames=1 << 19).process(raw)
    monkeypatch.setenv("IQGPU_FIR_NO_CONVERT", "1")
    b = gpu.Chain(cfg, 0, subtrain_frames=1 << 19).process(raw)
    monkeypatch.delenv("IQGPU_FIR_NO_CONVERT")
    assert a.size == b.size and np.array_equal(a, b)
    ref = CpuChain(cfg, _oracle_kind()).process(raw)
    assert a.size == ref.size and max_lsb(a, ref) <= INT_LSB_TOL


@pytest.mark.parametrize("S", [0, 1, 2, 3, 4, 5, 6])
def test_fused_front_every_cascade_depth(S, gpu, monkeypatch):
    """Every compiled cascade plan of the warp-streaming fused front (S = 0..6 halfband stages: register first stage
    for S >= 3, deep stages on 128 / 64 outputs per run) against the stage-by-stage kernels: same FMA order -> same
    bits; against the oracle: the north_star bar; ragged calls (incl. an empty one) == one call."""
    rng = np.random.Generator(np.random.PCG64(100 + S))
    fs = 10e6
    target = fs * 0.61 / (1 << S)
    n = 120000 + (40000 << S) + 77
    t = np.arange(n)
    x = 0.3 * np.exp(2j * np.pi * (0.11 / (1 << S)) * t) + 0.05 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    raw = np.empty(2 * n, dtype=np.int16)
    raw[0::2] = np.clip(np.round(x.real * 32767), -32768, 32767)
    raw[1::2] = np.clip(np.round(x.imag * 32767), -32768, 32767)
    cfg = ChainConfig(input_format="cs16", output_format="cf32", input_rate_hz=fs, target_rate_hz=target,
                      freq_shift_hz=-123e3)
    a = gpu.Chain(cfg, 0, fused=1)
    b = gpu.Chain(cfg, 0, fused=0)
    ya, ca = a.process(raw, return_chunk_counts=True)
    yb, cb = b.process(raw, return_chunk_counts=True)
    ia = a.info()
    assert ia.fused_front == 1 and b.info().fused_front == 0 and ia.num_halfband == S
    assert np.array_equal(ca, cb)
    assert ya.size == yb.size and np.array_equal(ya.view(np.uint32), yb.view(np.uint32))
    o = CpuChain(cfg, _oracle_kind())
    o.trace(n // 16384 + 4)
    ref = o.process(raw)
    assert np.array_equal(ca, o.traced())
    _check_final(cfg, ya.view(np.float32), ref)
    g = gpu.Chain(cfg, 0, fused=1)
    parts, pos = [], 0
    for m in (1, 0, 511, 513, 4096 << S, 16385, 100000, n):
        m = min(m, n - pos)
        if m == 0 and pos:
            parts.append(g.process(raw[:0]))
            continue
        if m <= 0:
            break
        parts.append(g.process(raw[2 * pos:2 * (pos + m)], chunk_frames=[m]))
        pos += m
    many = np.concatenate(parts)
    assert many.size == ya.size and np.array_equal(many.view(np.uint32), ya.view(np.uint32))
    # the polyphase stage with two and with four outputs per lane (picked by timing on long calls, forced here): same bits
    for mode in ("1", "2"):
        monkeypatch.setenv("IQGPU_ARB_PAIRS", mode)
        ym = gpu.Chain(cfg, 0, fused=1).process(raw)
        monkeypatch.delenv("IQGPU_ARB_PAIRS")
        assert ym.size == ya.size and np.array_equal(ym.view(np.uint32), ya.view(np.uint32))


@pytest.mark.parametrize("S", [7, 8, 9])
def test_deep_cascades_run_the_stage_kernels(S, gpu):
    """Cascades deeper than the fused front's compiled plans (S = 7..9 halfband stages, down to the 0.001 ratio floor;
    S = 8 is 20 Msps -> 48 kHz) run the stage-by-stage kernels even where the fused front is allowed: NCO pre-shift
    (and the DC blocker for S = 8), per-chunk counts equal to the oracle's, the north_star bar against the oracle, ragged
    calls (incl. an empty one) == one call."""
    rng = np.random.Generator(np.random.PCG64(200 + S))
    fs = 20e6
    target = fs * 0.61 / (1 << S)
    n = (1 << 20) + (20000 << S) + 77
    t = np.arange(n)
    # a tone that the pre-shift moves into the output band, plus wideband noise
    x = 0.3 * np.exp(2j * np.pi * ((123e3 + 0.1 * target) / fs) * t) + \
        0.05 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    raw = np.empty(2 * n, dtype=np.int16)
    raw[0::2] = np.clip(np.round(x.real * 32767), -32768, 32767)
    raw[1::2] = np.clip(np.round(x.imag * 32767), -32768, 32767)
    cfg = ChainConfig(input_format="cs16", output_format="cf32", input_rate_hz=fs, target_rate_hz=target,
                      freq_shift_hz=-123e3, dc_block=(S == 8))
    g = gpu.Chain(cfg, 0, fused=1)
    y, counts = g.process(raw, return_chunk_counts=True)
    info = g.info()
    assert info.fused_front == 0 and info.num_halfband == S
    o = CpuChain(cfg, _oracle_kind())
    o.trace(n // 16384 + 4)
    ref = o.process(raw)
    assert np.array_equal(counts, o.traced())
    _check_final(cfg, y.view(np.float32), ref)
    g = gpu.Chain(cfg, 0, fused=1, subtrain_frames=1 << 24)      # one chunk per call, the last one up to 9.1e6 frames
    parts, pos = [], 0
    for m in (1, 0, 511, 513, 4096 << S, 16385, 100000, n):
        m = min(m, n - pos)
        if m == 0 and pos:
            parts.append(g.process(raw[:0]))
            continue
        if m <= 0:
            break
        parts.append(g.process(raw[2 * pos:2 * (pos + m)], chunk_frames=[m]))
        pos += m
    many = np.concatenate(parts)
    assert many.size == y.size
    if cfg.dc_block:
        # the DC scan of the stage path restarts its runs at every call: two fp32 evaluation orders of the same arithmetic
        assert rel_rms_fullscale(many.view(np.complex64), y.view(np.complex64)) <= 1e-7
    else:
        assert np.array_equal(many.view(np.uint32), y.view(np.uint32))


@pytest.mark.parametrize("S", [1, 4, 6])
@pytest.mark.parametrize("rate", [0.505, 0.55, 0.66, 0.7, 0.8, 0.97])
def test_polyphase_variants_are_bit_identical_at_every_rate_class(S, rate, gpu, monkeypatch):
    """The four-output polyphase variant has a compiled form per (floor(2/rate), floor(3/rate)) = (3,5), (3,4), (2,4),
    (2,3); rates outside them fall back to two outputs per lane.  Every variant, shallow (skewed level, S = 1) and deep
    (plain level, S = 4, 6) cascades, DC blocker on (local DC state: the closed-form term uses the same row gains): the same
    bits as one output per lane."""
    rng = np.random.Generator(np.random.PCG64(int(1000 * rate) + S))
    fs = 8e6
    n = (1 << 19) + (3000 << S) + 13
    raw = rng.integers(-20000, 20000, size=2 * n, dtype=np.int16)
    cfg = ChainConfig(input_format="cs16", output_format="cf32", input_rate_hz=fs, target_rate_hz=fs * rate / (1 << S),
                      dc_block=True)
    outs = []
    for mode in ("0", "1", "2"):
        monkeypatch.setenv("IQGPU_ARB_PAIRS", mode)
        g = gpu.Chain(cfg, 0, fused=1)
        outs.append(g.process(raw))
        assert g.info().fused_front == 1 and g.info().num_halfband == S
        monkeypatch.delenv("IQGPU_ARB_PAIRS")
    assert outs[0].size == outs[1].size == outs[2].size
    assert np.array_equal(outs[0].view(np.uint32), outs[1].view(np.uint32))
    assert np.array_equal(outs[0].view(np.uint32), outs[2].view(np.uint32))


def test_fused_dc_local_state_equals_the_table_pre_pass(gpu, workloads, monkeypatch):
    """DC blocker inside the fused front, two evaluations: (a) v at every tick start from a pre-pass over the raw stream
    (IQGPU_DC_TABLE=1), (b) every warp carries v through its own stretch from zero and the missing decaying exponential —
    an eigenfunction of the linear cascade — is added to the resampler output in closed form (no second read of the input).
    Same stream within fp32 round-off, over hundreds of stretches, a DC offset 100x the blocker's usual load, ragged
    multi-call input (carried state, corrected cf32 tail), and the oracle's bar at the chain output."""
    import dataclasses
    wl = dataclasses.replace(workloads["cfg2"], dc=0.2)
    cfg = dataclasses.replace(wl.config, output_format="cf32", filters=[], filter_taps=0, filter_type_request=0)
    n = (1 << 23) + 12345
    raw = synth_numpy(wl, n)
    a = gpu.Chain(cfg, 0, fused=1, subtrain_frames=1 << 24).process(raw).view(np.complex64)
    cuts = [0, 3000001, 3000002, 5 << 20, n]
    g = gpu.Chain(cfg, 0, fused=1, subtrain_frames=1 << 24)
    parts = [g.process(raw[2 * lo:2 * hi], chunk_frames=[hi - lo]) for lo, hi in zip(cuts[:-1], cuts[1:])]
    b = np.concatenate(parts).view(np.complex64)
    monkeypatch.setenv("IQGPU_DC_TABLE", "1")
    t = gpu.Chain(cfg, 0, fused=1, subtrain_frames=1 << 24).process(raw).view(np.complex64)
    monkeypatch.delenv("IQGPU_DC_TABLE")
    assert a.size == t.size == b.size
    assert rel_rms_fullscale(a, t) <= 1e-7 and np.abs(a - t).max() <= 2e-6
    assert rel_rms_fullscale(b, t) <= 1e-7 and np.abs(b - t).max() <= 2e-6
    # the blocker did its job in both: the 0.2 offset is gone from the settled part of the stream
    assert abs(a[a.size // 2:].mean()) < 2e-3


def test_fir_adds_the_fronts_dc_term_while_staging_its_tiles(gpu, workloads, monkeypatch):
    """cfg2 as specified (DC offset, local DC state in the fused front, 255-tap FIR behind the resampler): the FIR adds the
    front's closed-form DC term to the samples it stages instead of a separate read-modify-write pass over the resampled
    stream (the newest taps-1 samples, the next call's history, get it in memory afterwards).  Same bytes as with the
    separate pass (IQGPU_NO_DC_FOLD=1), one call or ragged calls that are shorter than, equal to and longer than the
    filter history, cs16 output (FIR epilogue conversion), cf32 output (post kernel behind the FIR) and an asymmetric pass
    range (complex taps)."""
    import dataclasses
    wl = workloads["cfg2"]
    n = (1 << 22) + 7777
    raw = synth_numpy(wl, n)
    cuts = [0, 1 << 20, (1 << 20) + 3000, (1 << 20) + 3000 + 16384, 3 << 20, n]
    from iq_tool_b200.configs import pass_range
    variants = [("cs16", wl.config.filters), ("cf32", wl.config.filters), ("cu8", [pass_range(20e3, 180e3)])]   # last: complex taps
    for out_fmt, filters in variants:
        cfg = dataclasses.replace(wl.config, output_format=out_fmt, filters=filters)
        def run(split):
            if not split:
                return gpu.Chain(cfg, 0, subtrain_frames=1 << 20).process(raw)          # several sub-trains in one call
            g = gpu.Chain(cfg, 0, subtrain_frames=1 << 22)
            return np.concatenate([g.process(raw[2 * lo:2 * hi], chunk_frames=[hi - lo]) for lo, hi in zip(cuts[:-1], cuts[1:])])
        a, a_split = run(False), run(True)
        monkeypatch.setenv("IQGPU_NO_DC_FOLD", "1")
        b, b_split = run(False), run(True)
        monkeypatch.delenv("IQGPU_NO_DC_FOLD")
        view = (lambda v: v.view(np.uint32)) if out_fmt == "cf32" else (lambda v: v)
        assert a.size == b.size and np.array_equal(view(a), view(b))
        assert a_split.size == b_split.size and np.array_equal(view(a_split), view(b_split))


def test_long_post_resample_fir_runs_on_the_fft_block_kernel(gpu, workloads, monkeypatch):
    """A long time-domain FIR (F2, filter.c:449-462) after the resampler is evaluated by the overlap-save FFT kernel — the
    same causal convolution with ~20x fewer FLOPs.  It must equal the tiled time-domain kernel within fp32 round-off, be
    independent of how the stream is cut into calls (partial last blocks, history carried in the stream), keep the FIR's
    output count (no block quantisation), and meet the oracle's bar."""
    wl = workloads["cfg1"]
    cfg = ChainConfig(input_format="cs16", output_format="cf32", input_rate_hz=2.4e6, target_rate_hz=1.0e6,
                      filters=[lowpass(150e3)], filter_taps=1001, filter_type_request=FILTER_REQ_FIR)
    n = 700001
    raw = synth_numpy(wl, n)
    a = gpu.Chain(cfg, 0)
    ya = a.process(raw).view(np.complex64)
    assert a.info().filter_post_resample == 1 and a.info().filter_num_taps == 1001
    g = gpu.Chain(cfg, 0)
    parts, pos = [], 0
    for m in (5, 16384, 40000, 300001, n):
        m = min(m, n - pos)
        if m <= 0:
            break
        parts.append(g.process(raw[2 * pos:2 * (pos + m)], chunk_frames=[m]))
        pos += m
    yb = np.concatenate(parts).view(np.complex64)
    monkeypatch.setenv("IQGPU_FIR_TIME_DOMAIN", "1")
    yt = gpu.Chain(cfg, 0).process(raw).view(np.complex64)
    monkeypatch.delenv("IQGPU_FIR_TIME_DOMAIN")
    assert ya.size == yt.size == yb.size
    assert rel_rms_fullscale(ya, yt) <= 2e-6 and np.abs(ya - yt).max() <= 2e-5
    assert rel_rms_fullscale(yb, yt) <= 2e-6
    ref = CpuChain(cfg, _oracle_kind()).process(raw)
    _check_final(cfg, ya.view(np.float32), ref)


# ---------------------------------------------------------------------------------------------
# interpolation (r > 1): arbitrary stage first, then halfband interpolators (msresamp_crcf INTERP, resampler.c:49)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["interp_1p5", "interp_6", "upsample_prefilter"])
def test_interpolating_resampler_parity(name, gpu):
    """r = 1.5 (S = 0), r = 6 (S = 2: arbitrary stage at 1.5, two halfband interpolators) and an up-sampling chain whose
    user filter therefore stays pre-resample (filter.c:43-92): output counts exact, resampler stream <= 1e-6 / >= 120 dB,
    final stream at the north_star bar, ragged calls == one call bit for bit."""
    from test_host_logic import EXTRA
    cfg = EXTRA[name]
    rng = np.random.Generator(np.random.PCG64(61))
    n = 12 * 16384 + 777
    t = np.arange(n)
    x = 0.3 * np.exp(2j * np.pi * 0.037 * t) + 0.1 * np.exp(-2j * np.pi * 0.11 * t) + \
        0.02 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    if cfg.input_format == "cf32":
        raw = x.astype(np.complex64).view(np.float32)
    else:
        raw = np.empty(2 * n, dtype=np.int16)
        raw[0::2] = np.clip(np.rint(x.real * 32767), -32768, 32767)
        raw[1::2] = np.clip(np.rint(x.imag * 32767), -32768, 32767)
    g = gpu.Chain(cfg, 0, record_taps=2)
    o = CpuChain(cfg, _oracle_kind())
    o.capture(1, int(n * cfg.ratio) + 4096)            # the resampled stream is longer than the input here
    o.trace(n // 16384 + 4)
    ref = o.process(raw)
    out, counts = g.process(raw, return_chunk_counts=True)
    gi = g.info()
    assert gi.is_interp == 1 and gi.fused_front == 0
    assert np.array_equal(counts, o.traced())
    assert g.read_tap(1).size == o.captured(1).size
    assert rel_rms_fullscale(g.read_tap(1), o.captured(1)) <= 1e-6 and snr_db(g.read_tap(1), o.captured(1)) >= 120.0
    _check_final(cfg, out, ref)
    g2 = gpu.Chain(cfg, 0)
    parts, pos = [], 0
    for m in (1, 2, 127, 4097, 16384, 50001, n):
        m = min(m, n - pos)
        if m <= 0:
            break
        parts.append(g2.process(raw[2 * pos:2 * (pos + m)], chunk_frames=[m]))
        pos += m
    many = np.concatenate(parts)
    assert many.size == out.size and np.array_equal(many.view(np.uint8), out.view(np.uint8))


def test_fft_filter_remainder_survives_a_stream_discontinuity_like_the_reference(gpu):
    """SURVEY 8(a) F5: filter_reset (filter.c:417-436) clears liquid's overlap state but not post/pre_fft_remainder_len, so
    after a discontinuity the frames that were waiting for a full block are filtered in front of the new stream (with an
    empty overlap).  iqgpu_chain_reset reproduces that, post- and pre-resample; iqgpu_chain_restart is a fresh chain."""
    from iq_tool_b200.configs import FILTER_REQ_FFT
    rng = np.random.Generator(np.random.PCG64(71))
    n1, n2 = 3 * 16384 + 1500, 2 * 16384 + 4000
    x = ((rng.standard_normal(n1 + n2) + 1j * rng.standard_normal(n1 + n2)) * 0.2).astype(np.complex64).view(np.float32)
    for rates in ((2e6, 1e6), (1e6, 1e6)):                 # post-resample filter (decimation) / pre-resample (no_resample)
        cfg = ChainConfig(input_format="cf32", output_format="cf32", input_rate_hz=rates[0], target_rate_hz=rates[1],
                          no_resample=(rates[0] == rates[1]), filters=[lowpass(100e3)], filter_taps=301,
                          filter_type_request=FILTER_REQ_FFT, filter_fft_size=2048)
        g = gpu.Chain(cfg, 0)
        o = CpuChain(cfg, _oracle_kind())
        a1, b1 = g.process(x[: 2 * n1]), o.process(x[: 2 * n1])
        assert a1.size == b1.size and a1.size % (2 * 1024) == 0
        waiting = (n1 if cfg.no_resample else g.resampler_outputs_after(n1)) - a1.size // 2
        assert 0 < waiting < 1024                          # the case under test: frames are waiting at the discontinuity
        g.reset()
        a2 = g.process(x[2 * n1:])
        if not cfg.no_resample:
            o.reset()
            b2 = o.process(x[2 * n1:])
            assert a2.size == b2.size                      # the waiting frames count towards the new stream's blocks
            _check_final(cfg, a2, b2)
        else:
            # pre-resample placement: with frames waiting, the reference's pre stage copies its buffer onto itself
            # (input == scratch, SURVEY F4 / App. B10: documented, not replicated), so the yardstick here is F5's meaning —
            # a fresh stream that begins with the waiting frames
            lead = x[2 * (n1 - waiting): 2 * n1]
            b2 = gpu.Chain(cfg, 0).process(np.concatenate([lead, x[2 * n1:]]))
            assert a2.size == b2.size and np.array_equal(a2.view(np.uint32), b2.view(np.uint32))
        fresh = gpu.Chain(cfg, 0).process(x[2 * n1:])
        assert fresh.size != a2.size or not np.array_equal(fresh, a2)
        g.restart()
        assert np.array_equal(g.process(x[2 * n1:]).view(np.uint32), fresh.view(np.uint32))


def test_in_chain_iq_optimizer_equals_function_level_passes(gpu, workloads):
    """SURVEY 8(f) rank 3: the optimiser inside the chain (sample-clocked gate, counter-based directions, passes on the
    device, factors applied from the next train) == the function-level pass (iq_correct_run_optimization, K6) applied by
    hand to the same probe blocks with the same directions.  cfg4's chain, unfused so that the pre-processor output the
    probes are cut from can be read back; then the fused path (probe blocks re-computed from the raw frames)."""
    import ctypes as C
    wl = workloads["cfg4"]
    cfg = wl.config
    chunk, rate = 16384, int(cfg.input_rate_hz)
    trains = [40, 45, 100]                                   # chunks per call; 500 ms = 73.2 chunks at 2.4 Msps
    raw = synth_numpy(wl, sum(trains) * chunk)
    seed = 1234
    g = gpu.Chain(cfg, 0, fused=0, record_taps=2, iq_optimize=1, iq_optimize_seed=seed, subtrain_frames=1 << 22)
    mag, phase = np.float32(cfg.iq_mag), np.float32(cfg.iq_phase)
    applied = [(float(mag), float(phase))]
    last_t, attempts, passes, pos = -1e18, 0, 0, 0
    for n_chunks in trains:
        lo, hi = pos * 2, (pos + n_chunks * chunk) * 2
        g.process(raw[lo:hi])
        tap0 = g.read_tap(0)                                 # the pre-processor output of THIS call
        for c in range(n_chunks):
            p0 = pos + c * chunk
            t = p0 / rate
            if (t - last_t) * 1000.0 >= 500.0:
                last_t = t
                blk = tap0[c * chunk:c * chunk + 1024]
                dirs = np.array([gpu.lib.iqgpu_iq_direction(seed, attempts, k) for k in range(50)], dtype=np.float32)
                m2, p2, _, rng_db = gpu.iq_optimize(blk, dirs, float(mag), float(phase))
                attempts += 1
                if rng_db >= 20.0:
                    mag, phase, passes = np.float32(m2), np.float32(p2), passes + 1
        pos += n_chunks * chunk
        gm, gp, gpasses, gattempts = g.iq_state()
        assert (gattempts, gpasses) == (attempts, passes)
        assert np.float32(gm) == mag and np.float32(gp) == phase, (gm, mag, gp, phase)
        applied.append((gm, gp))
    assert attempts == 3 and passes >= 1 and applied[-1] != applied[0]
    # fused front: same gate, same generator; the probe blocks come from a second evaluation of the pre-processor chain
    # (fp32 round-off in the DC state: a metric comparison may tip the other way once, i.e. one step of 0.05 * 1e-4)
    f = gpu.Chain(cfg, 0, fused=1, iq_optimize=1, iq_optimize_seed=seed, subtrain_frames=1 << 22)
    pos = 0
    for n_chunks in trains:
        f.process(raw[pos * 2:(pos + n_chunks * chunk) * 2])
        pos += n_chunks * chunk
    fm, fp_, fpasses, fattempts = f.iq_state()
    assert f.info().fused_front == 1 and (fattempts, fpasses) == (attempts, passes)
    assert abs(fm - float(mag)) <= 3.3e-5 and abs(fp_ - float(phase)) <= 3.3e-5
