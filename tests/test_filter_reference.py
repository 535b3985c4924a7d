"""The user filter (K3 time-domain FIR, K4 FFT block filter) against an exact float64 convolution, on every kernel path.

The other filter tests compare with the CPU oracle, itself fp32, under normwise bars; a tap read one sample late, a
wrong twiddle in one inner pass or a history sample lost at a call boundary can hide under those.  Here the reference is
y[n] = sum_k h[k] x[n-k] in complex128 with the chain's own taps (Chain.filter_taps) and the exact filter input, and
the bars follow from fp32 error analysis (u = 2^-24):

  * FIR, any fp32 summation order (FFMA2 included), per output and component:
        |yhat[n] - y[n]| <= gamma_K (|h| * |x|)[n],  gamma_K = K u / (1 - K u),  K = 2 ntaps_padded + 1,
    and, because that bound is loose for long filters, RMS(yhat - y) <= 4 u sqrt(K) RMS(|h| * |x|).
  * FIR on isolated impulses (+-1, +-j, powers of two, at least ntaps apart): every output is one exact product or an
    exact zero in any order, so the read-back is exact.
  * FFT block filter, per block b of n outputs with its 2n-sample window w_b:
        ||yhat_b - y_b||_2 <= 8 log2(2n) u ||w_b||_2 max_k |H64_k|,   H64 = float64 DFT of the zero-padded taps,
    the textbook bound of a forward + pointwise + inverse FFT whose twiddles are rounded and partly fp32 products.
  * integer outputs (the FIR's conversion epilogue): the conversion is monotone, so every component lies between
    convert(fp32(y - bound)) and convert(fp32(y + bound)), with the reference converter (sample_convert.c).
The reference's own rounding is covered by an absolute slack of 1e-12 of its scale.

How each path gets a known filter input:
  * pre-resample placement: no_resample, cf32 in, gain 1 -> the filter input is the caller's array;
  * post-resample placement, filter alone: a decimating configuration with stage_select = IQGPU_STAGE_FILTER designs
    the post-resample filter and runs only it on the caller's cf32 data;
  * the conversion epilogue and the DC fold exist only inside a full chain: a run with record_taps=1 (which turns both
    off) yields the exact filter input as tap 1, the run without it is checked against that input.

The CPU self-checks at the end show that honest fp32 arithmetic meets these bars and that the faults above fail them.
"""
import dataclasses
import math
import zlib

import numpy as np
import pytest
import scipy.fft
from scipy import signal

from iq_tool_b200.configs import (BYTES_PER_SAMPLE, FILTER_IMPL_FFT_ASYM, FILTER_IMPL_FFT_SYM, FILTER_IMPL_FIR_ASYM,
                                  FILTER_IMPL_FIR_SYM, FILTER_REQ_FFT, FILTER_REQ_FIR, FORMAT_CODES, NUMPY_DTYPE,
                                  STAGE_FILTER, ChainConfig, lowpass, pass_range)

U = 2.0 ** -24
REF_SLACK = 1e-12
FFT_BOUND_C = 8.0
FIR_TILE, FIR_TC, FIR_PARAM_FLOATS = 1024, 256, 4096   # kernels.cu: outputs per CTA, taps per chunk, parameter bank
FIR_VIA_FFT_TAPS, FIR_VIA_FFT_BLOCK = (512, 8192), 8192  # chain.cu: post-resample FIRs evaluated by overlap-save blocks
FFT_SMEM_MAX, FFT_V2_MIN = 16384, 64                     # fft_filter.cu: one-CTA transforms, radix-16 kernel from 64


# ---------------------------------------------------------------------------------------------
# the yardstick
# ---------------------------------------------------------------------------------------------
def gamma(k):
    return k * U / (1.0 - k * U)


def padded(ntaps):
    return (ntaps + 7) & ~7


def fir_k(ntaps):
    return 2 * padded(ntaps) + 1


def causal_conv(h, x, with_abs=True):
    """y[n] = sum_k h[k] x[n-k] for 0 <= n < len(x), zero before x[0], in complex128; with (|h| * |x|)[n]."""
    h = np.asarray(h).astype(np.complex128)
    x = np.asarray(x).astype(np.complex128)
    n = x.size
    direct = h.size * n <= 1e8
    y = (np.convolve(x, h) if direct else signal.fftconvolve(x, h))[:n]
    if not with_abs:
        return y, None
    ax, ah = np.abs(x), np.abs(h)
    a = np.convolve(ax, ah)[:n] if direct else np.maximum(signal.fftconvolve(ax, ah)[:n], 0.0)
    return y, a


def _ratio(err, bound):
    """err / bound elementwise, where a zero bound admits only a zero error."""
    err, bound = np.broadcast_arrays(np.asarray(err, dtype=np.float64), np.asarray(bound, dtype=np.float64))
    out = np.where(err > 0, np.inf, 0.0)
    np.divide(err, bound, out=out, where=bound > 0)
    return out


def fir_ratios(yg, y, a, ntaps):
    """(largest per-component error / rigorous bound, RMS error / statistical bar) of an FIR output."""
    e = np.asarray(yg).astype(np.complex128) - y
    bound = gamma(fir_k(ntaps)) * a + REF_SLACK * (float(a.max()) if a.size else 0.0)
    worst = float(max(_ratio(np.abs(e.real), bound).max(initial=0.0), _ratio(np.abs(e.imag), bound).max(initial=0.0)))
    bar = 4.0 * U * math.sqrt(fir_k(ntaps)) * math.sqrt(float(np.mean(a ** 2))) if a.size else 0.0
    rms = math.sqrt(float(np.mean(np.abs(e) ** 2))) if e.size else 0.0
    return worst, float(_ratio(rms, bar))


def assert_fir_bound(yg, h, x, label):
    y, a = causal_conv(h, x)
    assert yg.size == x.size
    worst, stat = fir_ratios(yg, y, a, h.size)
    print(f"[fir-bound] {label}: err/bound {worst:.3g}, rms/bar {stat:.3g}")
    assert worst <= 1.0, f"{label}: an output exceeds the fp32 bound ({worst:.3g}x)"
    assert stat <= 1.0, f"{label}: RMS error {stat:.3g}x the statistical bar"


def block_list(starts_ends, B):
    """[(first output, count)] of blocks of at most B outputs laid from each start up to its end."""
    out = []
    for s, e in starts_ends:
        for b in range(s, e, B):
            out.append((b, min(B, e - b)))
    return out


def fft_ratios(yg, y, x, h, B, blocks):
    """Per block: ||yhat_b - y_b|| / (8 log2(2B) u ||w_b|| max|H64|), w_b = x[s-B, s+B) (zero outside the stream)."""
    N = 2 * B
    hmax = float(np.abs(np.fft.fft(np.asarray(h).astype(np.complex128), N)).max())
    xz = np.concatenate([np.zeros(B), np.asarray(x).astype(np.complex128), np.zeros(B)])
    e = np.asarray(yg).astype(np.complex128) - y[: yg.size]
    r = np.empty(len(blocks))
    for i, (s, cnt) in enumerate(blocks):
        wn = float(np.linalg.norm(xz[s: s + N]))
        bound = (FFT_BOUND_C * math.log2(N) * U + REF_SLACK) * wn * hmax
        r[i] = _ratio(float(np.linalg.norm(e[s: s + cnt])), bound)
    return r


def assert_fft_bound(yg, y, x, h, B, blocks, label):
    r = fft_ratios(yg, y, x, h, B, blocks)
    worst = float(r.max(initial=0.0))
    print(f"[fft-bound] {label}: max err/bound {worst:.4g} over {r.size} blocks")
    assert worst <= 1.0, f"{label}: block {int(r.argmax())} exceeds the FFT error bound ({worst:.3g}x)"
    return worst


IMPULSE_VALUES = (1.0, -1.0, 1j, -1j, 2.0, -0.5j, 0.25, -4.0, 0.125j, -2j)


def impulse_stream(n, span):
    """Isolated impulses at least `span` apart: on the first and the last sample, and elsewhere at offsets 0, +1, -1,
    -255, -256, -257 from a multiple of the FIR tile, so that a tile's first output sees the impulse at lag 0, 1, 255,
    256 or 257 (the tap-chunk edges), or the impulse is a tile's second sample.  Returns (x complex64, positions)."""
    offs = (0, 1, -1, -(FIR_TC - 1), -FIR_TC, -(FIR_TC + 1))
    pos, k = [0], 0
    while True:
        lo, d = pos[-1] + span, offs[k % len(offs)]
        k += 1
        p = -(-(lo - d) // FIR_TILE) * FIR_TILE + d
        if p > n - 1 - span:
            break
        pos.append(p)
    pos.append(n - 1)
    x = np.zeros(n, dtype=np.complex64)
    x[pos] = [IMPULSE_VALUES[i % len(IMPULSE_VALUES)] for i in range(len(pos))]
    return x, pos


def impulse_response(x, pos, h):
    """The exact output of isolated impulses: v h[i] at p + i, zero elsewhere (complex128, exact in complex64)."""
    h = np.asarray(h).astype(np.complex128)
    y = np.zeros(x.size, dtype=np.complex128)
    for p in pos:
        m = min(h.size, x.size - p)
        y[p: p + m] = complex(x[p]) * h[:m]
    assert np.array_equal(y.astype(np.complex64).astype(np.complex128), y)
    return y


def impulse_calls(n, pos, span):
    """Call lengths that cut the impulse stream twice inside one response (it continues through the history into the
    next two calls, the middle one shorter than the filter), once right before an impulse (the first sample of a call)
    and once right after one (the last sample of a call)."""
    p1, p2, p3 = pos[1], pos[2], pos[3]
    cuts = sorted({p1 + max(1, span // 3), p1 + max(2, 2 * span // 3), p2, p3 + 1})
    cuts = [c for c in cuts if 0 < c < n]
    return list(np.diff([0] + cuts + [n]))


def noise(n, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    return ((rng.standard_normal(n) + 1j * rng.standard_normal(n)) * 0.2).astype(np.complex64)


def seed_of(label):
    return zlib.crc32(label.encode())


def call_bounds(calls):
    c = np.cumsum([0] + list(calls))
    return list(zip(c[:-1].tolist(), c[1:].tolist()))


# ---------------------------------------------------------------------------------------------
# driving the chain
# ---------------------------------------------------------------------------------------------
REAL = [lowpass(100e3)]
CPLX = [pass_range(50e3, 150e3)]


def pre_cfg(filters, taps, req, fft_size=0):
    """Pre-resample placement: the filter input is the caller's cf32 array."""
    return ChainConfig(input_format="cf32", output_format="cf32", input_rate_hz=1e6, target_rate_hz=1e6, no_resample=True,
                       filters=filters, filter_taps=taps, filter_type_request=req, filter_fft_size=fft_size)


def post_cfg(filters, taps, req, fft_size=0, rates=(2e6, 1e6)):
    """Post-resample placement, the filter alone on the caller's cf32 data."""
    return ChainConfig(input_format="cf32", output_format="cf32", input_rate_hz=rates[0], target_rate_hz=rates[1],
                       filters=filters, filter_taps=taps, filter_type_request=req, filter_fft_size=fft_size,
                       stage_select=STAGE_FILTER)


def run(gpu, cfg, x, calls=None, **opts):
    """One chain over x (one call, or the given call lengths): (output complex64, info after the last call, taps)."""
    g = gpu.Chain(cfg, 0, **opts)
    try:
        xf = np.ascontiguousarray(x, dtype=np.complex64).view(np.float32)
        if calls is None:
            out = g.process(xf)
        else:
            parts, pos = [], 0
            for m in calls:
                parts.append(g.process(xf[2 * pos: 2 * (pos + m)], chunk_frames=[m]))
                pos += m
            assert pos == x.size
            out = np.concatenate(parts)
        return out.view(np.complex64).copy(), g.info(), g.filter_taps()
    finally:
        g.close()


def fir_path(ntaps, cplx, post):
    """The FIR kernel a tap count reaches (launch_fir, chain.cu)."""
    if post and FIR_VIA_FFT_TAPS[0] <= ntaps <= FIR_VIA_FFT_TAPS[1]:
        return "fir_via_fft"
    return "param" if padded(ntaps) * (2 if cplx else 1) <= FIR_PARAM_FLOATS else "fir_kernel"


def assert_filter_info(info, h, impl, post, ntaps=None, block=0):
    assert info.filter_impl == impl
    assert info.filter_post_resample == int(post)
    assert info.filter_num_taps == h.size
    if ntaps is not None:
        assert h.size == ntaps
    assert info.filter_block_size == block


# ---------------------------------------------------------------------------------------------
# FIR, time domain: exact impulse read-back and the fp32 bound on noise
# ---------------------------------------------------------------------------------------------
AUTO_1K = "auto"      # an auto-designed 1 kHz low-pass behind a 744 187.5 sps resampler: ~10 900 taps
FIR_CASES = [("pre", REAL, t) for t in (3, 8, 9, 255, 256, 257, 263, 4096, 4097)] + \
            [("pre", CPLX, 2048), ("pre", CPLX, 2049), ("post", REAL, 511), ("post", REAL, 8193), ("post", REAL, AUTO_1K)]


def _fir_cfg(place, filters, taps):
    if taps == AUTO_1K:
        return post_cfg(filters=[lowpass(1e3)], taps=0, req=FILTER_REQ_FIR, rates=(2e6, 744187.5))
    return (pre_cfg if place == "pre" else post_cfg)(filters, taps, FILTER_REQ_FIR)


def _fir_id(c):
    place, filters, taps = c
    cplx = filters is CPLX
    path = "fir_kernel" if taps == AUTO_1K else fir_path(taps, cplx, place == "post")
    return f"{path}-{place}-{'complex' if cplx else 'real'}-{'auto1k' if taps == AUTO_1K else taps}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", FIR_CASES, ids=[_fir_id(c) for c in FIR_CASES])
def test_fir_time_domain_against_float64(case, gpu):
    """Isolated impulses read back exactly, in one call and cut across the response; white noise within the bound."""
    place, filters, taps = case
    label = _fir_id(case)
    cplx = filters is CPLX
    cfg = _fir_cfg(place, filters, taps)
    xn = noise(3 * 16384 + 77, seed_of(label))
    yn, info, h = run(gpu, cfg, xn)
    assert_filter_info(info, h, FILTER_IMPL_FIR_ASYM if cplx else FILTER_IMPL_FIR_SYM, place == "post",
                       None if taps == AUTO_1K else taps)
    path = fir_path(h.size, cplx, place == "post")
    assert label.startswith(path + "-")
    if taps == AUTO_1K:
        assert h.size > FIR_VIA_FFT_TAPS[1]
    assert_fir_bound(yn, h, xn, label)

    span = h.size
    xi, pos = impulse_stream(max(16 * span, 20000) + 5, span)
    want = impulse_response(xi, pos, h).astype(np.complex64)
    one, _, _ = run(gpu, cfg, xi)
    assert np.array_equal(one, want), f"{label}: impulse read-back differs at {np.flatnonzero(one != want)[:8]}"
    cut, _, _ = run(gpu, cfg, xi, calls=impulse_calls(xi.size, pos, span))
    assert np.array_equal(cut, want), f"{label}: impulse read-back across calls differs at {np.flatnonzero(cut != want)[:8]}"


# ---------------------------------------------------------------------------------------------
# FIR via FFT: post-resample FIRs of 512..8192 taps on the overlap-save kernel, B = 8192, last block zero-completed
# ---------------------------------------------------------------------------------------------
FIR_FFT_CASES = [(f, t) for f in (REAL, CPLX) for t in (511, 512, 8192, 8193)]


def _fir_fft_id(c):
    filters, taps = c
    return f"{fir_path(taps, filters is CPLX, True)}-post-{'complex' if filters is CPLX else 'real'}-{taps}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in FIR_FFT_CASES if fir_path(c[1], c[0] is CPLX, True) == "fir_via_fft"],
                         ids=[_fir_fft_id(c) for c in FIR_FFT_CASES if fir_path(c[1], c[0] is CPLX, True) == "fir_via_fft"])
def test_fir_via_fft_against_float64(case, gpu):
    """Blocks are laid from each call's first output (a call's last block is completed with zeros), so the bound is
    taken per call-aligned block; a stream length that is not a multiple of the block exercises the completion."""
    filters, taps = case
    label = _fir_fft_id(case)
    cfg = post_cfg(filters, taps, FILTER_REQ_FIR)
    B = FIR_VIA_FFT_BLOCK
    for kind in ("noise", "impulses"):
        if kind == "noise":
            x, pos = noise(3 * B + 1234, seed_of(label)), None
            cut = [5, B - 1, B, B + 1]
            cut.append(x.size - sum(cut))
        else:
            x, pos = impulse_stream(max(12 * taps, 3 * B) + 999, taps)
            cut = impulse_calls(x.size, pos, taps)
        assert x.size % B != 0
        for calls in (None, cut):
            yg, info, h = run(gpu, cfg, x, calls=calls)
            assert_filter_info(info, h, FILTER_IMPL_FIR_ASYM if filters is CPLX else FILTER_IMPL_FIR_SYM, True, taps)
            assert yg.size == x.size
            y = causal_conv(h, x, with_abs=False)[0] if pos is None else impulse_response(x, pos, h)
            blocks = block_list(call_bounds(calls if calls is not None else [x.size]), B)
            assert_fft_bound(yg, y, x, h, B, blocks, f"{label}-{kind}-{'one' if calls is None else 'cut'}")


# ---------------------------------------------------------------------------------------------
# every fir_param_kernel instantiation: real/complex taps x {cf32, cs16, cu8, cs8} x DC fold on/off, in a full chain
# ---------------------------------------------------------------------------------------------
def assert_int_between(out, y, bound, fmt, label):
    from oracle.loader import convert_from_cf32
    code = FORMAT_CODES[fmt]

    def conv(re, im):
        v = (re.astype(np.float32) + 1j * im.astype(np.float32)).astype(np.complex64)
        return convert_from_cf32("oracle", v, code, NUMPY_DTYPE[fmt], BYTES_PER_SAMPLE[fmt]).astype(np.int64)

    lo, hi = conv(y.real - bound, y.imag - bound), conv(y.real + bound, y.imag + bound)
    o = np.asarray(out).astype(np.int64)
    assert o.size == lo.size
    bad = np.flatnonzero((o < lo) | (o > hi))
    print(f"[int-bound] {label}: {o.size // 2} frames, {int((lo != hi).sum())} components with two admissible codes")
    assert bad.size == 0, f"{label}: {bad.size} components outside [convert(y - bound), convert(y + bound)], first {bad[:6]}"


@pytest.mark.gpu
@pytest.mark.parametrize("fold", [True, False], ids=["fold", "nofold"])
@pytest.mark.parametrize("fmt", ["cf32", "cs16", "cu8", "cs8"])
@pytest.mark.parametrize("cplx", [False, True], ids=["real", "complex"])
def test_fir_param_kernel_every_instantiation(cplx, fmt, fold, gpu, workloads, monkeypatch):
    """cfg2's chain (DC offset removed by the fused front, 255-tap FIR behind the resampler): the FIR adds the front's DC
    term while staging its tiles (fold) or finds it in memory (IQGPU_NO_DC_FOLD=1), and converts to the output format
    in its epilogue (cs16/cu8/cs8) or leaves cf32 to the post kernel.  A run with record_taps=1 turns both off and
    yields the exact filter input; both runs give the same bytes, and the output meets the bound against that input."""
    from iq_tool_b200.synth import synth_numpy
    wl = workloads["cfg2"]
    assert wl.dc != 0.0 and wl.config.dc_block
    filters = [pass_range(20e3, 180e3)] if cplx else wl.config.filters
    cfg = dataclasses.replace(wl.config, output_format=fmt, filters=filters)
    raw = synth_numpy(wl, (1 << 20) + 4321)
    if not fold:
        monkeypatch.setenv("IQGPU_NO_DC_FOLD", "1")
    g = gpu.Chain(cfg, 0, record_taps=1, subtrain_frames=1 << 18)
    try:
        plain = g.process(raw)
        x = g.read_tap(1)
    finally:
        g.close()
    g = gpu.Chain(cfg, 0, subtrain_frames=1 << 18)
    try:
        out = g.process(raw)
        info, h = g.info(), g.filter_taps()
    finally:
        g.close()
    label = f"{'complex' if cplx else 'real'}-{fmt}-{'fold' if fold else 'nofold'}"
    assert info.fused_front == 1
    assert_filter_info(info, h, FILTER_IMPL_FIR_ASYM if cplx else FILTER_IMPL_FIR_SYM, True, 255)
    assert fir_path(h.size, cplx, True) == "param"
    assert out.size == plain.size == 2 * x.size
    assert np.array_equal(out.view(np.uint8), plain.view(np.uint8)), f"{label}: fold/epilogue differ from the plain path"
    if fmt == "cf32":
        assert_fir_bound(out.view(np.complex64), h, x, label)
    else:
        y, a = causal_conv(h, x)
        bound = gamma(fir_k(h.size)) * a + REF_SLACK * float(a.max())
        assert_int_between(out, y, bound, fmt, label)


# ---------------------------------------------------------------------------------------------
# FFT block filter: every transform size and pass plan, taps = block + 1 and a short filter, pre and post placement
# ---------------------------------------------------------------------------------------------
def fft_family(N):
    if N < FFT_V2_MIN:
        return "fft_r4"
    if N <= FFT_SMEM_MAX:
        n16 = (int(math.log2(N)) - 2) // 4
        rest = int(math.log2(N)) - 2 - 4 * n16
        return f"fftfilt2_plan{n16}{rest // 2}{rest % 2}"
    return f"fft_split{int(math.log2(N)) - 14}"


FFT_SIZES = [1 << k for k in range(2, 22)]
FFT_CASES = []
for _N in FFT_SIZES:
    _B = _N // 2
    FFT_CASES.append((_N, _B + 1, REAL, "pre"))
    _short = max(3, _B // 16 + 1)
    if _short < _B + 1:
        FFT_CASES.append((_N, _short, REAL, "post"))
    if _N <= FFT_SMEM_MAX:
        FFT_CASES.append((_N, _B + 1, CPLX, "post" if (_N.bit_length() % 2) else "pre"))
FFT_CASES += [(8192, 4097, REAL, "post"), (1 << 18, (1 << 17) + 1, REAL, "post")]


def _fft_id(c):
    N, taps, filters, place = c
    return f"{fft_family(N)}-n{N}-{place}-{'complex' if filters is CPLX else 'real'}-{taps}"


def _fft_frames(B):
    return max(3 * B + B // 2 + 1, 3 * 4096 + 1)


_ONE_CTA_LAUNCHES = {}


def one_cta_launches(gpu, place):
    """kernel_launches of a call whose FFT filter is one 16384-point CTA transform (same placement)."""
    if place not in _ONE_CTA_LAUNCHES:
        B = FFT_SMEM_MAX // 2
        cfg = (pre_cfg if place == "pre" else post_cfg)(REAL, B + 1, FILTER_REQ_FFT, FFT_SMEM_MAX)
        _, info, _ = run(gpu, cfg, noise(3 * B + 5, 1))
        _ONE_CTA_LAUNCHES[place] = info.kernel_launches
    return _ONE_CTA_LAUNCHES[place]


@pytest.mark.gpu
@pytest.mark.parametrize("case", FFT_CASES, ids=[_fft_id(c) for c in FFT_CASES])
def test_fft_block_filter_against_float64(case, gpu):
    """Noise and isolated impulses, 3.5 blocks or more, within the per-block bound; the split path launches its global
    radix-2 stages (one per doubling beyond 16384 points, each way) plus gather and scatter."""
    N, taps, filters, place = case
    label = _fft_id(case)
    B = N // 2
    cplx = filters is CPLX
    cfg = (pre_cfg if place == "pre" else post_cfg)(filters, taps, FILTER_REQ_FFT, N)
    n = _fft_frames(B)
    x = noise(n, seed_of(label))
    yg, info, h = run(gpu, cfg, x)
    assert_filter_info(info, h, FILTER_IMPL_FFT_ASYM if cplx else FILTER_IMPL_FFT_SYM, place == "post", taps, B)
    assert yg.size == (n // B) * B and yg.size >= 3 * B
    if N > FFT_SMEM_MAX:
        assert info.kernel_launches == one_cta_launches(gpu, place) + 2 * (int(math.log2(N)) - 14) + 2
    blocks = block_list([(0, yg.size)], B)
    y = causal_conv(h, x, with_abs=False)[0]
    assert_fft_bound(yg, y, x, h, B, blocks, label + "-noise")
    xi, pos = impulse_stream(n, taps)
    yi, _, _ = run(gpu, cfg, xi)
    assert yi.size == yg.size
    assert_fft_bound(yi, impulse_response(xi, pos, h), xi, h, B, blocks, label + "-impulses")


# ---------------------------------------------------------------------------------------------
# stream edges: ragged calls, calls shorter than the filter, the history moved to the buffer front
# ---------------------------------------------------------------------------------------------
EDGE_SUBTRAIN = 16384
EDGE_CASES = [
    ("fir_kernel-pre-real-4097", "pre", REAL, 4097, FILTER_REQ_FIR, 0),
    ("param-post-real-511", "post", REAL, 511, FILTER_REQ_FIR, 0),
    ("fir_via_fft-post-complex-1001", "post", CPLX, 1001, FILTER_REQ_FIR, 0),
    ("fft_r4-n32-pre-real-17", "pre", REAL, 17, FILTER_REQ_FFT, 32),
    ("fftfilt2_plan211-n8192-post-complex-4097", "post", CPLX, 4097, FILTER_REQ_FFT, 8192),
    ("fft_split1-n32768-pre-real-16385", "pre", REAL, 16385, FILTER_REQ_FFT, 32768),
]


def edge_calls(n, span):
    """1, 7, 1023, 1024, 1025 frames, four calls shorter than the filter, then calls of up to one sub-train."""
    calls = [1, 7, 1023, 1024, 1025] + [max(1, span // 3)] * 4
    rest, k = n - sum(calls), 0
    while rest > 0:
        m = min(rest, (EDGE_SUBTRAIN, 9999)[k % 2])
        calls.append(m)
        rest -= m
        k += 1
    return calls


@pytest.mark.gpu
@pytest.mark.parametrize("case", EDGE_CASES, ids=[c[0] for c in EDGE_CASES])
def test_stream_edges_equal_one_call(case, gpu):
    """Ragged calls at a 16384-frame sub-train (the stream buffers move their history to the front several times)
    give the one-call output bit for bit, and both meet the reference.  The FIR-via-FFT path lays its blocks from each
    call's first output, so there the two differ in rounding and each meets the bound of its own blocks."""
    label, place, filters, taps, req, N = case
    cplx = filters is CPLX
    cfg = (pre_cfg if place == "pre" else post_cfg)(filters, taps, req, N)
    n = max(6 * taps, 12 * EDGE_SUBTRAIN) + 321
    calls = edge_calls(n, taps)
    assert min(calls[5:9]) < taps
    for kind in ("noise", "impulses"):
        if kind == "noise":
            x, pos = noise(n, seed_of(label)), None
        else:
            x, pos = impulse_stream(n, taps)
        one, info, h = run(gpu, cfg, x)
        many, info_m, _ = run(gpu, cfg, x, calls=calls, subtrain_frames=EDGE_SUBTRAIN)
        fft = req == FILTER_REQ_FFT
        impl = (FILTER_IMPL_FFT_ASYM if cplx else FILTER_IMPL_FFT_SYM) if fft else \
            (FILTER_IMPL_FIR_ASYM if cplx else FILTER_IMPL_FIR_SYM)
        assert_filter_info(info, h, impl, place == "post", taps, N // 2 if fft else 0)
        assert one.size == many.size
        via_fft = not fft and fir_path(taps, cplx, place == "post") == "fir_via_fft"
        assert label.startswith(fft_family(N) if fft else fir_path(taps, cplx, place == "post"))
        if not via_fft:
            assert np.array_equal(one.view(np.uint32), many.view(np.uint32)), f"{label}-{kind}: ragged calls differ"
        tag = f"{label}-{kind}"
        if fft:
            B = N // 2
            y = causal_conv(h, x, with_abs=False)[0] if pos is None else impulse_response(x, pos, h)
            assert_fft_bound(one, y, x, h, B, block_list([(0, one.size)], B), tag)
        elif via_fft:
            B = FIR_VIA_FFT_BLOCK
            y = causal_conv(h, x, with_abs=False)[0] if pos is None else impulse_response(x, pos, h)
            assert_fft_bound(one, y, x, h, B, block_list([(0, n)], B), tag + "-one")
            assert_fft_bound(many, y, x, h, B, block_list(call_bounds(calls), B), tag + "-cut")
        elif pos is None:
            assert_fir_bound(many, h, x, tag)
        else:
            assert np.array_equal(many, impulse_response(x, pos, h).astype(np.complex64)), f"{tag}: impulse read-back"


# ---------------------------------------------------------------------------------------------
# CPU self-checks of the yardstick: honest fp32 arithmetic meets it, the faults it is meant to catch fail it
# ---------------------------------------------------------------------------------------------
def kaiser_lowpass(ntaps, fc, beta=5.653):
    """A Kaiser-window low-pass (60 dB), unit DC gain."""
    t = np.arange(ntaps) - (ntaps - 1) / 2.0
    h = np.sinc(2.0 * fc * t) * np.kaiser(ntaps, beta)
    return h / h.sum()


def f32_conv(h, x):
    return np.convolve(np.asarray(x, dtype=np.complex64), np.asarray(h, dtype=np.complex64))[: len(x)]


def _taps(ntaps, cplx):
    h = kaiser_lowpass(ntaps, 0.05)
    if cplx:
        h = h * np.exp(2j * np.pi * 0.1 * np.arange(ntaps))
    return h.astype(np.complex64)


@pytest.mark.parametrize("ntaps,cplx", [(3, False), (255, False), (301, True), (4097, False)])
def test_float32_convolution_meets_the_fir_bound(ntaps, cplx):
    h = _taps(ntaps, cplx)
    x = noise(20000, ntaps)
    y, a = causal_conv(h, x)
    worst, stat = fir_ratios(f32_conv(h, x), y, a, ntaps)
    assert 0.0 < worst <= 1.0 and stat <= 1.0
    xi, pos = impulse_stream(max(16 * ntaps, 20000), ntaps)
    assert np.array_equal(f32_conv(h, xi), impulse_response(xi, pos, h).astype(np.complex64))


def test_a_dropped_tap_or_history_sample_fails_the_impulse_check():
    ntaps = 4097
    h = _taps(ntaps, False)
    xi, pos = impulse_stream(20 * ntaps, ntaps)
    want = impulse_response(xi, pos, h).astype(np.complex64)
    for k in (0, ntaps // 2, ntaps - 1):
        hd = h.copy()
        hd[k] = 0
        assert not np.array_equal(f32_conv(hd, xi), want)
    # a call boundary right behind an impulse, and the next call misses that sample in its history
    c = pos[2] + 1
    lost = xi.copy()
    lost[c - 1] = 0
    y = np.concatenate([f32_conv(h, xi)[:c], f32_conv(h, lost)[c:]])
    assert not np.array_equal(y, want)


def test_the_statistical_bar_catches_a_mid_filter_tap_but_not_a_kaiser_tail_tap():
    ntaps = 4097
    h = _taps(ntaps, False)
    x = noise(30000, 7)
    y, a = causal_conv(h, x)
    mid, tail = h.copy(), h.copy()
    mid[ntaps // 2 + 3] = 0
    tail[ntaps - 1] = 0
    assert fir_ratios(f32_conv(mid, x), y, a, ntaps)[1] > 1.0
    assert fir_ratios(f32_conv(tail, x), y, a, ntaps)[1] <= 1.0       # below the bar ...
    xi, pos = impulse_stream(20 * ntaps, ntaps)
    assert not np.array_equal(f32_conv(tail, xi), impulse_response(xi, pos, h).astype(np.complex64))   # ... not below B


def f32_overlap_save(h, x, B, H=None):
    """Overlap-save in complex64 (scipy.fft computes single precision in single precision): whole blocks only."""
    N = 2 * B
    if H is None:
        H = scipy.fft.fft(np.asarray(h, dtype=np.complex64), N)
    xz = np.concatenate([np.zeros(B, dtype=np.complex64), np.asarray(x, dtype=np.complex64)])
    nb = x.size // B
    w = np.stack([xz[b * B: b * B + N] for b in range(nb)])
    Y = scipy.fft.ifft(scipy.fft.fft(w, axis=1) * H[None, :], axis=1)
    assert Y.dtype == np.complex64
    return Y[:, B:].reshape(-1)


def test_float32_overlap_save_meets_the_fft_bound_and_a_rotated_bin_fails_it():
    B = 512
    h = _taps(B + 1, False)
    x = noise(9 * B + 17, 11)
    y = causal_conv(h, x, with_abs=False)[0]
    blocks = block_list([(0, 9 * B)], B)
    good = fft_ratios(f32_overlap_save(h, x, B), y, x, h, B, blocks)
    assert 0.0 < good.max() <= 1.0
    H = scipy.fft.fft(h, 2 * B)
    k = int(np.argmax(np.abs(H)))                  # a passband bin
    H[k] *= np.complex64(np.exp(2j * np.pi / (2 * B)))
    assert fft_ratios(f32_overlap_save(h, x, B, H), y, x, h, B, blocks).max() > 1.0


def test_impulse_layout_reaches_tile_and_chunk_edges():
    """The impulses sit on the first and last sample and at every tile offset the layout promises, at least span apart."""
    for span in (3, 255, 4097):
        n = max(16 * span, 20000) + 5
        x, pos = impulse_stream(n, span)
        assert pos[0] == 0 and pos[-1] == n - 1 and min(np.diff(pos)) >= span
        offs = {((p + FIR_TC + 1) % FIR_TILE) - FIR_TC - 1 for p in pos[1:-1]}
        assert {0, 1, -1, -(FIR_TC - 1), -FIR_TC, -(FIR_TC + 1)} <= offs
        calls = impulse_calls(n, pos, span)
        assert sum(calls) == n and min(calls) >= 1 and len(calls) == 5
