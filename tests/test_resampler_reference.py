"""The resampling front (K2: halfband cascade + 256-arm polyphase stage, fused front and stage kernels) against an exact
float64 reference, elementwise, at stream positions from 0 up to the 2^62 ceiling (include/iqgpu.h).

The other resampler tests compare with the CPU oracle (itself fp32) under normwise bars, or the fused front with the stage
kernels bit for bit; both share the host's design and bookkeeping, and a normwise bar over many outputs lets one wrong
output through.  Here every output is held to a reference computed in Python integers (positions) and complex128 (values)
from the chain's own taps (Chain.halfband_taps, Chain.arb_taps, bank layout of design.cpp), with frames before the seek
position read as zeros (seek resets the history):

  * position model: halfband depth d (design stage g = S-1-d) maps stage-input index i to output k with
        y[k] = (sum_{j<2m} h1[j] u[2(k-2m+1+j)] + u[2(k-m)+1]) * scale,   scale = zeta on the last stage, else 1,
    outputs k in [P >> (d+1), (P+n) >> (d+1)); the polyphase stage makes the outputs o in [R(P), R(P+n)),
    R(N) = ceil((N >> S) 2^24 / step), with P(o) = o step, k(o) = P >> 24, row(o) = (P >> 16) & 255, all exact integers.
    Interpolation runs the polyphase stage first (on the input stream), then halfband interpolators
    y[2k] = x[k-m], y[2k+1] = sum_{j<2m} h1[j] x[k-2m+1+j].
  * bar, rigorous and elementwise (u = 2^-24, gamma_K = K u / (1 - K u)), propagated stage by stage in float64:
        A_s = |H_s|(A_{s-1}),   E_s = |H_s|(E_{s-1}) + gamma_{K_s} |H_s|(A_{s-1} + E_{s-1}),
    K_s = 2m + 1 per halfband output (2m products and the centre term; zeta is a power of two), 14 per polyphase output;
    every output component must satisfy |yhat - y| <= E + 1e-12 max(A).  A_0 = |x|; E_0 = 0 when the kernel sees the
    caller's cf32 samples, and 4u|x| where the fused front forms the samples itself (conversion and NCO product rounded
    in its own order: two products and a sum, gamma_2 (|x.re| + |x.im|) <= 4u|x|).  A statistical bar,
    RMS(yhat - y) <= RMS(E) / 4, catches errors the loose rigorous bound hides.
  * input: the pre-processed stream is restated in fp32 (conversion as load_frame does it, then the LUT-NCO mix in the
    kernel's order, from the phase (P + i) dtheta mod 2^32 and the host libm's sinf table) and pinned bit for bit
    against tap 0 at 0, past 2^32, past 2^(40+S) and near 2^62; the reference is fed with that restatement.
  * DC blocker: the reference runs it in exact arithmetic, y[n] = x[n] - a v[n-1], v[n] = x[n] + c v[n-1], v = 0 before
    P, with the chain's fp32 pole c and a = 1 - c.  The kernels differ from it only through their state v, which every
    output sees through one product a v.  In either mode the fp32 arithmetic that forms v for a frame (a lane's
    recurrence over its 4 or 16 frames, the 5-step shuffle scan of the row or tick, the fold into the double carry and
    its conversion, the product with a and the subtraction) rounds at most 48 times along any path, each time relative
    to a sum of terms c^j |x|, so |v - vhat| a <= gamma_48 a V[n-1], V the same recurrence over |x|.  The local mode
    adds its closed-form correction through c_out (double, rounded to fp32), __expf (2^-22 relative), the fp32 row
    gain G and two products: at most (2^-22 + gamma_4) of a term whose cascade image is bounded by that of a V.  So
    E_0 += (gamma_48 + 2^-20) a V, and every output (or, ahead of the FIR, every staged sample) gets u (A + E) for the
    correction's own addition.  On the tested signals (DC offset 0.09, full-scale noise) that allowance is below 2e-7
    at the input, four orders below the ~1e-3 of a wrong row or pairing; the local mode with the FIR's fold is checked
    through the FIR, y = h * x with the FIR's own gamma_{2 padded + 1} term.
  * impulses, exact (no tolerance): an impulse at an odd stage-input index passes a halfband decimator only through its
    centre tap, y = (x + 0) scale, exact; positions are chosen odd at every depth, so the impulse reaches the polyphase
    stage as one known sample at a known index K, every output whose 14-tap window covers K is the single product
    fp32(bank[row(o)][K - k(o) + 13] v zeta), every other output is exactly zero.  A noise call runs first through the
    same chain, so an output left unwritten shows as stale data.  This pins pairing parity, centre delay, row and output
    index at every position tested.
  * translation invariance, bit for bit: full chains (local DC with the FIR's DC fold, table DC behind an NCO, digital
    AGC, post shift) seeked to P and to P + j T, T = 5 * 2^36 frames (a multiple of the polyphase phase period of
    rate_arb = 0.8, step = 5 * 2^22, of 2^32 / gcd with any NCO increment before and after the resampler, and of every
    tick, super-tick, stretch and run length of the fused front), must give the same bytes and chunk counts: the digital
    AGC and the post shift, which the elementwise reference does not model, and the DC paths once more.

The CPU part shows that honest fp32 arithmetic meets the bar, that the faults above (row +-1, a pair one sample late, a
dropped tap, output index +1, step phase off by 2^16, zeta off by 2^-20) fail it, and emulates in uint64 the kernels'
position arithmetic of the parent formulas (o * step and (o * step >> 24) << S, wrapping from polyphase input 2^40) and
the fixed ones (relative to a 128-bit base per launch) at the tested positions.
"""
import ctypes
import ctypes.util
import math
import zlib

import numpy as np
import pytest

from iq_tool_b200.configs import ChainConfig

U = 2.0 ** -24
REF_SLACK = 1e-12
MAX_POS = 1 << 62
T_SHIFT = 5 << 36
IMPULSE_VALUES = (1.0, -1.0, 1j, -1j, 0.5, -0.5j, 0.25, -1.0, 0.125j, -0.5)


def gamma(k):
    return k * U / (1.0 - k * U)


def seed_of(label):
    return zlib.crc32(label.encode())


def noise(n, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    return ((rng.standard_normal(n) + 1j * rng.standard_normal(n)) * 0.2).astype(np.complex64)


# ---------------------------------------------------------------------------------------------
# the design as the chain reports it
# ---------------------------------------------------------------------------------------------
class Design:
    """Taps and positions of one resampler (decimating or interpolating)."""

    def __init__(self, chain):
        info = chain.info()
        self.S = int(info.num_halfband)
        self.step = int(info.arb_step)
        self.interp = bool(info.is_interp)
        self.m = [int(info.halfband_m[g]) for g in range(self.S)]           # by design index
        self.h1 = []
        for g in range(self.S):
            h = chain.halfband_taps(g).astype(np.float64)
            m = self.m[g]
            assert h.size == 4 * m + 1
            self.h1.append(np.array([h[4 * m - 1 - 2 * j] for j in range(2 * m)]))
        arb = chain.arb_taps().astype(np.float64)
        assert arb.size == 256 * 14
        self.bank = np.empty((256, 14))
        for i in range(256):
            for k in range(14):
                self.bank[i, 13 - k] = arb[i + 256 * k]
        self.zeta = 2.0 ** -self.S

    def R(self, n):
        """resampler outputs after n input frames (design.cpp resampler_outputs_after), exact integers"""
        if self.interp:
            return (((n << 24) + self.step - 1) // self.step) << self.S
        return (((n >> self.S) << 24) + self.step - 1) // self.step

    def depth_m(self, d):
        return self.m[self.S - 1 - d]


def _at(stream, a0, idx):
    """stream[idx - a0] for an integer index array, zero before a0"""
    rel = idx - a0
    out = np.zeros(rel.shape, dtype=stream.dtype)
    ok = (rel >= 0) & (rel < stream.size)
    out[ok] = stream[rel[ok]]
    return out


def _hb_decim(u, a0, h1, m, k0, k1, scale, dtype=np.complex128):
    k = np.arange(k0, k1, dtype=np.int64)
    acc = np.zeros(k.size, dtype=dtype)
    single = dtype is np.complex64
    for j in range(2 * m):
        hj = np.float32(h1[j]) if single else h1[j]
        acc = acc + hj * _at(u, a0, 2 * (k - 2 * m + 1 + j))
    acc = _at(u, a0, 2 * (k - m) + 1) + acc
    return acc * (np.float32(scale) if single else scale)


def _hb_interp(x, a0, h1, m, dtype=np.complex128):
    k = np.arange(a0, a0 + x.size, dtype=np.int64)
    acc = np.zeros(k.size, dtype=dtype)
    for j in range(2 * m):
        hj = np.float32(h1[j]) if dtype is np.complex64 else h1[j]
        acc = acc + hj * _at(x, a0, k - 2 * m + 1 + j)
    y = np.empty(2 * k.size, dtype=dtype)
    y[0::2] = _at(x, a0, k - m)
    y[1::2] = acc
    return y


def _arb_positions(o0, o1, step, phase_off=0):
    P = np.arange(o0, o1, dtype=object) * step + phase_off
    k = np.array([int(p >> 24) for p in P], dtype=object)
    row = np.array([int((p >> 16) & 255) for p in P], dtype=np.int64)
    return k, row


def _arb(x, a0, bank, k, row, dtype=np.complex128):
    """y = sum_i bank[row][i] x[k-13+i], k as Python ints (absolute), a0 the absolute index of x[0]"""
    krel = np.array([int(v - a0) for v in k], dtype=np.int64) if k.size else np.zeros(0, dtype=np.int64)
    acc = np.zeros(krel.size, dtype=dtype)
    for i in range(14):
        h = bank[row, i].astype(np.float32) if dtype is np.complex64 else bank[row, i]
        acc = acc + h * _at(x, 0, krel - 13 + i)
    return acc


class Mut:
    """Faults the reference can be given, to show that the checks catch them (CPU self-check)."""
    NONE, ROW, PAIR_LATE, DROP_TAP, OUT_SHIFT, STEP_PHASE, ZETA = range(7)


def reference(D, x, P, mut=Mut.NONE, e0=0.0, e_in=None):
    """(O0, y, A, E, K) of a call of len(x) frames from position P: exact value, magnitude and error bound per output.
    The kernel's input may differ from x by e0 |x| + e_in per frame."""
    n = x.size
    x = x.astype(np.complex128)
    A = np.abs(x)
    E = e0 * A + (0.0 if e_in is None else e_in)
    if not D.interp:
        u, a0 = x, P
        for d in range(D.S):
            g = D.S - 1 - d
            m = D.m[g]
            h1 = D.h1[g].copy()
            if mut == Mut.DROP_TAP and d == 0:
                h1[m - 1] = 0.0
            scale = D.zeta if d + 1 == D.S else 1.0
            if mut == Mut.ZETA and d + 1 == D.S:
                scale *= 1.0 + 2.0 ** -20
            k0, k1 = P >> (d + 1), (P + n) >> (d + 1)
            kk0 = k0 + (1 if mut == Mut.PAIR_LATE and d == 0 else 0)
            y = _hb_decim(u, a0 - (kk0 - k0) * 2, h1, m, k0, k1, scale)
            Aa = _hb_decim(A, a0, np.abs(h1), m, k0, k1, abs(scale)).real
            Ea = _hb_decim(E, a0, np.abs(h1), m, k0, k1, abs(scale)).real
            Eb = _hb_decim(A + E, a0, np.abs(h1), m, k0, k1, abs(scale)).real
            u, A, E, a0 = y, Aa, Ea + gamma(2 * m + 1) * Eb, k0
        O0, O1 = D.R(P), D.R(P + n)
        k, row = _arb_positions(O0, O1, D.step, (1 << 16) if mut == Mut.STEP_PHASE else 0)
        if mut == Mut.ROW:
            row = (row + 1) & 255
        bank = D.bank.copy()
        if mut == Mut.DROP_TAP:
            bank[:, 13] = 0.0
        y = _arb(u, a0, bank, k, row)
        Aa = _arb(A.astype(np.complex128), a0, np.abs(D.bank), k, row).real
        Ea = _arb(E.astype(np.complex128), a0, np.abs(D.bank), k, row).real
        Eb = _arb((A + E).astype(np.complex128), a0, np.abs(D.bank), k, row).real
        E = Ea + gamma(14) * Eb
        if mut == Mut.OUT_SHIFT:
            y = np.concatenate([[0.0], y[:-1]])
        return O0, y, Aa, E, [14] + [2 * D.m[D.S - 1 - d] + 1 for d in range(D.S)]
    # interpolation: polyphase stage on the input stream, then halfband interpolators in design order
    Oa0 = ((P << 24) + D.step - 1) // D.step
    Oa1 = (((P + n) << 24) + D.step - 1) // D.step
    k, row = _arb_positions(Oa0, Oa1, D.step, (1 << 16) if mut == Mut.STEP_PHASE else 0)
    if mut == Mut.ROW:
        row = (row + 1) & 255
    y = _arb(x, P, D.bank, k, row)
    absb = np.abs(D.bank)
    Aa = _arb(A.astype(np.complex128), P, absb, k, row).real
    E = _arb(E.astype(np.complex128), P, absb, k, row).real + gamma(14) * _arb((A + E).astype(np.complex128), P, absb, k, row).real
    A, a0 = Aa, Oa0
    for s in range(D.S):
        m, h1 = D.m[s], D.h1[s]
        yn = _hb_interp(y, a0, h1, m)
        An = _hb_interp(A.astype(np.complex128), a0, np.abs(h1), m).real
        En = _hb_interp(E.astype(np.complex128), a0, np.abs(h1), m).real
        Eb = _hb_interp((A + E).astype(np.complex128), a0, np.abs(h1), m).real
        En[1::2] += gamma(2 * m + 1) * Eb[1::2]
        y, A, E, a0 = yn, An, En, 2 * a0
    if mut == Mut.OUT_SHIFT:
        y = np.concatenate([[0.0], y[:-1]])
    return a0, y, A, E, [14] + [2 * m + 1 for m in D.m]


def bound_ratios(yg, y, A, E):
    """(largest per-component error / rigorous bound, RMS error / statistical bar)"""
    yg = np.asarray(yg).astype(np.complex128)
    assert yg.size == y.size, (yg.size, y.size)
    e = yg - y
    b = E + REF_SLACK * (float(A.max()) if A.size else 0.0)
    worst = 0.0
    for comp in (np.abs(e.real), np.abs(e.imag)):
        r = np.where(comp > 0, np.inf, 0.0)
        np.divide(comp, b, out=r, where=b > 0)
        worst = max(worst, float(r.max(initial=0.0)))
    bar = 0.25 * math.sqrt(float(np.mean(E ** 2))) if E.size else 0.0
    rms = math.sqrt(float(np.mean(np.abs(e) ** 2))) if e.size else 0.0
    return worst, (rms / bar if bar > 0 else (0.0 if rms == 0 else math.inf))


# ---------------------------------------------------------------------------------------------
# impulses
# ---------------------------------------------------------------------------------------------
def impulse_path(D, p):
    """the decimated index K the impulse at raw position p reaches through centre taps only, or None when p is even at
    some depth (then it would also meet the stage's other taps)"""
    for d in range(D.S):
        if p % 2 == 0:
            return None
        p = (p - 1) // 2 + D.depth_m(d)
    return p


def impulse_positions(D, P, n):
    """raw offsets (from P) of impulses whose polyphase windows do not overlap: decimated indices at least 16 apart"""
    offs, lastK, i = [], None, 1
    span = 1 << D.S
    while i < n - 64 * span:
        K = impulse_path(D, P + i)
        if K is not None and (lastK is None or K - lastK >= 16) and K - 30 > (P >> D.S):
            offs.append(i)
            lastK = K
            i += 16 * span
        else:
            i += 1
    return offs


def impulse_expect(D, P, n, offs, vals, mut=Mut.NONE):
    """exact complex64 output of the decimating resampler for the impulses vals at P + offs"""
    O0, O1 = D.R(P), D.R(P + n)
    k, row = _arb_positions(O0, O1, D.step, (1 << 16) if mut == Mut.STEP_PHASE else 0)
    if mut == Mut.ROW:
        row = (row + 1) & 255
    kk = np.array([int(v) for v in k], dtype=object)
    y = np.zeros(O1 - O0, dtype=np.complex64)
    zeta = np.float32(D.zeta * ((1.0 + 2.0 ** -20) if mut == Mut.ZETA else 1.0))
    bank32 = D.bank.astype(np.float32)
    if mut == Mut.DROP_TAP:
        bank32[:, 13] = 0
    krel = np.array([int(v) - int(kk[0]) for v in kk], dtype=np.int64) if kk.size else np.zeros(0, dtype=np.int64)
    for off, v in zip(offs, vals):
        K = impulse_path(D, P + off) + (1 if mut == Mut.PAIR_LATE else 0) - (int(kk[0]) if kk.size else 0)
        vz = np.complex64(v) * zeta
        lo, hi = np.searchsorted(krel, K), np.searchsorted(krel, K + 14)      # outputs with k(o) in [K, K + 13]
        for idx in range(lo, hi):
            h = bank32[row[idx], K - krel[idx] + 13]
            y[idx] = np.complex64(complex(np.float32(h * vz.real), np.float32(h * vz.imag)))
    if mut == Mut.OUT_SHIFT:
        y = np.concatenate([[0], y[:-1]]).astype(np.complex64)
    return y


def fp32_cascade(D, x, P):
    """an honest fp32 evaluation of the decimating cascade (products and sums rounded one by one)"""
    n = x.size
    u, a0 = x.astype(np.complex64), P
    for d in range(D.S):
        g = D.S - 1 - d
        m = D.m[g]
        k0, k1 = P >> (d + 1), (P + n) >> (d + 1)
        u, a0 = _hb_decim(u, a0, D.h1[g], m, k0, k1, D.zeta if d + 1 == D.S else 1.0, np.complex64), k0
    k, row = _arb_positions(D.R(P), D.R(P + n), D.step)
    return _arb(u, a0, D.bank, k, row, np.complex64)


# ---------------------------------------------------------------------------------------------
# chains
# ---------------------------------------------------------------------------------------------
IN_RATE = 1_024_000


def decim_cfg(S, rate_arb, fmt="cf32"):
    return ChainConfig(input_format=fmt, output_format="cf32", input_rate_hz=IN_RATE << S,
                       target_rate_hz=IN_RATE * rate_arb)


def interp_cfg(ratio):
    return ChainConfig(input_format="cf32", output_format="cf32", input_rate_hz=IN_RATE, target_rate_hz=IN_RATE * ratio)


def call_frames(S):
    return 1 << max(15, S + 8)


def positions(S, n, interp_ratio=None):
    """item-6 positions: 0, a small odd offset, calls straddling 2^31 and 2^32 raw frames, 2^(39+S), 2^(40+S), 2^(41+S)
    (polyphase input 2^39, 2^40, 2^41), 2^52 and the ceiling"""
    half = n // 2
    top = MAX_POS if interp_ratio is None else int(MAX_POS / interp_ratio / 1.01)
    ps = [0, 3, (1 << 31) - half + 1, (1 << 32) - half - 7]
    for e in (39, 40, 41):
        if e + S < 61:
            ps.append((1 << (e + S)) - half - 5)
    ps += [(1 << 52) + 7, top - n - 1 - (1 << S)]
    return ps


def _raw_cf32(x):
    return np.ascontiguousarray(x.astype(np.complex64)).view(np.float32)


def run(chain, P, x, chunk=None):
    chain.seek(P)
    raw = _raw_cf32(x)
    out, counts = chain.process(raw, chunk_frames=chunk, return_chunk_counts=True)
    return out.view(np.complex64), counts


def closed_form_counts(D, P, chunks):
    c = np.cumsum([0] + list(chunks))
    return [D.R(P + int(b)) - D.R(P + int(a)) for a, b in zip(c[:-1], c[1:])]


# ---------------------------------------------------------------------------------------------
# CPU part: the yardstick and the position arithmetic
# ---------------------------------------------------------------------------------------------
def _plan(cfg):
    from iq_tool_b200 import gpu
    return gpu.Chain(cfg, -1)


SELF_CASES = [(0, 0.7), (1, 0.55), (2, 0.8), (4, 0.66)]


@pytest.mark.parametrize("S,rate", SELF_CASES)
def test_fp32_cascade_meets_the_bound(S, rate):
    D = Design(_plan(decim_cfg(S, rate)))
    n = 4096 << S
    P = (1 << (40 + S)) - n // 2 - 5
    x = noise(n, seed_of(f"self{S}"))
    O0, y, A, E, _ = reference(D, x, P)
    yg = fp32_cascade(D, x, P)
    worst, stat = bound_ratios(yg, y, A, E)
    print(f"[resampler-bound] fp32 cascade S={S} r={rate}: err/bound {worst:.3g}, rms/bar {stat:.3g}")
    assert worst <= 1.0 and stat <= 1.0
    assert worst < 0.25, "the bound should leave room for other summation orders"


@pytest.mark.parametrize("mut", ["ROW", "PAIR_LATE", "DROP_TAP", "OUT_SHIFT", "STEP_PHASE", "ZETA"])
@pytest.mark.parametrize("S", [1, 4])
def test_reference_faults_fail_the_checks(S, mut):
    D = Design(_plan(decim_cfg(S, 0.7)))
    n = 4096 << S
    P = (1 << 32) - n // 2 + 1
    mu = getattr(Mut, mut)
    x = noise(n, seed_of(f"mut{S}"))
    _, y, A, E, _ = reference(D, x, P, mut=mu)
    worst, stat = bound_ratios(fp32_cascade(D, x, P), y, A, E)
    offs = impulse_positions(D, P, n)
    vals = [IMPULSE_VALUES[i % len(IMPULSE_VALUES)] for i in range(len(offs))]
    xi = np.zeros(n, dtype=np.complex64)
    xi[offs] = vals
    honest = fp32_cascade(D, xi, P)
    assert np.array_equal(honest, impulse_expect(D, P, n, offs, vals)), "the exact impulse read-back must hold for fp32"
    impulse_caught = not np.array_equal(honest, impulse_expect(D, P, n, offs, vals, mut=mu))
    print(f"[mutation] S={S} {mut}: err/bound {worst:.3g}, impulse read-back differs: {impulse_caught}")
    assert worst > 1.0 or stat > 1.0 or impulse_caught


# ---- position arithmetic of the kernels, emulated in uint64 ----
def _u64(v):
    return np.uint64(v & ((1 << 64) - 1))


def parent_sites(o, step, S, O0):
    """the parent's formulas, with uint64 wrap-around: polyphase k, quad steps e1..e3, DC fold frame"""
    with np.errstate(over="ignore"):
        P = np.uint64(o) * np.uint64(step)
        k = int(P >> np.uint64(24))
        steps = [int((P + np.uint64(q * step)) >> np.uint64(24)) - k for q in (1, 2, 3)]
    return k, steps, k << S


def fixed_sites(o, step, S, O0):
    """the fixed formulas: relative to the launch's 128-bit base (kernels.hpp ArbBase)"""
    Pb = O0 * step
    k_base, p_base = Pb >> 24, _u64(Pb) & np.uint64(~0xffffff & ((1 << 64) - 1))
    with np.errstate(over="ignore"):
        Dp = np.uint64(o) * np.uint64(step) - p_base
        k = k_base + int(Dp >> np.uint64(24))
        steps = [int((Dp + np.uint64(q * step)) >> np.uint64(24)) - int(Dp >> np.uint64(24)) for q in (1, 2, 3)]
    return k, steps, k << S


def parent_o_cur(k_emit, step):
    with np.errstate(over="ignore"):
        return int((np.uint64(k_emit) << np.uint64(24)) + np.uint64(step - 1)) // step


def fixed_o_cur(k_emit, step, O0):
    Pb = O0 * step
    D = ((k_emit - (Pb >> 24)) << 24) - (Pb & 0xffffff)
    return O0 + (-((-D) // step) if D < 0 else (D + step - 1) // step)


@pytest.mark.parametrize("S,rate", [(0, 0.8), (1, 0.7), (4, 0.8), (6, 0.55)])
def test_position_arithmetic_emulation(S, rate):
    """Where the parent's uint64 formulas leave the exact integers, and that the fixed ones never do.  Decides what may run
    on a GPU: the parent's w2_dc_correct_kernel skips w <= 0, so its wrapped fold frames drop the DC term (no read outside
    corr[]), and its fused front leaves the outputs past the wrap unwritten."""
    D = Design(_plan(decim_cfg(S, rate)))
    n = call_frames(S)
    for P in positions(S, n):
        O0, O1 = D.R(P), D.R(P + n)
        bad_parent = 0
        for o in sorted({O0, O0 + 1, (O0 + O1) // 2, O1 - 1} | {o for o in range(O0, O1) if (o * D.step) >> 64 != ((o + 3) * D.step) >> 64}):
            exact_k = (o * D.step) >> 24
            exact_steps = [(((o + q) * D.step) >> 24) - exact_k for q in (1, 2, 3)]
            k, st, nk = fixed_sites(o, D.step, S, O0)
            assert (k, st, nk) == (exact_k, exact_steps, exact_k << S), (P, o)
            pk, pst, pnk = parent_sites(o, D.step, S, O0)
            if (pk, pst, pnk) != (exact_k, exact_steps, exact_k << S):
                bad_parent += 1
                # The first stretch of a launch starts at B0 = P rounded down to a super-tick (at most 128 ticks of
                # 512 frames below P).  A wrapped fold frame lies about 2^(40+S) below it, so (pnk - B0) / L_full <= 0: the DC
                # pass (w2_dc_correct_kernel) skips the term, and the FIR's fold (fir_param_kernel) either starts a
                # tile there (w < 0: no record read) or keeps the record of the stretch it had (no new index): in no
                # case is corr[] read outside its range.  The term is dropped or taken from the wrong stretch.
                assert pnk == exact_k << S or pnk < P - (1 << 16)
        k_emit = P >> S
        assert fixed_o_cur(k_emit, D.step, O0) == -(-(k_emit << 24) // D.step)
        parent_ok = parent_o_cur(k_emit, D.step) == -(-(k_emit << 24) // D.step)
        assert parent_ok == ((k_emit << 24) < 1 << 64)
        assert (bad_parent > 0 or not parent_ok) == (O1 * D.step >= 1 << 64), (S, P)
        print(f"[emulation] S={S} P={P:#x}: parent wrong at {bad_parent} sampled outputs, per-warp start "
              f"{'ok' if parent_ok else 'wrong'}")


def test_seek_refuses_positions_past_the_ceiling():
    from iq_tool_b200 import gpu
    c = _plan(decim_cfg(2, 0.7))
    assert c.seek(MAX_POS - 1) == Design(c).R(MAX_POS - 1)
    for bad in (MAX_POS, MAX_POS + 1, (1 << 64) - 1):
        with pytest.raises(gpu.IqGpuError, match="IQGPU_MAX_STREAM_POSITION"):
            c.seek(bad)
    # an interpolating chain reaches the ceiling on its output index first
    ci = _plan(interp_cfg(6.0))
    Di = Design(ci)
    top = MAX_POS // 6 - (1 << 20)
    assert Di.R(top + 1) <= MAX_POS
    ci.seek(top)
    with pytest.raises(gpu.IqGpuError, match="IQGPU_MAX_STREAM_POSITION"):
        ci.seek(MAX_POS // 5)


# ---------------------------------------------------------------------------------------------
# GPU part
# ---------------------------------------------------------------------------------------------
def _impulse_input(D, P, n):
    offs = impulse_positions(D, P, n)
    vals = [IMPULSE_VALUES[i % len(IMPULSE_VALUES)] for i in range(len(offs))]
    x = np.zeros(n, dtype=np.complex64)
    x[offs] = vals
    return x, offs, vals


def check_decim(gpu, cfg, S, P, fused, label, chunk=None):
    chain = gpu.Chain(cfg, 0, fused=fused)
    D = Design(chain)
    assert D.S == S and not D.interp
    n = call_frames(S)
    chunks = chunk or [n // 4, n // 4 + 1, n // 2 - 1]
    # stale data first, then the impulses: every output must be written, and written exactly
    run(chain, P, noise(n, seed_of(label + "stale")), chunks)
    xi, offs, vals = _impulse_input(D, P, n)
    yi, counts = run(chain, P, xi, chunks)
    assert list(counts) == closed_form_counts(D, P, chunks), f"{label}: per-chunk counts"
    expect = impulse_expect(D, P, n, offs, vals)
    assert yi.size == expect.size, (label, yi.size, expect.size)
    bad = np.flatnonzero(yi != expect)
    assert bad.size == 0, f"{label}: {bad.size} outputs differ from the exact impulse read-back, first at {bad[:4]}"
    # noise against the float64 reference
    x = noise(n, seed_of(label))
    yg, _ = run(chain, P, x, chunks)
    _, y, A, E, _ = reference(D, x, P)
    worst, stat = bound_ratios(yg, y, A, E)
    print(f"[resampler-bound] {label}: err/bound {worst:.3g}, rms/bar {stat:.3g}, impulses {len(offs)}")
    assert worst <= 1.0, f"{label}: an output exceeds the rigorous bound ({worst:.3g}x)"
    assert stat <= 1.0, f"{label}: RMS error {stat:.3g}x the statistical bar"
    if fused and S <= 6:
        assert chain.info().fused_front == 1, f"{label}: the fused front did not run"
    return yg, chain


DECIM = [(S, 0.7) for S in range(10)]


@pytest.mark.gpu
@pytest.mark.parametrize("S,rate", DECIM)
def test_cascade_against_reference_at_every_position(gpu, S, rate):
    n = call_frames(S)
    for P in positions(S, n):
        for f in (1, 0):
            check_decim(gpu, decim_cfg(S, rate), S, P, f, f"S={S} r={rate} fused={f} P={P:#x}")


RATE_CLASSES = [0.55, 0.66, 0.7, 0.8, 0.599, 0.601, 0.6666, 0.6668, 0.749, 0.751, 0.97]


@pytest.mark.gpu
@pytest.mark.parametrize("rate", RATE_CLASSES)
def test_polyphase_rate_classes_and_variants(gpu, rate, monkeypatch):
    """every quad class (floor(2/r), floor(3/r)) and both sides of its edges, with each polyphase variant forced, at the
    positions where o * step wraps; the variant that ran is read back, so a class cannot lose its four-output coverage
    to the fall-back to two outputs per lane unnoticed"""
    for S in (0, 1, 4, 6):
        n = call_frames(S)
        for P in positions(S, n)[4:7]:
            for pairs, lanes in ((0, 1), (1, 2), (2, 4 if quad_class(rate) else 2)):
                monkeypatch.setenv("IQGPU_ARB_PAIRS", str(pairs))
                label = f"S={S} r={rate} pairs={pairs} P={P:#x}"
                chain = check_decim(gpu, decim_cfg(S, rate), S, P, 1, label)[1]
                assert chain.info().polyphase_variant == lanes, f"{label}: ran {chain.info().polyphase_variant} per lane"


def quad_class(rate):
    """fused_front.cu: the four-output variant serves (floor(2/r), floor(3/r)) in (2,3), (2,4), (3,4), (3,5)"""
    step = round((1 << 24) / float(np.float32(rate)))
    b2, b3 = (2 * step) >> 24, (3 * step) >> 24
    return (b2, b3) in ((2, 3), (2, 4), (3, 4), (3, 5))


# ---- the pre-processor, restated ----
_LIBM = ctypes.CDLL(ctypes.util.find_library("m"))
_LIBM.sinf.restype = ctypes.c_float
_LIBM.sinf.argtypes = [ctypes.c_float]
FULL_SCALE = {"cs16": 32768.0, "cu8": 128.0}
K_DC = 48                    # rounded operations along any path into the DC state (module docstring)
DC_REL = gamma(K_DC) + 2.0 ** -20


def nco_table():
    """design.cpp nco_sine_table: sinf (the host's libm) of the float angle 2 pi i / 1024"""
    return np.array([_LIBM.sinf(float(np.float32(2.0 * math.pi * float(i) / 1024.0))) for i in range(1024)],
                    dtype=np.float32)


def convert(raw, fmt):
    """load_frame (device_common.cuh), gain 1: fp32 (v - offset) times the power-of-two scale, exact"""
    v = raw.astype(np.float32)
    if fmt == "cu8":
        v = v - np.float32(127.5)
    v = v * np.float32(1.0 / FULL_SCALE[fmt])
    x = np.empty(v.size // 2, dtype=np.complex64)
    x.real, x.imag = v[0::2], v[1::2]
    return x


def nco_rows(P, n, dtheta, sign):
    """(sign sin, cos) of the table entry nearest to the phase (P + i) dtheta mod 2^32 (nco_mix, pre_params)"""
    theta = (np.uint64((P * dtheta) & 0xffffffff) + np.arange(n, dtype=np.uint64) * np.uint64(dtheta)) & np.uint64(0xffffffff)
    idx = ((theta + np.uint64(1 << 21)) >> np.uint64(22)) & np.uint64(0x3ff)
    tab = nco_table()
    return tab[idx.astype(np.int64)] * np.float32(sign), tab[((idx + np.uint64(256)) & np.uint64(0x3ff)).astype(np.int64)]


def mix_fp32(x, s, c):
    """the kernel's order: re = x.re c - x.im s, im = x.re s + x.im c, every product and sum rounded to fp32"""
    xr, xi = x.real.astype(np.float32), x.imag.astype(np.float32)
    y = np.empty(x.size, dtype=np.complex64)
    y.real = xr * c - xi * s
    y.imag = xr * s + xi * c
    return y


def dc_pole(in_rate):
    """design.cpp design_dc: c = -(float)(-1 + (float)(2 pi 10 / fs)), a = 1 - c (exact)"""
    alpha = np.float32(2.0 * math.pi * 10.0 / float(in_rate))
    c = -np.float32(np.float32(-1.0) + alpha)
    return float(c), float(np.float32(1.0) - c)


def dc_exact(x, c, a):
    """y[n] = x[n] - a v[n-1], v[n] = x[n] + c v[n-1], v = 0 before the seek position; with a V[n-1], V the same
    recurrence over |x| (the absolute state every DC rounding is relative to)"""
    from scipy import signal
    x = np.asarray(x, dtype=np.complex128)
    v = signal.lfilter([1.0], [1.0, -c], x)
    V = signal.lfilter([1.0], [1.0, -c], np.abs(x))
    y = x - a * np.concatenate([[0.0], v[:-1]])
    return y, a * np.concatenate([[0.0], V[:-1]])


def pre_reference(cfg, raw, P, info):
    """(x, e_in): the pre-processed stream (conversion, DC blocker in exact arithmetic, LUT-NCO mix with the chain's
    fp32 table) and the kernel's DC error allowance per frame"""
    n = raw.size // 2
    x = convert(raw, cfg.input_format).astype(np.complex128)
    e_in = np.zeros(n)
    if cfg.dc_block:
        c, a = dc_pole(int(cfg.input_rate_hz))
        x, aV = dc_exact(x, c, a)
        e_in = DC_REL * aV
    if cfg.freq_shift_hz and not cfg.shift_after_resample:
        s, co = nco_rows(P, n, int(info.nco_dtheta), 1.0 if cfg.freq_shift_hz >= 0 else -1.0)
        x = x * (co.astype(np.float64) + 1j * s.astype(np.float64))
    return x, e_in


def int_raw(fmt, n, seed, offset=0):
    from iq_tool_b200.configs import NUMPY_DTYPE
    rng = np.random.Generator(np.random.PCG64(seed))
    lo, hi = (0, 256) if fmt == "cu8" else (-12000, 12000)
    return np.clip(rng.integers(lo, hi, 2 * n) + offset, lo, hi - 1).astype(NUMPY_DTYPE[fmt])


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["cs16", "cu8"])
def test_integer_inputs_and_nco(gpu, fmt):
    """the pre-processed stream restated in fp32 (conversion, then the LUT-NCO mix in the kernel's order from
    (P + i) dtheta mod 2^32) equals tap 0 bit for bit, at 0, past 2^32, past 2^(40+S) and near 2^62 (which pins the pre
    kernel's NCO phase); the stage path and the fused front (which converts and mixes in its own order: + 4u|x|) are
    then held to the reference fed with that restatement"""
    S = 4
    n = call_frames(S)
    for P in (0, (1 << 32) - n // 2 + 5, (1 << (40 + S)) - n // 2 - 3, MAX_POS - n - 17):
        for shift in (0.0, 12_345.0, -23_456.0):
            cfg = decim_cfg(S, 0.7, fmt)
            cfg.freq_shift_hz = shift
            raw = int_raw(fmt, n, seed_of(f"{fmt}{P}{shift}"))
            st = gpu.Chain(cfg, 0, record_taps=2)
            st.seek(P)
            ys = st.process(raw).view(np.complex64)
            x = convert(raw, fmt)
            if shift:
                x = mix_fp32(x, *nco_rows(P, n, int(st.info().nco_dtheta), 1.0 if shift > 0 else -1.0))
            assert np.array_equal(st.read_tap(0).view(np.uint32), x.view(np.uint32)), \
                f"{fmt} shift={shift} P={P:#x}: the pre-processed stream differs from its restatement"
            D = Design(st)
            _, y, A, E, _ = reference(D, x, P)
            worst, stat = bound_ratios(ys, y, A, E)
            assert worst <= 1.0 and stat <= 1.0, (fmt, P, shift, worst, stat)
            fu = gpu.Chain(cfg, 0, fused=1)
            fu.seek(P)
            yf = fu.process(raw).view(np.complex64)
            _, y, A, E, _ = reference(D, x, P, e0=4 * U)
            worst, stat = bound_ratios(yf, y, A, E)
            print(f"[resampler-bound] {fmt} shift={shift} P={P:#x} fused: err/bound {worst:.3g}, rms/bar {stat:.3g}")
            assert worst <= 1.0 and stat <= 1.0, (fmt, P, shift, worst, stat)
            assert fu.info().fused_front == 1


def dc_cfg(mode):
    from iq_tool_b200.configs import lowpass
    S = 4
    cfg = ChainConfig(input_format="cs16", output_format="cf32", input_rate_hz=IN_RATE << S,
                      target_rate_hz=IN_RATE * 0.7, dc_block=True)
    if mode == "table":             # DC followed by a table NCO: the fused front's DC pre-pass
        cfg.freq_shift_hz = 12_345.0
    if mode == "fold":              # local DC with a 255-tap FIR behind the front, which adds the DC term itself
        cfg.filters = [lowpass(100e3)]
        cfg.filter_taps = 255
    return S, cfg


def fir_after(h, y, A, E):
    """the time-domain FIR y[n] = sum_k h[k] x[n-k] on the reference stream, with its fp32 bound (K = 2 padded + 1)"""
    h = np.asarray(h).astype(np.complex128)
    K = 2 * ((h.size + 7) & ~7) + 1
    ah = np.abs(h)
    conv = lambda a, b: np.convolve(a, b)[: y.size]
    return conv(y, h), conv(A, ah), conv(E, ah) + gamma(K) * conv(A + E, ah)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["local", "table", "fold"])
def test_dc_chains_against_reference(gpu, mode):
    """the DC blocker in each mode of the fused front (local state with the closed-form correction pass, the table
    pre-pass behind which the NCO mixes, the local state whose term the FIR adds while it stages its tiles) and on the
    stage path, held to the exact reference with the DC allowance of the module docstring, at every item position"""
    S, cfg = dc_cfg(mode)
    n = call_frames(S)
    chunks = [n // 4, n // 4 + 1, n // 2 - 1]
    for P in positions(S, n):
        raw = int_raw("cs16", n, seed_of(f"dc{mode}{P}"), offset=3000)
        for fused in (1, 0):
            chain = gpu.Chain(cfg, 0, fused=fused)
            D = Design(chain)
            chain.seek(P)
            yg, counts = chain.process(raw, chunk_frames=chunks, return_chunk_counts=True)
            yg = yg.view(np.complex64)
            assert list(counts) == closed_form_counts(D, P, chunks)
            x, e_in = pre_reference(cfg, raw, P, chain.info())
            _, y, A, E, _ = reference(D, x, P, e0=4 * U, e_in=e_in)
            E = E + U * (A + E)              # the correction term's own addition to each output (or staged sample)
            if mode == "fold":
                y, A, E = fir_after(chain.filter_taps(), y, A, E)
            worst, stat = bound_ratios(yg, y, A, E)
            print(f"[resampler-bound] DC {mode} fused={fused} P={P:#x}: err/bound {worst:.3g}, rms/bar {stat:.3g}, "
                  f"DC allowance at the input {float(e_in.max()):.2g}")
            assert float(e_in.max()) < 1e-5, "the DC allowance must stay far below what a wrong row or pairing makes"
            assert worst <= 1.0, f"DC {mode} fused={fused} P={P:#x}: an output exceeds the bound ({worst:.3g}x)"
            assert stat <= 1.0, f"DC {mode} fused={fused} P={P:#x}: RMS error {stat:.3g}x the statistical bar"
            if fused:
                assert chain.info().fused_front == 1


@pytest.mark.gpu
@pytest.mark.parametrize("ratio", [1.5, 6.0])
def test_interpolation_against_reference(gpu, ratio):
    chain = gpu.Chain(interp_cfg(ratio), 0)
    D = Design(chain)
    assert D.interp
    n = 1 << 14
    for P in positions(D.S, n, interp_ratio=ratio):
        chunks = [n // 2, n // 2]
        run(chain, P, noise(n, seed_of(f"istale{P}")), chunks)
        x = noise(n, seed_of(f"interp{ratio}{P}"))
        yg, counts = run(chain, P, x, chunks)
        assert list(counts) == closed_form_counts(D, P, chunks)
        a0, y, A, E, _ = reference(D, x, P)
        assert a0 == D.R(P)
        worst, stat = bound_ratios(yg, y, A, E)
        print(f"[resampler-bound] interp r={ratio} P={P:#x}: err/bound {worst:.3g}, rms/bar {stat:.3g}")
        assert worst <= 1.0 and stat <= 1.0, (ratio, P, worst, stat)
        # copies of the polyphase stage's outputs, single products where the impulses lie 16 input frames apart
        # (a window spans 14): exact
        xi = np.zeros(n, dtype=np.complex64)
        xi[3::16] = [IMPULSE_VALUES[i % len(IMPULSE_VALUES)] for i in range(xi[3::16].size)]
        yi, _ = run(chain, P, xi, chunks)
        a0, y, A, E, _ = reference(D, xi.astype(np.complex128), P)
        off = 0
        for s in range(D.S):
            off = 2 * (off + D.m[s])
        copies = np.arange(off, y.size, 1 << D.S)
        assert np.array_equal(yi[copies], y[copies].astype(np.complex64)), (ratio, P)
        assert np.count_nonzero(yi[copies]) > copies.size // 2


def full_cfg(kind):
    from iq_tool_b200.configs import lowpass
    if kind == "cfg2":          # local DC, 255-tap FIR with the DC fold, cs16 out
        return ChainConfig(input_format="cs16", output_format="cs16", input_rate_hz=2_000_000, target_rate_hz=100_000,
                           dc_block=True, filters=[lowpass(30e3)], filter_taps=255)
    if kind == "cfg1":          # pre shift, digital AGC, cu8 out
        from iq_tool_b200.configs import AGC_DIGITAL
        return ChainConfig(input_format="cs16", output_format="cu8", input_rate_hz=2_000_000, target_rate_hz=800_000,
                           freq_shift_hz=100_000.0, agc_enable=True, agc_profile=AGC_DIGITAL)
    if kind == "cfg5":          # table DC behind a pre shift, cf32 out, S = 6
        return ChainConfig(input_format="cs16", output_format="cf32", input_rate_hz=2_048_000, target_rate_hz=25_600,
                           dc_block=True, freq_shift_hz=-50_000.0)
    if kind == "s0":            # S = 0 high rate
        return ChainConfig(input_format="cs16", output_format="cs16", input_rate_hz=61_440_000, target_rate_hz=49_152_000)
    if kind == "post":          # post shift
        return ChainConfig(input_format="cu8", output_format="cf32", input_rate_hz=2_000_000, target_rate_hz=400_000,
                           freq_shift_hz=25_000.0, shift_after_resample=True)
    raise KeyError(kind)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["cfg2", "cfg1", "cfg5", "s0", "post"])
def test_full_chains_are_translation_invariant(gpu, kind):
    """a full chain at P + j T gives the bytes and chunk counts it gives at P (T = 5 * 2^36 frames, module docstring)"""
    from iq_tool_b200.configs import NUMPY_DTYPE
    cfg = full_cfg(kind)
    chain = gpu.Chain(cfg, 0)
    D = Design(chain)
    assert D.step % (5 << 22) == 0 or D.step == 1 << 24, f"{kind}: step {D.step} is not periodic in T"
    n = 3 * 16384 + 4097
    chunks = [16384, 16384, 16384, 4097]
    rng = np.random.Generator(np.random.PCG64(seed_of(kind)))
    dt = NUMPY_DTYPE[cfg.input_format]
    lo, hi = (0, 256) if cfg.input_format == "cu8" else (-12000, 12000)
    raw = (rng.integers(lo, hi, 2 * n) + (300 if cfg.dc_block else 0)).astype(dt)
    outs = {}
    wraps = [(1 << (e + D.S)) - n // 2 - 3 for e in (39, 40, 41)] + [(1 << 52) + 11, MAX_POS - n - 5]
    for W in wraps:
        P0, j = W % T_SHIFT, W // T_SHIFT
        for P in (P0, W):
            if P not in outs:
                chain.seek(P)
                o, cnt = chain.process(raw, chunk_frames=chunks, return_chunk_counts=True)
                assert list(cnt) == closed_form_counts(D, P, chunks), (kind, P)
                outs[P] = o.copy()
        assert j > 0
        assert np.array_equal(outs[P0].view(np.uint8), outs[W].view(np.uint8)), \
            f"{kind}: output at {W:#x} differs from the output at {P0:#x} = {W:#x} - {j} T"
    assert chain.info().fused_front == 1


@pytest.mark.gpu
def test_process_refuses_positions_past_the_ceiling(gpu):
    chain = gpu.Chain(decim_cfg(1, 0.7), 0)
    n = 4096
    chain.seek(MAX_POS - n)
    chain.process(_raw_cf32(noise(n, 1)))
    chain.seek(MAX_POS - n + 1)
    with pytest.raises(gpu.IqGpuError, match="IQGPU_MAX_STREAM_POSITION"):
        chain.process(_raw_cf32(noise(n, 1)))
    ci = gpu.Chain(interp_cfg(6.0), 0)
    Di = Design(ci)
    top = MAX_POS // 6 - n
    while Di.R(top + n) <= MAX_POS:
        top += n // 4
    ci.seek(top - n)
    ci.process(_raw_cf32(noise(n // 2, 2)))
    ci.seek(top)
    with pytest.raises(gpu.IqGpuError, match="IQGPU_MAX_STREAM_POSITION"):
        ci.process(_raw_cf32(noise(n, 2)))
