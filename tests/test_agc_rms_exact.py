"""The RMS AGC (liquid agc_crcf) bit for bit against the plain serial loop.

The GPU evaluates the recurrence time-parallel (guessed block start states, grid-wide sweeps to a fixed point, early stops
on 256-sample checkpoints, an out-of-line path for rare operands) and re-runs it from a new state at any frame for time
shards (the resume kernel).  DESIGN.md promises that all of this gives the serial loop's bits.  A near miss (a sweep too
few, a merge on a stale checkpoint, a wrong exp branch) is a few-ulp trajectory that re-merges within thousands of
samples, an error near 1e-7 that the 1e-5 parity bar cannot see, so every GPU test here compares bits.

The serial reference is tests/native/agc_rms_serial.cpp (built with g++ here, with the GPU's log / exp from agc_math.h).
The CPU tests show it is liquid's recurrence (against the oracle's agc_crcf) and that the log / exp it shares with the GPU
are correctly rounded over every argument the recurrence can reach.
"""
import ctypes as C
import dataclasses
import math
import os
import re
import subprocess

import numpy as np
import pytest

from helpers import rel_rms_fullscale, snr_db
from iq_tool_b200.configs import AGC_DX, AGC_LOCAL, FORMAT_CODES, NUMPY_DTYPE, FILTER_REQ_FIR, ChainConfig, lowpass

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NATIVE = os.path.join(ROOT, "tests", "native")
CHUNK = 16384
ALPHA = {AGC_LOCAL: 1e-2, AGC_DX: 1e-4}
# the plan's block length (kernels.cu agc_rms_plan: 30 time constants, at most 65536, a multiple of 4) for every n
# below (co-resident threads) x 3000, i.e. every n these tests use
BLOCK = {AGC_LOCAL: 3000, AGC_DX: 65536}
PROFILE_ID = {AGC_LOCAL: "local", AGC_DX: "dx"}
RESET = (1.0, 1.0)                         # {g, y2'} after create / reset (liquid agc_crcf_set_gain(1) after set_signal_level)
FAR_STATES = [(3.0, 1e-3), (0.05, 40.0)]   # resume states far from any true state


# ------------------------------------------------------------------------------------------------
# the serial reference
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def serial(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("agcserial") / "libagc_rms_serial.so")
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-ffp-contract=off", "-o", out,
                    os.path.join(NATIVE, "agc_rms_serial.cpp")], check=True)
    lib = C.CDLL(out)
    lib.agc_rms_serial.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_void_p, C.c_void_p]
    lib.agc_rms_serial.restype = None

    def run(x, alpha, state=RESET, stats=None):
        """(y complex64, end state float32[2]) of the serial loop over x from `state`; stats: uint64[5] to add to."""
        x = np.ascontiguousarray(x, dtype=np.complex64)
        y = np.empty_like(x)
        st = np.array(state, dtype=np.float32)
        lib.agc_rms_serial(x.ctypes.data, y.ctypes.data, x.size, alpha, st.ctypes.data,
                           stats.ctypes.data if stats is not None else None)
        return y, st
    return run


def _stats():
    return np.zeros(5, dtype=np.uint64)


FROZEN, EXP_SMALL, EXP_LIBM, CLAMPED, GENERIC = range(5)


# ------------------------------------------------------------------------------------------------
# signals (lengths in time constants 1/alpha where the feature needs them)
# ------------------------------------------------------------------------------------------------
def _tone(n, amp, seed, f=0.0123, noise=0.03):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    x = np.exp(2j * np.pi * f * t) + noise * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return (amp * x).astype(np.complex64)


def _corners(n, seed):
    """full scale on both rails: (+-1 +-1j), |x|^2 = 2"""
    rng = np.random.default_rng(seed)
    return np.array([1 + 1j, 1 - 1j, -1 + 1j, -1 - 1j], dtype=np.complex64)[rng.integers(0, 4, n)]


def _cuts(n, fractions):
    edges = np.round(np.cumsum([0.0] + list(fractions)) / sum(fractions) * n).astype(int)
    return list(zip(edges[:-1], edges[1:]))


def signal(kind, n, alpha, seed=1):
    x = _tone(n, 0.3, seed)
    if kind == "tone":                     # the straight-line path (up to the rare y2' == 1.0f)
        return x
    if kind == "steps":                    # +40, -60, +60, -40 dB
        for (a, b), amp in zip(_cuts(n, [1] * 5), [0.01, 1.0, 0.001, 1.0, 0.01]):
            x[a:b] *= amp / 0.3
        return x
    if kind == "zeros":                    # exact zeros: y2' decays below 1e-6 (gain frozen, alpha*y2 = 0) and on into
        a, b = _cuts(n, [1, 6, 1])[1]      # subnormals, then the tone wakes it up
        x[a:b] = 0
        return x
    if kind == "unit":                     # |x| == 1 exactly from the reset state: y2' == 1.0f, t = -0 in every step
        rng = np.random.default_rng(seed)
        return np.array([1, -1, 1j, -1j], dtype=np.complex64)[rng.integers(0, 4, n)]
    if kind == "clamp_burst":              # 1e-7 until g sits at its 1e6 clamp, then a full-scale burst: y2' ~ 1e10 .. 1e11
        b = _cuts(n, [2, 1])[0][1]
        x[:b] = _tone(b, 1e-7, seed, noise=0.0)
        x[b:] = _corners(n - b, seed)
        return x
    if kind == "subnormal":                # samples below the smallest normal float
        a, b = _cuts(n, [1, 2, 1])[1]
        x[a:b] = _tone(b - a, 3e-39, seed, noise=0.0)
        x[a:b] += np.float32(1e-45) * np.complex64(1 + 1j)
        return x
    if kind == "live":                     # for the long, ragged, sub-train and resume runs: the gain stays live.  Steps of
        tc = int(1 / alpha)                # +40 / -40 / -60 / +60 dB, subnormal samples, then exact zeros (the gain rises to
        lv = [(3, 0.3), (2, 30.0), (4, 0.3), (3, 3e-4), (3, 0.3), (0.5, 1e-40), (15, 0.3),   # its clamp and freezes for a
              (16, 0.0), (3, 1e-6), (3, 1e-4), (3, 1e-2), (3, 0.3)]                          # while) and back in 40 dB steps
        pat = np.concatenate([_tone(int(k * tc), amp, seed + i, noise=0.03 if amp > 1e-30 else 0.0)
                              for i, (k, amp) in enumerate(lv)])
        return np.resize(pat, n).astype(np.complex64)
    raise ValueError(kind)


SIGNALS = ["tone", "steps", "zeros", "unit", "clamp_burst", "subnormal"]


def live_signal(serial, n, alpha, seed=1):
    """The "live" signal, checked on the serial loop to keep the AGC live over the whole run: most steps take the GPU's
    straight-line path, a frozen gain wakes up again, the outputs stay far from 0 and the end gain is a normal float (a
    run that ends dead, g subnormal and every output 0, would check nothing of the straight-line step or of checkpoint
    merges)."""
    x = signal("live", n, alpha, seed)
    st = _stats()
    y, end = serial(x, alpha, stats=st)
    assert st[GENERIC] <= n // 3, st.tolist()
    assert 1.17549435e-38 <= end[0] <= 1e6, end.tolist()   # g a normal float
    assert (np.abs(y[np.abs(x) > 1e-30]) > 1e-30).mean() >= 0.98   # the outputs of normal inputs are alive
    if n >= 60 / alpha:                    # a whole pattern: the frozen stretch is there, and it ends
        assert 0 < st[FROZEN] <= n // 8, st.tolist()
    return x
# long enough for every feature: zeros reach subnormal y2' (87 time constants), the quiet part of clamp_burst holds g at 1e6
SIGNAL_N = {AGC_LOCAL: 60 * 3000 + 17, AGC_DX: 24 * 65536 + 17}


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_agc_log_exp_are_correctly_rounded_over_the_reachable_range(tmp_path):
    """agc_math.h: log over every 97th float in [1e-6, FLT_MAX] (y2' up to the ~1e12 of a burst behind a clamped gain, and
    beyond), agc_exp_tiny on 1e-12 <= |t| <= 0.125 and agc_exp_small on 0.125 <= |t| <= 0.5: pre-rounding error below
    2e-15 (so the float result is the correctly rounded one except within 2e-15 of a rounding boundary) and, on these
    arguments, no result off the correctly rounded float."""
    exe = str(tmp_path / "agc_math_check")
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-o", exe, os.path.join(NATIVE, "agc_math_check.cpp")], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    print(r.stdout)
    assert r.returncode == 0, r.stdout
    got = {m.group(1): (int(m.group(2)), int(m.group(3)), float(m.group(4)))
           for m in re.finditer(r"^(\w+): (\d+) arguments, (\d+) differ from the correctly rounded float.*error (\S+) at",
                                r.stdout, re.M)}
    assert set(got) == {"logf", "agc_exp_tiny", "agc_exp_small"}
    assert got["logf"][0] > 12_000_000 and got["agc_exp_small"][0] > 300_000
    for name, (n, off, worst) in got.items():
        assert off == 0 and worst <= 2e-15, (name, n, off, worst)


@pytest.mark.parametrize("profile", [AGC_LOCAL, AGC_DX], ids=PROFILE_ID.get)
@pytest.mark.parametrize("kind", SIGNALS + ["live"])
def test_serial_reference_is_liquids_recurrence(serial, profile, kind):
    """The serial reference against the oracle's agc_crcf_execute_block (glibc logf / expf, the product (1 - alpha) y2'
    rounded on its own): the same recurrence up to those roundings, 1e-6 relative RMS.  The signals reach what they are
    meant to reach (counted by the reference)."""
    from oracle.loader import CpuChain
    alpha = ALPHA[profile]
    n = SIGNAL_N[profile]
    x = signal(kind, n, alpha)
    st = _stats()
    y, _ = serial(x, alpha, stats=st)
    cfg = ChainConfig(input_format="cf32", output_format="cf32", input_rate_hz=1e6, target_rate_hz=1e6, no_resample=True,
                      agc_enable=True, agc_profile=profile)
    ref = CpuChain(cfg, "oracle").process(x.view(np.float32)).view(np.complex64)
    assert ref.size == n
    d = y.astype(np.complex128) - ref.astype(np.complex128)
    rel = math.sqrt(np.mean(np.abs(d) ** 2) / np.mean(np.abs(ref.astype(np.complex128)) ** 2))
    print(f"{kind}: serial vs oracle relative RMS {rel:.3g}, stats {st.tolist()}")
    assert rel <= 1e-6
    if kind == "zeros":
        assert st[FROZEN] > 0
    if kind == "unit":
        assert st[GENERIC] == n and st[FROZEN] == 0
    if kind == "live":
        live_signal(serial, n, alpha)
    if kind == "clamp_burst":
        assert st[CLAMPED] > 0
        if profile == AGC_LOCAL:              # |t| <= alpha/2 ln(1e12) = 0.0014 at DX: the small-exp range needs LOCAL
            assert st[EXP_SMALL] > 0
    if kind == "tone":
        assert st[GENERIC] <= n // 1000


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _cfg(profile, output_format="cf32", **kw):
    """cf32 in, no resampler and no pre stages: the AGC's input is the raw input and its output the chain's."""
    return ChainConfig(input_format="cf32", output_format=output_format, input_rate_hz=1e6, target_rate_hz=1e6,
                       no_resample=True, agc_enable=True, agc_profile=profile, **kw)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _same_bits(a, b):
    return a.shape == b.shape and bool(np.array_equal(_bits(a), _bits(b)))


def _diff_report(got, want):
    g, w = got.astype(np.complex128), want.astype(np.complex128)
    bad = np.flatnonzero(np.any(_bits(got.view(np.float32).reshape(-1, 2)) != _bits(want.view(np.float32).reshape(-1, 2)),
                                axis=1))
    if not bad.size:
        return "same bits"
    return (f"{bad.size} of {got.size} samples differ (first {bad[0]}, last {bad[-1]}), "
            f"max |error| {np.abs(g - w).max():.3g}, max |want| {np.abs(w).max():.3g}")


def _assert_same(got, want, what=""):
    assert _same_bits(got, want), f"{what}: {_diff_report(got, want)}"


def _assert_state(chain, want, what=""):
    g, y2 = chain.get_agc_rms_state()
    got = np.array([g, y2], dtype=np.float32)
    assert _same_bits(got, np.asarray(want, dtype=np.float32)), f"{what}: state {got.tolist()} != serial {list(want)}"


class _Run:
    """One chain on cuda:0 and one device input / output pair."""

    def __init__(self, gpu, cfg, x, **opts):
        import torch
        self.torch = torch
        self.cfg = cfg
        self.chain = gpu.Chain(cfg, 0, **opts)
        self.x = x
        self.dx = torch.from_numpy(np.ascontiguousarray(x).view(np.float32).copy()).cuda()
        self.out = torch.zeros(max(1, self.chain.out_capacity_frames(x.size)) * cfg.out_bytes, dtype=torch.uint8,
                               device="cuda")

    def process(self, first=0, frames=None, out_off=0):
        frames = self.x.size - first if frames is None else frames
        k = self.chain.process_device(self.dx.data_ptr() + 8 * first, frames, self.out.data_ptr() + out_off * self.cfg.out_bytes,
                                      self.out.numel() - out_off * self.cfg.out_bytes)
        self.torch.cuda.synchronize()
        return k

    def output(self, n):
        raw = self.out[: n * self.cfg.out_bytes].cpu().numpy()
        return raw.view(np.complex64) if self.cfg.output_format == "cf32" else raw.view(NUMPY_DTYPE[self.cfg.output_format])


def _agc_debug_lines(text):
    return [tuple(int(v) for v in m.groups())
            for m in re.finditer(r"rms agc: n=(\d+) alpha=\S+ block=(\d+) blocks=(\d+) sweeps=(\d+)", text)]


def _plan_edges(profile):
    B = BLOCK[profile]
    many = 129 * B + 77                    # > 128 blocks: more than one CTA of the cooperative grid
    return [1, 7, 8, 9, B - 1, B, B + 1, 3 * B + 5, many]


@pytest.mark.gpu
@pytest.mark.parametrize("profile,n", [pytest.param(p, n, id=f"{PROFILE_ID[p]}-{n}")
                                       for p in (AGC_LOCAL, AGC_DX) for n in _plan_edges(p)])
def test_plan_edges_give_the_serial_bits(gpu, serial, profile, n, monkeypatch, capfd):
    """One call of n frames: block counts around the plan's block length B (30 time constants), a tail shorter than the
    eight-sample groups, and more than 128 blocks.  The plan is the one intended (IQGPU_DEBUG_AGC line) and the long DX
    call needs more than two sweeps, so the multi-sweep path with early stops ran."""
    monkeypatch.setenv("IQGPU_DEBUG_AGC", "1")
    alpha, B = ALPHA[profile], BLOCK[profile]
    x = live_signal(serial, n, alpha)
    opts = {"subtrain_frames": n + CHUNK} if n > (1 << 22) else {}
    r = _Run(gpu, _cfg(profile), x, **opts)
    assert r.process() == n
    y, st = serial(x, alpha)
    _assert_same(r.output(n), y, f"n={n}")
    _assert_state(r.chain, st, f"n={n}")
    lines = _agc_debug_lines(capfd.readouterr().err)
    assert len(lines) == 1, lines
    nn, block, blocks, sweeps = lines[0]
    assert (nn, block, blocks) == (n, B, -(-n // B))
    if n > 128 * B and profile == AGC_DX:
        assert sweeps > 2, lines


@pytest.mark.gpu
@pytest.mark.parametrize("profile", [AGC_LOCAL, AGC_DX], ids=PROFILE_ID.get)
@pytest.mark.parametrize("kind", SIGNALS)
def test_signals_give_the_serial_bits(gpu, serial, profile, kind):
    """Level steps, exact zeros into a frozen gain and subnormal y2', |x| = 1 (every step off the straight-line path), a
    burst behind a clamped gain (agc_exp_small at LOCAL), subnormal samples: output and end state are the serial loop's."""
    alpha, n = ALPHA[profile], SIGNAL_N[profile]
    x = signal(kind, n, alpha)
    r = _Run(gpu, _cfg(profile), x)
    assert r.process() == n
    y, st = serial(x, alpha)
    _assert_same(r.output(n), y, kind)
    _assert_state(r.chain, st, kind)


RAGGED = [1, 3, 2999, 3001, 100_003, 8, 65_536, 7, 256, 70_001]


@pytest.mark.gpu
@pytest.mark.parametrize("profile", [AGC_LOCAL, AGC_DX], ids=PROFILE_ID.get)
@pytest.mark.parametrize("small_subtrains", [False, True], ids=["one_subtrain", "small_subtrains"])
def test_ragged_calls_give_one_serial_run(gpu, serial, profile, small_subtrains):
    """Calls of ragged sizes (odd input and output offsets: the element-wise load / store path) carry {g, y2'} from call
    to call; with small sub-trains every call is cut into several AGC launches.  The stitched output is one serial run."""
    alpha = ALPHA[profile]
    n = sum(RAGGED)
    x = live_signal(serial, n, alpha, seed=5)
    opts = {"chunk_frames": 4096, "subtrain_frames": 10_000} if small_subtrains else {}
    r = _Run(gpu, _cfg(profile), x, **opts)
    at = 0
    for f in RAGGED:
        assert r.process(first=at, frames=f, out_off=at) == f
        at += f
    y, st = serial(x, alpha)
    _assert_same(r.output(n), y, "ragged")
    _assert_state(r.chain, st, "ragged")


@pytest.mark.gpu
@pytest.mark.parametrize("ragged", [False, True], ids=["one_call", "ragged_calls"])
def test_post_shift_inside_the_agc_kernel(gpu, serial, ragged):
    """shift_after_resample with the RMS AGC: the NCO mix runs inside the AGC kernel.  Expected: the serial loop over the
    same chain's output with the AGC off (the shifted stream)."""
    alpha = ALPHA[AGC_LOCAL]
    n = sum(RAGGED)
    x = signal("steps", n, alpha, seed=9)
    sizes = RAGGED if ragged else [n]
    outs = []
    for agc in (False, True):
        cfg = dataclasses.replace(_cfg(AGC_LOCAL), freq_shift_hz=123_456.7, shift_after_resample=True, agc_enable=agc)
        r = _Run(gpu, cfg, x)
        at = 0
        for f in sizes:
            assert r.process(first=at, frames=f, out_off=at) == f
            at += f
        outs.append((r, r.output(n)))
    shifted = outs[0][1]
    assert not _same_bits(shifted, x)           # the shift ran
    y, st = serial(shifted, alpha)
    _assert_same(outs[1][1], y, "post shift")
    _assert_state(outs[1][0].chain, st, "post shift")


# ---- resume -----------------------------------------------------------------------------------------------------------
class _Resumer:
    """A chain after one process_device call over x, and the model every resume has to meet: outputs in front of `first`
    keep their bytes, outputs from `first` on are the serial loop from the given state, the end state is that loop's,
    `changed` says whether the end state moved."""

    def __init__(self, gpu, serial, profile, x, output_format="cf32"):
        import torch
        self.gpu, self.serial, self.alpha, self.x = gpu, serial, ALPHA[profile], x
        self.cfg = _cfg(profile, output_format)
        self.run = _Run(gpu, self.cfg, x, subtrain_frames=x.size + CHUNK)
        self.n = x.size
        assert self.run.process() == self.n
        self.model, self.end = serial(x, self.alpha)
        self.dev_state = torch.zeros(2, dtype=torch.float32, device="cuda")
        self.changed = torch.full((1,), -1, dtype=torch.int32, device="cuda")
        self.check("process")

    def expected_bytes(self):
        if self.cfg.output_format == "cf32":
            return self.model
        return self.gpu.convert_cf32_to_block(self.model, FORMAT_CODES[self.cfg.output_format],
                                              NUMPY_DTYPE[self.cfg.output_format], self.cfg.out_bytes)

    def check(self, what):
        got, want = self.run.output(self.n), self.expected_bytes()
        if self.cfg.output_format == "cf32":
            _assert_same(got, want, what)
        else:
            bad = np.flatnonzero(got != want)
            assert not bad.size, f"{what}: {bad.size} of {want.size} values differ, first at {bad[0]}"
        _assert_state(self.run.chain, self.end, what)

    def true_state(self, first):
        return tuple(self.serial(self.x[:first], self.alpha)[1]) if first else RESET

    def resume(self, first, state):
        self.dev_state.copy_(self.run.torch.tensor(state, dtype=self.run.torch.float32))
        self.changed.fill_(-1)
        self.run.chain.agc_rms_resume_device(first, self.dev_state.data_ptr(), self.run.out.data_ptr(), self.run.out.numel(),
                                             self.changed.data_ptr())
        self.run.torch.cuda.synchronize()
        y, end = self.serial(self.x[first:], self.alpha, state)
        self.model = np.concatenate([self.model[:first], y])
        moved = not _same_bits(end, self.end)
        self.end = end
        what = f"resume at {first} from {tuple(float(v) for v in state)}"
        self.check(what)
        assert int(self.changed.item()) == int(moved), what
        return moved


def _resume_firsts(profile, n):
    B = BLOCK[profile]
    return [0, 1, 8, 255, 256, 257, B - 1, B, B + 1, 5 * B + 123, n - 1, n]


RESUME_N = {AGC_LOCAL: 12 * 3000 + 77, AGC_DX: 8 * 65536 + 77}


@pytest.mark.gpu
@pytest.mark.parametrize("profile,first", [pytest.param(p, f, id=f"{PROFILE_ID[p]}-{f}")
                                           for p in (AGC_LOCAL, AGC_DX) for f in _resume_firsts(p, RESUME_N[p])])
def test_resume_at_one_frame_gives_the_serial_bits(gpu, serial, profile, first):
    """Resumes at checkpoint, block and call edges: from the true state (nothing changes), from far states s1, s2, s1 (each
    is the serial loop from its state; the trajectory in memory before each is another resume's), s1 once more (the
    on-device no-op) and the true state again (back to the call's own trajectory)."""
    x = live_signal(serial, RESUME_N[profile], ALPHA[profile], seed=3)
    R = _Resumer(gpu, serial, profile, x)
    truth = R.true_state(first)
    assert not R.resume(first, truth)
    s1, s2 = FAR_STATES
    for s in (s1, s2, s1):
        R.resume(first, s)
    assert not R.resume(first, s1)
    R.resume(first, truth)


@pytest.mark.gpu
@pytest.mark.parametrize("profile", [AGC_LOCAL, AGC_DX], ids=PROFILE_ID.get)
def test_resume_at_later_and_earlier_frames(gpu, serial, profile):
    """Resumes of one call at different frames.  Later: the trajectory in memory from the earlier frame on is the earlier
    resume's, and that is what the later one continues.  Earlier (the case the time-shard hand-over never makes): the
    earlier resume meets the call's own trajectory in front of the later frame, so the outputs from the later frame on
    have to go back to the call's."""
    B, n = BLOCK[profile], RESUME_N[profile]
    x = live_signal(serial, n, ALPHA[profile], seed=4)
    R = _Resumer(gpu, serial, profile, x)
    s1, s2 = FAR_STATES
    R.resume(5 * B + 123, s1)
    R.resume(7 * B + 5, s2)                        # later
    R.resume(B + 3, R.true_state(B + 3))           # earlier, from the true state: back to the call's trajectory
    R.resume(5 * B + 123, s1)
    R.resume(257, s2)                              # earlier, from a far state
    R.resume(2 * B, s1)                            # later again
    R.resume(0, RESET)                             # earliest: everything back to the call's own output


@pytest.mark.gpu
def test_resume_reconverts_integer_output(gpu, serial):
    """cs16 output: the resume converts only the range it rewrote (from the group of four around `first`); the bytes are
    the host conversion of the serial result, in front of `first` too."""
    profile = AGC_LOCAL
    B, n = BLOCK[profile], RESUME_N[profile]
    x = signal("steps", n, ALPHA[profile], seed=6) * np.float32(0.2)
    R = _Resumer(gpu, serial, profile, x, output_format="cs16")
    s1, s2 = FAR_STATES
    for first, s in [(257, s1), (257, s2), (B + 1, s1), (3, s2), (5 * B + 123, R.true_state(5 * B + 123)), (n - 1, s1)]:
        R.resume(first, s)


# ---- DX against the oracle --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_dx_chain_meets_the_bar_against_the_oracle(gpu):
    """A decimating chain into the DX AGC (cu8 2.4 Msps -> 1 Msps, post shift, 255-tap FIR) against the oracle at the
    north_star bar (1e-5 relative RMS, 100 dB): the DX profile's first comparison with the oracle."""
    from oracle.loader import CpuChain
    cfg = ChainConfig(input_format="cu8", output_format="cf32", input_rate_hz=2.4e6, target_rate_hz=1e6,
                      freq_shift_hz=50e3, filters=[lowpass(400e3)], filter_taps=255, filter_type_request=FILTER_REQ_FIR,
                      agc_enable=True, agc_profile=AGC_DX)
    n = 1 << 21
    rng = np.random.default_rng(21)
    t = np.arange(n)
    env = np.ones(n)
    env[n // 4: n // 2] = 0.05
    env[3 * n // 4:] = 3.0
    s = env * (0.2 * np.exp(2j * np.pi * 0.071 * t)) + 0.01 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    raw = np.empty(2 * n, dtype=np.uint8)
    raw[0::2] = np.clip(np.rint(127.5 + 127.0 * s.real), 0, 255)
    raw[1::2] = np.clip(np.rint(127.5 + 127.0 * s.imag), 0, 255)
    out = gpu.Chain(cfg, 0).process(raw)
    ref = CpuChain(cfg, "oracle").process(raw)
    assert out.size == ref.size and out.size > 1_600_000
    a, b = out.view(np.complex64), ref.view(np.complex64)
    rel, snr = rel_rms_fullscale(a, b), snr_db(a, b)
    print(f"DX chain vs oracle: relative RMS {rel:.3g}, SNR {snr:.1f} dB")
    assert rel <= 1e-5 and snr >= 100.0
