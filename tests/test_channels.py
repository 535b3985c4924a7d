"""Several channels out of one capture (include/iqgpu.h: iqgpu_chain_process_multi, iqgpu_rawfile_run_channels,
iqgpu_wavfile_run_channels): K chains consume one input that crosses PCIe once per sub-train.  Every channel is an
ordinary chain, so each is checked byte for byte against the same configuration run alone on the same input.

CPU: the refusals on plan-only chains, and the K-channel file plumbing (rawfile.cpp / wavfile.cpp / channels.cpp)
against the test double of the chain (tests/native/stream_stub.cpp).  GPU: the chains themselves."""
import ctypes as C
import dataclasses
import os
import struct
import subprocess
import wave

import numpy as np
import pytest

from iq_tool_b200 import gpu as G
from iq_tool_b200.configs import (AGC_DIGITAL, AGC_LOCAL, FILTER_REQ_FFT, FORMAT_CODES, NUMPY_DTYPE, ChainConfig,
                                  pass_range)
from iq_tool_b200.synth import synth_numpy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 16384
EINVAL, ENODEVICE, ECAPACITY = -1, -2, -5


def nrsc5(shift_hz: float, base: ChainConfig) -> ChainConfig:
    return dataclasses.replace(base, freq_shift_hz=shift_hz)


# ------------------------------------------------------------------------------------------------ CPU: refusals
def test_refusals_before_any_work_name_the_channel():
    base = ChainConfig()
    a, b = G.Chain(base, -1), G.Chain(base, -1)
    cases = [([a, G.Chain(dataclasses.replace(base, input_format="cu8"), -1)], "channel 1", "input_format"),
             ([a, b, G.Chain(dataclasses.replace(base, input_rate_hz=2.4e6), -1)], "channel 2", "input_rate_hz"),
             ([a, b, a], "channel 2", "already listed as channel 0"),
             ([], "n_chains", "at least 1")]
    raw = np.zeros(2 * 4096, dtype=np.int16)
    for chains, where, what in cases:
        with pytest.raises(G.IqGpuError) as e:
            G.process_channels(chains, raw)
        assert e.value.code == EINVAL and where in str(e.value) and what in str(e.value), str(e.value)


def test_a_valid_set_of_plan_only_chains_needs_a_device():
    cfgs = [ChainConfig(freq_shift_hz=s, output_format=f) for s, f in ((-1e5, "cu8"), (2e5, "cf32"), (0.0, "cs16"))]
    with pytest.raises(G.IqGpuError) as e:
        G.process_channels([G.Chain(c, -1) for c in cfgs], np.zeros(2 * 4096, dtype=np.int16))
    assert e.value.code == ENODEVICE


# ------------------------------------------------------------------------------------------------ CPU: file plumbing
@pytest.fixture(scope="module")
def stub(tmp_path_factory):
    """rawfile.cpp / wavfile.cpp / channels.cpp linked against the chain's test double (every second frame kept),
    with the K-chain call made of K single calls."""
    d = tmp_path_factory.mktemp("channelstub")
    src = d / "multi_stub.cpp"
    src.write_text('#include "%s"\n' % os.path.join(ROOT, "tests", "native", "stream_stub.cpp") + r'''
extern "C" int iqgpu_chain_process_multi(iqgpu_chain* const* chains, size_t n, const void* in, size_t n_frames,
                                         const uint32_t* cf, size_t nc, void* const* out, const size_t* cap,
                                         size_t* out_frames, uint32_t* const* pc)
{
    if (n == 0) { g_err = "stub: no chains"; return IQGPU_EINVAL; }
    for (size_t k = 0; k < n; k++)
        if (chains[k]->cfg.input_format != chains[0]->cfg.input_format) {
            g_err = "channel " + std::to_string(k) + ": input_format differs from channel 0's";
            return IQGPU_EINVAL;
        }
    for (size_t k = 0; k < n; k++) out_frames[k] = 0;
    if (n_frames == 0) return IQGPU_OK;
    for (size_t k = 0; k < n; k++) {
        const int rc = iqgpu_chain_process(chains[k], in, n_frames, cf, nc, out[k], cap[k], &out_frames[k], pc ? pc[k] : nullptr);
        if (rc) return rc;
    }
    return IQGPU_OK;
}
''')
    out = str(d / "libchannelstub.so")
    csrc = os.path.join(ROOT, "iq_tool_b200", "csrc")
    subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-shared", "-fPIC", "-pthread", "-Wall", "-o", out, str(src),
                    os.path.join(csrc, "rawfile.cpp"), os.path.join(csrc, "wavfile.cpp"), os.path.join(csrc, "channels.cpp")],
                   check=True)
    lib = C.CDLL(out)
    lib.iqgpu_rawfile_last_error.restype = C.c_char_p
    return lib


def _cfgs(fmts):
    return (G.ChainConfigC * len(fmts))(*[ChainConfig(input_format=f, output_format=f, input_rate_hz=2.0e6,
                                                      target_rate_hz=1.0e6).to_c() for f in fmts])


def _paths(paths):
    return (C.c_char_p * len(paths))(*[os.fsencode(p) for p in paths])


def test_stub_raw_channels_write_every_output_from_one_read(stub, tmp_path):
    frames = 5 * CHUNK + 77
    raw = np.random.default_rng(3).integers(-32768, 32767, size=2 * frames, dtype=np.int16)
    src = tmp_path / "in.cs16"
    src.write_bytes(raw.tobytes() + b"\x01")
    outs = [tmp_path / f"o{k}.cs16" for k in range(3)]
    st = (G.RawfileStatsC * 3)()
    rc = stub.iqgpu_rawfile_run_channels(_cfgs(["cs16"] * 3), C.c_size_t(3), 0, os.fsencode(src), _paths(outs), C.c_size_t(2), st)
    assert rc == 0, stub.iqgpu_rawfile_last_error()
    want = raw.reshape(-1, 2)[::2].reshape(-1).tobytes()
    for k, o in enumerate(outs):
        assert o.read_bytes() == want
        assert (st[k].frames_in, st[k].frames_out, st[k].bytes_written, st[k].trains) == (frames, (frames + 1) // 2, len(want), 3)


def test_stub_refusals_leave_no_output(stub, tmp_path):
    src = tmp_path / "in.cs16"
    src.write_bytes(b"\0" * 4096)
    outs = [tmp_path / "a.cs16", tmp_path / "no_dir" / "b.cs16", tmp_path / "c.cs16"]
    assert stub.iqgpu_rawfile_run_channels(_cfgs(["cs16"] * 3), C.c_size_t(3), 0, os.fsencode(src), _paths(outs), C.c_size_t(0), None) == EINVAL
    assert b"cannot open output file " + os.fsencode(outs[1]) in stub.iqgpu_rawfile_last_error()
    assert not any(o.exists() for o in outs)
    # a channel the others cannot share the input with is refused before any output is created
    good = [tmp_path / "a.cs16", tmp_path / "b.cs16"]
    assert stub.iqgpu_rawfile_run_channels(_cfgs(["cs16", "cu8"]), C.c_size_t(2), 0, os.fsencode(src), _paths(good), C.c_size_t(0), None) == EINVAL
    assert b"channel 1: input_format" in stub.iqgpu_rawfile_last_error()
    assert not any(o.exists() for o in good)


def test_stub_wav_channels_get_their_own_header_and_rate(stub, tmp_path):
    frames = 3 * CHUNK + 9
    raw = np.arange(2 * frames, dtype=np.int64).astype(np.int16)
    body = struct.pack("<HHIIHH", 1, 2, 2_000_000, 8_000_000, 4, 16)
    src = tmp_path / "in.wav"
    src.write_bytes(b"RIFF" + struct.pack("<I", 4 + 8 + len(body) + 8 + raw.nbytes) + b"WAVE" + b"fmt " + struct.pack("<I", len(body))
                    + body + b"data" + struct.pack("<I", raw.nbytes) + raw.tobytes())
    cfgs = _cfgs(["cs16"] * 3)
    cfgs[1].target_rate_hz = 500_000.0
    outs = [tmp_path / "a.wav", tmp_path / "b.wav", tmp_path / "c.raw"]
    conts = (C.c_int * 3)(1, 1, 0)
    st = (G.RawfileStatsC * 3)()
    rc = stub.iqgpu_wavfile_run_channels(cfgs, C.c_size_t(3), 0, os.fsencode(src), 1, _paths(outs), conts, None, C.c_size_t(1), st, None)
    assert rc == 0, stub.iqgpu_rawfile_last_error()
    want = raw.reshape(-1, 2)[::2].tobytes()
    for o, rate in zip(outs[:2], (1_000_000, 500_000)):
        with wave.open(str(o), "rb") as w:
            assert w.getframerate() == rate and w.readframes(w.getnframes()) == want
    assert outs[2].read_bytes() == want
    # a centre target needs a WAV input; the message names the channel
    t = (C.c_float * 3)(0.0, 0.0, 1e6)
    assert stub.iqgpu_wavfile_run_channels(cfgs, C.c_size_t(3), 0, os.fsencode(outs[2]), 0, _paths(outs), conts, t, C.c_size_t(0), None, None) == EINVAL
    assert b"channel 2: Option --wav-center-target-freq needs a WAV input" in stub.iqgpu_rawfile_last_error()


# ------------------------------------------------------------------------------------------------ GPU
def _alone(cfg, raw_calls, chunk_calls=None, reset_after=None, **options):
    """cfg run alone on a fresh chain over the same calls: (outputs per call, counts per call, chain)."""
    ch = G.Chain(cfg, 0, **options)
    outs, counts = [], []
    for i, raw in enumerate(raw_calls):
        o, c = ch.process(raw, chunk_frames=chunk_calls[i] if chunk_calls else None, return_chunk_counts=True)
        outs.append(o)
        counts.append(c)
        if reset_after == i:
            ch.reset()
    return outs, counts, ch


def _agc(ch: G.Chain):
    return ch.get_agc_state().as_tuple(), ch.get_agc_rms_state(), ch.info().frames_in_total, ch.info().frames_out_total


@pytest.mark.gpu
def test_four_nrsc5_channels_from_one_capture(gpu, workloads):
    wl = workloads["cfg1"]
    cfgs = [nrsc5(s, wl.config) for s in (-300e3, -100e3, 100e3, 250e3)]
    raws = [synth_numpy(wl, 37 * CHUNK + 1234), synth_numpy(wl, 11 * CHUNK + 5, start=37 * CHUNK + 1234)]
    chains = [gpu.Chain(c, 0) for c in cfgs]
    got = [gpu.process_channels(chains, r, return_chunk_counts=True) for r in raws]
    for k, cfg in enumerate(cfgs):
        outs, counts, alone = _alone(cfg, raws)
        for i in range(len(raws)):
            assert got[i][k][0].tobytes() == outs[i].tobytes(), (k, i)
            assert np.array_equal(got[i][k][1], counts[i]), (k, i)
        assert _agc(chains[k]) == _agc(alone), k


def _mixed_configs(cfg2: ChainConfig):
    return [cfg2,
            ChainConfig(input_format="cs16", output_format="cs16", input_rate_hz=20e6, target_rate_hz=10e6,
                        filters=[pass_range(1e6, 3e6)], filter_taps=1023, filter_type_request=FILTER_REQ_FFT),
            ChainConfig(input_format="cs16", output_format="cf32", input_rate_hz=20e6, target_rate_hz=1e6,
                        freq_shift_hz=2e6, agc_enable=True, agc_profile=AGC_LOCAL),
            ChainConfig(input_format="cs16", output_format="cu8", input_rate_hz=20e6, target_rate_hz=744187.5,
                        freq_shift_hz=-3e6, agc_enable=True, agc_profile=AGC_DIGITAL),
            ChainConfig(input_format="cs16", output_format="cs16", input_rate_hz=20e6, target_rate_hz=20e6,
                        no_resample=True, freq_shift_hz=1e6)]


@pytest.mark.gpu
def test_mixed_chains_over_ragged_calls_and_a_reset(gpu, workloads):
    """cfg2, an FFT band-pass (remainder carried across calls), an RMS AGC to cf32, a digital AGC to cu8 and a
    native-rate channel on one 20 Msps input.  One chain has a small subtrain_frames, so every channel is cut at it:
    each lone run is given the same cut (the DC blocker's block sums follow the sub-train cut in the last bit)."""
    wl = workloads["cfg2"]
    cfgs = _mixed_configs(wl.config)
    rng = np.random.default_rng(7)
    sizes = [int(x) for x in rng.integers(1, 20000, size=40)]
    chunk_calls = [sizes[:13], sizes[13:14], sizes[14:]]
    raws, at = [], 0
    for cc in chunk_calls:
        raws.append(synth_numpy(wl, sum(cc), start=at))
        at += sum(cc)
    small = 3 * 20000 + 17
    chains = [gpu.Chain(c, 0) for c in cfgs]
    chains[2].set_option("subtrain_frames", small)
    got = []
    for i, (raw, cc) in enumerate(zip(raws, chunk_calls)):
        got.append(gpu.process_channels(chains, raw, chunk_frames=cc, return_chunk_counts=True))
        if i == 1:
            for ch in chains:
                ch.reset()
    for k, cfg in enumerate(cfgs):
        outs, counts, alone = _alone(cfg, raws, chunk_calls, reset_after=1, subtrain_frames=small)
        for i in range(len(raws)):
            assert got[i][k][0].tobytes() == outs[i].tobytes(), (k, i)
            assert np.array_equal(got[i][k][1], counts[i]), (k, i)
        assert _agc(chains[k]) == _agc(alone), k


@pytest.mark.gpu
def test_a_channel_without_room_leaves_every_chain_where_it_was(gpu, workloads):
    wl = workloads["cfg1"]
    cfgs = [nrsc5(s, wl.config) for s in (-100e3, 100e3)] + [dataclasses.replace(wl.config, output_format="cf32")]
    raw = synth_numpy(wl, 9 * CHUNK + 3)
    n = raw.size // 2
    chains = [gpu.Chain(c, 0) for c in cfgs]
    outs = [np.zeros(ch.out_capacity_frames(n) * ch.cfg.out_bytes, dtype=np.uint8) for ch in chains]
    caps = [o.nbytes for o in outs]
    caps[2] = 16                                             # channel 2 cannot take this call
    K = len(chains)
    rc = gpu.lib.iqgpu_chain_process_multi((C.c_void_p * K)(*[c._h for c in chains]), K, raw.ctypes.data, n, None, 0,
                                           (C.c_void_p * K)(*[o.ctypes.data for o in outs]), (C.c_size_t * K)(*caps),
                                           (C.c_size_t * K)(), None)
    assert rc == ECAPACITY and b"channel 2" in gpu.lib.iqgpu_last_error()
    assert all(c.info().frames_in_total == 0 and c.info().frames_out_total == 0 for c in chains)
    got = gpu.process_channels(chains, raw)
    for k, cfg in enumerate(cfgs):
        assert got[k].tobytes() == gpu.Chain(cfg, 0).process(raw).tobytes(), k


@pytest.mark.gpu
def test_raw_file_channels_equal_one_run_per_channel(gpu, workloads, tmp_path):
    wl = workloads["cfg1"]
    cfgs = [nrsc5(s, wl.config) for s in (-300e3, 100e3)] + [dataclasses.replace(wl.config, output_format="cs16", agc_enable=False)]
    raw = synth_numpy(wl, 45 * CHUNK + 999)
    src = tmp_path / "capture.cs16"
    src.write_bytes(raw.tobytes() + b"\x7f")
    multi = [tmp_path / f"m{k}.raw" for k in range(3)]
    st = gpu.rawfile_run_channels(cfgs, str(src), [str(p) for p in multi], train_chunks=16)
    for k, cfg in enumerate(cfgs):
        one = tmp_path / f"s{k}.raw"
        s1 = gpu.rawfile_run(cfg, str(src), str(one), train_chunks=16)
        assert multi[k].read_bytes() == one.read_bytes(), k
        assert (st[k].frames_in, st[k].frames_out, st[k].bytes_written, st[k].trains) == \
            (s1.frames_in, s1.frames_out, s1.bytes_written, s1.trains)


SDRC_XML = (b'<?xml version="1.0"?>\r\n<SDR-XML-Root xml:lang="EN" Description="Saved recording data" Created="04-Aug-2015 20:56">\r\n'
            b'<Definition CurrentTimeUTC="04-08-2015 20:56:28" Filename="x.wav" RadioModel="Airspy" '
            b"SoftwareName='SDR Console' SoftwareVersion=\"Version 3.0 build 1\" RadioCenterFreq=\"97300000\" "
            b'SampleRate="2000000" UTCSeconds="1438721788"/>\r\n</SDR-XML-Root>\r\n')


def _chunk(cid: bytes, body: bytes) -> bytes:
    return cid + struct.pack("<I", len(body)) + body + (b"\0" if len(body) & 1 else b"")


@pytest.mark.gpu
def test_wav_channels_with_centre_targets_equal_one_run_per_channel(gpu, workloads, tmp_path):
    """Three stations out of one SDR Console recording (centre 97.3 MHz): each output and its header equal a lone
    wavfile_run with that channel's centre target, each header with its own channel's rate."""
    wl = workloads["cfg1"]
    raw = synth_numpy(wl, 23 * CHUNK + 321)
    body = _chunk(b"fmt ", struct.pack("<HHIIHH", 1, 2, 2_000_000, 8_000_000, 4, 16)) + _chunk(b"auxi", SDRC_XML) \
        + _chunk(b"data", raw.tobytes())
    src = tmp_path / "rec.wav"
    src.write_bytes(b"RIFF" + struct.pack("<I", len(body) + 4) + b"WAVE" + body)
    base = dataclasses.replace(wl.config, freq_shift_hz=0.0, input_rate_hz=1.0)     # the header decides the rate
    cfgs = [base, dataclasses.replace(base, output_format="cs16", target_rate_hz=1e6, agc_enable=False),
            dataclasses.replace(base, output_format="cs16")]
    targets = [97.2e6, 97.45e6, 97.35e6]
    conts = [G.CONTAINER_WAV, G.CONTAINER_WAV, G.CONTAINER_RF64]
    multi = [tmp_path / f"m{k}.wav" for k in range(3)]
    st, info = gpu.wavfile_run_channels(cfgs, str(src), [str(p) for p in multi], out_containers=conts,
                                        center_targets_hz=targets, train_chunks=8)
    assert info.center_freq_hz == 97.3e6
    for k in range(3):
        one = tmp_path / f"s{k}.wav"
        s1, _ = gpu.wavfile_run(cfgs[k], str(src), str(one), out_container=conts[k], center_target_hz=targets[k], train_chunks=8)
        assert multi[k].read_bytes() == one.read_bytes(), k
        assert (st[k].frames_out, st[k].bytes_written) == (s1.frames_out, s1.bytes_written)
    with wave.open(str(multi[1]), "rb") as w:
        assert w.getframerate() == 1_000_000
    with wave.open(str(multi[0]), "rb") as w:
        assert w.getframerate() == 744187


@pytest.mark.gpu
def test_an_output_that_cannot_be_opened_fails_with_nothing_written(gpu, workloads, tmp_path):
    wl = workloads["cfg1"]
    src = tmp_path / "capture.cs16"
    src.write_bytes(synth_numpy(wl, 4 * CHUNK).tobytes())
    outs = [tmp_path / "a.raw", tmp_path / "missing_dir" / "b.raw", tmp_path / "c.raw"]
    cfgs = [nrsc5(s, wl.config) for s in (-100e3, 0.0, 100e3)]
    with pytest.raises(G.IqGpuError) as e:
        gpu.rawfile_run_channels(cfgs, str(src), [str(p) for p in outs])
    assert e.value.code == EINVAL and str(outs[1]) in str(e.value)
    assert not any(p.exists() for p in outs)
