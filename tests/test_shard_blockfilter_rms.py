"""Time-sharding of FFT-block-filter chains (block-aligned seek) and of RMS-AGC chains (end-state hand-over between
shards): shard plans on CPU (plan-only chains), shard-stitch parity on the GPU (`-m gpu`, ranks simulated one after the
other on cuda:0, one live chain per rank where the RMS rounds need it)."""
import dataclasses
import math

import numpy as np
import pytest

from iq_tool_b200.configs import AGC_DIGITAL, AGC_DX, AGC_LOCAL, FILTER_REQ_FFT, FILTER_REQ_FIR, ChainConfig, lowpass

CHUNK = 16384


def _with_digital_agc(cfg):
    return dataclasses.replace(cfg, agc_enable=True, agc_profile=AGC_DIGITAL)


def _rms_config(profile):
    """cu8 2.4 Msps -> 1 Msps cf32, no DC blocker, a 255-tap time-domain FIR: the AGC's input is the same bits sharded
    and single, so the hand-over alone decides whether the output is."""
    return ChainConfig(input_format="cu8", output_format="cf32", input_rate_hz=2.4e6, target_rate_hz=1e6,
                       freq_shift_hz=50e3, filters=[lowpass(400e3)], filter_taps=255, filter_type_request=FILTER_REQ_FIR,
                       agc_enable=True, agc_profile=profile)


def _plan_configs(workloads):
    return {"cfg3": workloads["cfg3"].config, "cfg4": workloads["cfg4"].config,
            "cfg3_digital": _with_digital_agc(workloads["cfg3"].config)}


# ------------------------------------------------------------------------------------------------
# CPU: shard plans
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,total", [("cfg3", 300 * CHUNK + 4321), ("cfg4", 900 * CHUNK + 17), ("cfg3_digital", 64 * CHUNK)])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_block_filter_and_rms_shard_plans_tile_the_capture(name, total, world, workloads):
    from iq_tool_b200 import gpu
    from iq_tool_b200.shard import plan_shards
    cfg = _plan_configs(workloads)[name]
    probe = gpu.Chain(cfg, -1)
    info = probe.info()
    fft = info.filter_impl in (3, 4)              # IQGPU_FILTER_IMPL_FFT_SYM / _ASYM (include/iqgpu.h)
    assert fft == name.startswith("cfg3")
    halo = probe.halo_frames()
    if fft:
        # two blocks of the filter behind the resampler's exact region
        assert halo >= math.ceil(2 * info.filter_block_size / cfg.ratio)
    shards = plan_shards(probe, total, world)
    assert shards[0].start == 0 and shards[0].lead == 0 and shards[0].drop == 0
    assert sum(s.frames for s in shards) == total
    for a, b in zip(shards[:-1], shards[1:]):
        assert a.start + a.frames == b.start and a.out_end == b.out_start
        assert b.start - b.lead >= min(halo, b.start) and b.skip_chunks * CHUNK == b.start - b.lead
        assert b.out_lead <= b.out_start
    assert shards[-1].out_end == probe.predict_output(total)
    for s in shards:
        if fft:
            n = info.filter_block_size
            assert s.out_lead % n == 0 and s.out_start % n == 0 and s.out_end % n == 0
        assert gpu.Chain(cfg, -1).seek(s.lead) == s.out_lead      # seek accepts the chain and lands on the plan


def test_outputs_after_is_the_block_quantised_resampler_count(workloads):
    from iq_tool_b200 import gpu
    ks = [0, 1, 5000, CHUNK, 3 * CHUNK + 11, 1_000_003, 77 * CHUNK + 5, 50_000_000]
    for name, wl in workloads.items():
        probe = gpu.Chain(wl.config, -1)
        info = probe.info()
        for k in ks:
            r = probe.resampler_outputs_after(k)
            got = probe.outputs_after(k)
            assert got == gpu.Chain(wl.config, -1).predict_output(k), (name, k)
            if info.filter_impl in (3, 4):
                assert got == r - r % info.filter_block_size
            else:
                assert got == r, (name, k)


@pytest.mark.parametrize("name,total", [("cfg1", 40 * CHUNK + 777), ("cfg2", 1000 * CHUNK), ("cfg5", 257 * CHUNK + 1)])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_plans_without_block_filter_are_unchanged(name, total, world, workloads):
    """Chains without an FFT filter: the plan's output indices are the resampler's closed form, as they always were."""
    from iq_tool_b200 import gpu
    from iq_tool_b200.shard import plan_shards
    probe = gpu.Chain(workloads[name].config, -1)
    halo = probe.halo_frames()
    halo += (-halo) % CHUNK
    n_chunks = (total + CHUNK - 1) // CHUNK
    base, extra = divmod(n_chunks, world)
    c0 = 0
    for r, s in enumerate(plan_shards(probe, total, world)):
        nc = base + (1 if r < extra else 0)
        start, end = min(c0 * CHUNK, total), min((c0 + nc) * CHUNK, total)
        lead = max(0, start - halo)
        assert (s.start, s.frames, s.lead, s.skip_chunks) == (start, end - start, lead, (start - lead) // CHUNK)
        assert (s.out_lead, s.out_start, s.out_end) == tuple(probe.resampler_outputs_after(v) for v in (lead, start, end))
        c0 += nc


def test_seek_refuses_a_pre_resample_fft_filter():
    from iq_tool_b200 import gpu
    # no_resample keeps the filter in front of the (absent) resampler
    cfg = ChainConfig(input_format="cs16", output_format="cs16", input_rate_hz=1e6, target_rate_hz=1e6, no_resample=True,
                      filters=[lowpass(100e3)], filter_taps=1023, filter_type_request=FILTER_REQ_FFT)
    probe = gpu.Chain(cfg, -1)
    info = probe.info()
    assert info.filter_impl in (3, 4) and info.filter_post_resample == 0
    with pytest.raises(gpu.IqGpuError, match="pre-resample FFT filter"):
        probe.seek(CHUNK)


def test_rms_chain_seeks():
    from iq_tool_b200 import gpu
    for profile in (AGC_LOCAL, AGC_DX):
        probe = gpu.Chain(_rms_config(profile), -1)
        assert probe.seek(4 * CHUNK) == probe.outputs_after(4 * CHUNK)


# ------------------------------------------------------------------------------------------------
# GPU: shard-stitch parity
# ------------------------------------------------------------------------------------------------
def _single(gpu, cfg, raw, subtrain=0):
    import torch
    opts = {"subtrain_frames": subtrain} if subtrain else {}
    ch = gpu.Chain(cfg, 0, **opts)
    total = raw.numel() * raw.element_size() // cfg.in_bytes
    out = torch.zeros(ch.out_capacity_frames(total) * cfg.out_bytes, dtype=torch.uint8, device=raw.device)
    n = ch.process_device(raw.data_ptr(), total, out.data_ptr(), out.numel())
    torch.cuda.synchronize()
    return out[: n * cfg.out_bytes]


def _sharded(gpu, cfg, raw, world, changed_log=None):
    """`raw` (device tensor) as `world` time shards, one rank after the other on cuda:0.  Digital AGC: the device-side peak
    exchange (lower shards' peaks from a gathered buffer).  RMS AGC: one live chain per rank, then the world-1 hand-over
    rounds (all ranks publish their end states into one gathered buffer, then every rank resumes)."""
    import torch
    from iq_tool_b200.shard import ShardedChain, lower_shard_pieces
    dev = raw.device
    total = raw.numel() * raw.element_size() // cfg.in_bytes
    base = raw.data_ptr()
    probe_sc = ShardedChain(cfg, 0, shard_frames_hint=total // world + CHUNK)
    shards = probe_sc.plan(total, world)
    rms = probe_sc.rms_agc
    scs = [probe_sc] + [ShardedChain(cfg, 0, shard_frames_hint=total // world + CHUNK) for _ in range(world - 1)] if rms \
        else [probe_sc] * world
    m = max((sh.frames + CHUNK - 1) // CHUNK for sh in shards)
    gathered = torch.zeros(world * max(m, 1), dtype=torch.float32, device=dev)
    outs, produced = [], []
    for sh, sc in zip(shards, scs):
        ch = sc.chain
        assert ch.seek(sh.lead) == sh.out_lead
        out = torch.zeros(ch.out_capacity_frames(sh.read_frames) * cfg.out_bytes, dtype=torch.uint8, device=dev)
        ptr = base + sh.lead * cfg.in_bytes
        if sc.digital_agc:
            ch.process_device_begin(ptr, sh.read_frames)
            mine = gathered[sh.rank * m: sh.rank * m + m]
            assert ch.pending_chunk_peaks_device(sh.skip_chunks, mine.data_ptr(), m) == (sh.frames + CHUNK - 1) // CHUNK
            for p, first, frames in lower_shard_pieces(shards, sh.rank, m, gathered.data_ptr(), sc.lock_frames):
                ch.agc_advance_device(p, first, frames)
            k = ch.process_device_finish(sh.skip_chunks, out.data_ptr(), out.numel())
        else:
            k = ch.process_device(ptr, sh.read_frames, out.data_ptr(), out.numel())
        torch.cuda.synchronize()
        assert k - sh.drop == sh.out_frames
        outs.append(out)
        produced.append(k)
    if rms:
        states = torch.zeros(2 * world, dtype=torch.float32, device=dev)
        changed = torch.zeros((max(world - 1, 1), world), dtype=torch.int32, device=dev)
        for rnd in range(world - 1):
            for sh, sc in zip(shards, scs):
                sc.chain.agc_rms_state_device(states[2 * sh.rank:].data_ptr())
            torch.cuda.synchronize()
            for sh, sc, out in zip(shards, scs, outs):
                sc.rms_resume(sh, states.data_ptr(), out.data_ptr(), out.numel(), changed_ptr=changed[rnd, sh.rank:].data_ptr())
            torch.cuda.synchronize()
        if changed_log is not None:
            changed_log.append(changed.cpu().numpy())
    parts = [out[sh.drop * cfg.out_bytes: k * cfg.out_bytes] for sh, out, k in zip(shards, outs, produced)]
    return torch.cat(parts)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_cfg3_equals_single_stream_byte_for_byte(world, gpu, workloads):
    """cfg3 (4095-tap band-pass in the FFT block filter behind the resampler, post shift): the shards cut the single
    stream's blocks (block-aligned seek) and the halo covers two blocks, so the stitched cs16 output is the same bytes."""
    from iq_tool_b200.synth import synth_torch
    wl = workloads["cfg3"]
    raw = synth_torch(wl, 1 << 23, "cuda")
    single = _single(gpu, wl.config, raw)
    sharded = _sharded(gpu, wl.config, raw, world)
    assert sharded.numel() == single.numel()
    assert bool((sharded == single).all())


@pytest.mark.gpu
def test_sharded_cfg3_with_digital_agc_equals_single_stream(gpu, workloads):
    """cfg3 + digital AGC through the device peak exchange: the per-chunk frame counts of the lower shards are the FFT
    filter's block-quantised counts, so the state each shard starts from is the single stream's.  2^27 frames (13 s of
    output) let the AGC lock (2 s) and ratchet on a loud stretch in the last shard."""
    import torch
    from iq_tool_b200.synth import synth_torch
    wl = workloads["cfg3"]
    cfg = _with_digital_agc(wl.config)
    total = 1 << 27
    raw = synth_torch(wl, total, "cuda")
    h = total - total // 6
    seg = raw[2 * h: 2 * (h + 64 * CHUNK)]
    raw[2 * h: 2 * (h + 64 * CHUNK)] = torch.clamp(seg.to(torch.int32) * 3, -32768, 32767).to(torch.int16)
    single = _single(gpu, cfg, raw, subtrain=total + CHUNK)
    sharded = _sharded(gpu, cfg, raw, 3)
    assert sharded.numel() == single.numel()
    assert bool((sharded == single).all())


def _rms_capture(n, seed):
    """cu8 frames: two tones and noise, with quiet and loud stretches for the AGC to follow."""
    import torch
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    env = np.ones(n)
    env[n // 5: 2 * n // 5] = 0.15
    env[3 * n // 5: 3 * n // 5 + n // 10] = 2.5
    x = env * (0.25 * np.exp(2j * np.pi * 0.083 * t) + 0.08 * np.exp(-2j * np.pi * 0.125 * t))
    x = x + 0.01 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    raw = np.empty(2 * n, dtype=np.uint8)
    raw[0::2] = np.clip(np.rint(127.5 + 127.0 * x.real), 0, 255)
    raw[1::2] = np.clip(np.rint(127.5 + 127.0 * x.imag), 0, 255)
    return torch.from_numpy(raw).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("profile,chunks,world", [(AGC_LOCAL, 120, 3), (AGC_LOCAL, 64, 8), (AGC_DX, 200, 2), (AGC_DX, 32, 8)])
def test_sharded_rms_agc_equals_single_stream_byte_for_byte(profile, chunks, world, gpu):
    """RMS AGC with the same AGC input sharded and single: after the world-1 hand-over rounds the cf32 output is the single
    stream's, bit for bit.  DX on 32 chunks / 8 ranks: a shard (4 chunks, 27 k outputs) is far shorter than the DX loop's
    merge time (time constant 2/alpha = 20 k samples), so a changed start state changes the end state too and has to travel
    on through the ranks behind it — the case that needs every round."""
    cfg = _rms_config(profile)
    raw = _rms_capture(chunks * CHUNK - 999, seed=chunks)
    single = _single(gpu, cfg, raw)
    log = []
    sharded = _sharded(gpu, cfg, raw, world, changed_log=log)
    assert sharded.numel() == single.numel()
    assert bool((sharded == single).all())
    changed = log[0]
    if profile == AGC_DX and world == 8:
        assert changed[0, 1:].all()                # round 1: every resumed rank's end state moved
        # round r >= 2 resumes rank g from a state that changed in round r-1: the change crossed more than one rank
        assert changed[1:, 2:].any()
        assert changed[world - 2, world - 1] == 1
    if profile == AGC_LOCAL:
        assert not changed[1:].any()               # shards longer than the merge time: one round settles every rank


@pytest.mark.gpu
def test_sharded_cfg4_meets_the_bar(gpu, workloads):
    """cfg4 (DC block, I/Q apply, notch FIR through the FFT block kernel, LOCAL AGC) sharded against single.  Not exact:
    the DC blocker's state is rebuilt by a 16-time-constant halo and the FIR-via-FFT blocks sit at other positions
    relative to the shard; the AGC hand-over itself is exact.  Bar: 1e-5 relative RMS (100 dB SNR); measured on a B200:
    2.45e-6 (112.2 dB) on these 2^24 frames in four shards, asserted with a small margin."""
    import torch
    from iq_tool_b200.synth import synth_torch
    wl = workloads["cfg4"]
    cfg = wl.config
    raw = synth_torch(wl, 1 << 24, "cuda")
    single = _single(gpu, cfg, raw).view(torch.float32).double()
    sharded = _sharded(gpu, cfg, raw, 4).view(torch.float32).double()
    assert sharded.numel() == single.numel()
    rel = float(torch.sqrt(torch.mean((sharded - single) ** 2) / torch.mean(single ** 2)))
    snr_db = -20.0 * math.log10(max(rel, 1e-30))
    print(f"cfg4 sharded vs single: relative RMS {rel:.3e}, SNR {snr_db:.1f} dB")
    assert rel <= 4e-6 and snr_db >= 108.0


def _rms_gloo_worker(rank, world, port, profile, chunks):
    import os
    import torch
    import torch.distributed as dist
    from iq_tool_b200 import gpu
    from iq_tool_b200.shard import ShardedChain
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        cfg = _rms_config(profile)
        raw = _rms_capture(chunks * CHUNK - 999, seed=chunks)
        total = raw.numel() // 2
        single = _single(gpu, cfg, raw)
        sc = ShardedChain(cfg, 0, shard_frames_hint=total // world + CHUNK)
        sh = sc.plan(total, world)[rank]
        out = torch.zeros(sc.chain.out_capacity_frames(sh.read_frames) * cfg.out_bytes, dtype=torch.uint8, device="cuda")
        produced, drop = sc.process_device(sh, raw.data_ptr() + sh.lead * cfg.in_bytes, out.data_ptr(), out.numel())
        torch.cuda.synchronize()
        b = cfg.out_bytes
        assert produced - drop == sh.out_frames
        assert bool((out[drop * b: produced * b] == single[sh.out_start * b: sh.out_end * b]).all())
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_rms_handover_over_gloo_through_sharded_chain(gpu):
    """ShardedChain.process_device itself (host form of the rounds: end states through a gloo group) with three ranks on
    one GPU: every rank's owned output equals the single stream's slice, bit for bit (DX, shards shorter than the merge
    time, so the third rank needs the second round)."""
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_rms_gloo_worker, args=(3, port, AGC_DX, 12), nprocs=3, join=True)
