"""Time-sharding of a long capture across the GPUs of one box (SURVEY.md §8(e), DESIGN.md §5).

A capture of `total_frames` input frames is cut into contiguous shards whose starts are
multiples of the reference chunk (16384 frames, include/constants.h:123), so that chunk
boundaries — and with them the per-chunk digital-AGC blocks — are those of the single stream.
Everything that positions a shard is closed-form integer arithmetic (NCO phase, halfband
pairing, polyphase phase, FFT-filter block position, output index: `iqgpu_chain_seek`,
`iqgpu_chain_outputs_after`); finite-memory filter state is rebuilt by re-processing a halo in
front of the shard and dropping its outputs.

The AGC is the only data-dependent exchange, and no sample data crosses GPUs:
- the digital AGC (src/agc.c:105-222) is a scalar state machine over per-chunk peaks, so a shard
  needs the state left by all earlier chunks.  The ranks all-gather their per-chunk peaks
  (4 bytes per 16384 input frames) and each replays the state machine over the chunks that
  precede its shard (`exchange_agc_state`, or on the device);
- the RMS AGC (liquid agc_crcf) is a per-sample recurrence in {g, y2'}.  Every shard runs it from
  the reset state at its lead, then `world - 1` rounds follow: the ranks all-gather their end
  states (8 bytes each) and rank g >= 1 resumes its AGC at its first owned output from rank
  g-1's end state.  After round k ranks 0..k are exact; a resume whose start state did not change
  is a no-op on the device, so once the shards are longer than the recurrence's merge time the
  later rounds cost only their collectives.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

from . import gpu
from .configs import AGC_DIGITAL, AGC_DX, AGC_LOCAL, CHUNK_SAMPLES


@dataclass
class Shard:
    rank: int
    world: int
    start: int          # first input frame the shard owns
    frames: int         # input frames owned
    lead: int           # first input frame the rank reads (start - halo, chunk aligned, >= 0)
    skip_chunks: int    # whole reference chunks in [lead, start): the halo
    out_lead: int       # absolute output index of the first frame the chain emits from `lead`
    out_start: int      # absolute output index of the first frame the shard owns
    out_end: int        # one past the last output frame the shard owns

    @property
    def read_frames(self) -> int:
        return self.start - self.lead + self.frames

    @property
    def drop(self) -> int:
        """outputs produced from the halo, to be discarded"""
        return self.out_start - self.out_lead

    @property
    def out_frames(self) -> int:
        return self.out_end - self.out_start


def plan_shards(chain: "gpu.Chain", total_frames: int, world: int, halo_frames: Optional[int] = None,
                chunk: int = CHUNK_SAMPLES) -> List[Shard]:
    """Cut [0, total_frames) into `world` chunk-aligned shards.  `chain` may be plan-only
    (device=-1): only closed forms are used."""
    if world < 1 or total_frames < 0:
        raise ValueError("bad shard request")
    halo = chain.halo_frames() if halo_frames is None else int(halo_frames)
    halo += (-halo) % chunk
    n_chunks = (total_frames + chunk - 1) // chunk
    base, extra = divmod(n_chunks, world)
    shards, c0 = [], 0
    for r in range(world):
        nc = base + (1 if r < extra else 0)
        start = min(c0 * chunk, total_frames)
        end = min((c0 + nc) * chunk, total_frames)
        lead = max(0, start - halo)
        shards.append(Shard(rank=r, world=world, start=start, frames=end - start, lead=lead,
                            skip_chunks=(start - lead) // chunk,
                            out_lead=chain.outputs_after(lead),
                            out_start=chain.outputs_after(start),
                            out_end=chain.outputs_after(end)))
        c0 += nc
    return shards


def _all_gather_var(arr: np.ndarray, group, device) -> List[np.ndarray]:
    """all_gather of per-rank 1-D arrays of different lengths (float32 / uint32 payloads)."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    n = torch.tensor([arr.size], dtype=torch.int64, device=device)
    got = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(got, n, group=group)
    sizes = [int(v) for v in torch.cat(got).cpu().tolist()]
    m = max(max(sizes), 1)
    host = np.zeros(m, dtype=np.int32)
    host[: arr.size] = arr.view(np.int32)
    out = torch.empty(world * m, dtype=torch.int32, device=device)
    dist.all_gather_into_tensor(out, torch.from_numpy(host).to(device), group=group)
    tab = out.cpu().numpy().reshape(world, m)
    return [tab[r, : sizes[r]].view(arr.dtype) for r in range(world)]


def _all_gather_tables(peaks: np.ndarray, counts: np.ndarray, group, device, sizes=None):
    """all_gather of every rank's (peaks float32[n_r], counts uint32[n_r]) chunk tables in ONE payload collective.
    `sizes` = the per-rank table lengths when the caller knows them (they follow from the shard plan); otherwise one
    small all_gather of the lengths comes first."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    if sizes is None:
        n = torch.tensor([peaks.size], dtype=torch.int64, device=device)
        got = [torch.zeros_like(n) for _ in range(world)]
        dist.all_gather(got, n, group=group)
        sizes = [int(v) for v in torch.cat(got).cpu().tolist()]
    assert len(sizes) == world and sizes[dist.get_rank(group)] == peaks.size == counts.size
    m = max(max(sizes), 1)
    host = np.zeros(2 * m, dtype=np.int32)
    host[: peaks.size] = peaks.view(np.int32)
    host[m: m + counts.size] = counts.view(np.int32)
    buf = torch.from_numpy(host).to(device)
    out = torch.empty(world * 2 * m, dtype=torch.int32, device=device)
    dist.all_gather_into_tensor(out, buf, group=group)
    tab = out.cpu().numpy().reshape(world, 2, m)
    return ([tab[r, 0, : sizes[r]].view(np.float32) for r in range(world)],
            [tab[r, 1, : sizes[r]].view(np.uint32) for r in range(world)])


def exchange_agc_state(peaks: np.ndarray, counts: np.ndarray, target: float, target_rate_hz: float,
                       group=None, device="cpu", sizes=None) -> "gpu.AgcStateC":
    """Digital-AGC state at the start of this rank's shard: all-gather every rank's live per-chunk
    peaks/counts and replay the state machine over the chunks of the ranks below this one."""
    import torch.distributed as dist

    rank = dist.get_rank(group)
    all_peaks, all_counts = _all_gather_tables(np.ascontiguousarray(peaks, dtype=np.float32),
                                               np.ascontiguousarray(counts, dtype=np.uint32), group, device, sizes)
    state = gpu.agc_initial_state()
    if rank:
        # one replay over the concatenated tables of the ranks below (the state machine is sequential in the chunks)
        gpu.agc_digital_advance(state, target, target_rate_hz, np.concatenate(all_peaks[:rank]), np.concatenate(all_counts[:rank]))
    return state


def lower_shard_pieces(shards: List[Shard], rank: int, m: int, base_ptr: int, lock_frames: int):
    """The scan calls that advance rank `rank`'s digital-AGC state over the shards below it: [device pointer, first frame,
    frames] per call.  `base_ptr` is the gathered peak buffer (float32, rank r's live chunks at element r*m)."""
    pieces = []
    for r in range(rank):
        sh_r = shards[r]
        if not sh_r.frames:
            continue
        ptr, first, frames = base_ptr + 4 * r * m, sh_r.start, sh_r.frames
        if sh_r.start < lock_frames < sh_r.start + sh_r.frames and (lock_frames - sh_r.start) % CHUNK_SAMPLES == 0:
            head = lock_frames - sh_r.start
            pieces.append([ptr, first, head])
            pieces.append([ptr + 4 * (head // CHUNK_SAMPLES), first + head, frames - head])
            continue
        last = pieces[-1] if pieces else None
        if (last is not None and last[1] >= lock_frames and last[2] % CHUNK_SAMPLES == 0 and
                last[1] + last[2] == first and last[0] + 4 * (last[2] // CHUNK_SAMPLES) == ptr):
            last[2] += frames
        else:
            pieces.append([ptr, first, frames])
    return pieces


class ShardedChain:
    """One rank's chain of a time-sharded run.  `process_device` reads the rank's frames
    [shard.lead, shard.start + shard.frames) from device memory and writes the converted output
    of that range; the first `shard.drop` output frames belong to the halo."""

    def __init__(self, cfg, device: int, shard_frames_hint: int = 0, **options):
        opts = dict(options)
        self.cfg = cfg
        self.digital_agc = bool(cfg.agc_enable and cfg.agc_profile == AGC_DIGITAL)
        self.rms_agc = bool(cfg.agc_enable and cfg.agc_profile in (AGC_DX, AGC_LOCAL))
        self.device = device
        self._probe = gpu.Chain(cfg, -1)
        halo = self._probe.halo_frames()
        halo += (-halo) % CHUNK_SAMPLES
        self.halo = halo
        if (self.digital_agc or self.rms_agc) and shard_frames_hint:
            # the shard's call must be one sub-train: the AGC's input (and for the RMS AGC its output and checkpoints) is
            # kept on the device across the exchange
            opts["subtrain_frames"] = max(int(opts.get("subtrain_frames", 0)), shard_frames_hint + halo + CHUNK_SAMPLES)
        self.chain = gpu.Chain(cfg, device, **opts)
        self.agc_target = cfg.agc_target_level_arg if cfg.agc_target_level_arg > 0 else 0.9   # agc.c:108-110, constants.h:184
        self.target_rate = float(np.float32(cfg.target_rate_hz))
        # input frames (whole chunks) after which the digital AGC is certainly locked: more than 2 s of output samples
        # (agc.c:145-149) plus two chunks of slack.  Output counts are the chain's (outputs_after): an FFT filter's block
        # lag (n output frames, several chunks at cfg3's rates) is part of them.
        lock_out = int(2.0 * self.target_rate) + 2
        k = 0
        if self.digital_agc:
            step = max(1, int(lock_out / max(cfg.ratio, 1e-9)) // CHUNK_SAMPLES)
            while self._probe.outputs_after(k * CHUNK_SAMPLES) <= lock_out:
                k += step if self._probe.outputs_after((k + step) * CHUNK_SAMPLES) <= lock_out else 1
        self.lock_frames = (k + 2) * CHUNK_SAMPLES

    def plan(self, total_frames: int, world: int) -> List[Shard]:
        shards = plan_shards(self._probe, total_frames, world, self.halo)
        # live chunks per rank: the lengths of the tables the ranks exchange (no length exchange needed at run time)
        self._table_sizes = {(s.world, s.rank, s.start, s.frames): [(t.frames + CHUNK_SAMPLES - 1) // CHUNK_SAMPLES for t in shards]
                             for s in shards}
        self._plans = {(s.world, s.rank, s.start, s.frames): shards for s in shards}
        return shards

    def _exchange_buffers(self, world: int, m: int, device):
        import torch
        key = (world, m, str(device))
        bufs = getattr(self, "_xbufs", None)
        if bufs is None or bufs[0] != key:
            bufs = (key, torch.zeros(m, dtype=torch.float32, device=device),
                    torch.zeros(world * m, dtype=torch.float32, device=device))
            self._xbufs = bufs
        return bufs[1], bufs[2]

    @staticmethod
    def _on_stream(stream: int):
        """torch's current stream must be the stream the chain runs on: the copy of the peaks into the send buffer, the
        all-gather and the scan kernel that reads the gathered buffer are ordered by that one stream (ADVICE r1)."""
        import torch
        if not stream:
            raise ValueError("the device-side AGC exchange needs an explicit CUDA stream (stream=0 would leave the chain on "
                             "its private stream and the collective on torch's: unordered)")
        return torch.cuda.stream(torch.cuda.ExternalStream(stream))

    def _finish_device_exchange(self, shard: Shard, shards: List[Shard], dev_out_ptr: int, out_capacity_bytes: int,
                                stream: int, group, device) -> int:
        """The digital-AGC exchange without a host round trip: the shard's per-chunk peaks go from the chain into the
        send buffer of ONE all-gather (NCCL over NVLink), and every rank advances its device-resident AGC state over the
        lower ranks' slices of the gathered buffer with the chunk-table scan kernel (chunk frame counts are closed
        form), then finishes its own shard.  Same kernel, same chunks, same order as the single stream -> same bits.

        A rank whose shard is empty (more ranks than chunks) takes part in the same collective with a zero-filled send
        buffer, so that every rank issues the same sequence of collectives."""
        import torch.distributed as dist

        ch = self.chain
        sizes = [(t.frames + CHUNK_SAMPLES - 1) // CHUNK_SAMPLES for t in shards]
        m = max(max(sizes), 1)
        mine, gathered = self._exchange_buffers(shard.world, m, device)
        marks = getattr(self, "exchange_marks", None)        # optional: CUDA events around the exchange (bench diagnostics)

        def mark():
            if marks is not None:
                import torch
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(torch.cuda.current_stream())
                marks[-1].append(ev)

        with self._on_stream(stream):
            if marks is not None:
                marks.append([])
            mark()                                            # front + peaks queued before this point
            if shard.read_frames:
                live = ch.pending_chunk_peaks_device(shard.skip_chunks, mine.data_ptr(), m, stream)
                assert live == sizes[shard.rank]
            else:
                mine.zero_()
            dist.all_gather_into_tensor(gathered, mine, group=group)
            mark()                                            # all-gather done (includes waiting for the slowest rank)
            if not shard.read_frames:
                return 0
            # Lower shards, in rank order, as few scan launches as possible: pieces of the gathered buffer that are contiguous
            # in memory AND in the capture (full tables of whole chunks) go in ONE call — a locked, quiet stretch is then
            # settled by the grid-wide quiet test in a few microseconds however long it is.  The head of the capture (until the
            # AGC locks, 2 s of output samples, agc.c:145-149) is a piece of its own: it needs the sequential tile walk.
            pieces = lower_shard_pieces(shards, shard.rank, m, gathered.data_ptr(), self.lock_frames)
            for ptr, first, frames in pieces:
                ch.agc_advance_device(ptr, first, frames, stream)
            mark()                                            # state advanced over the lower shards
            produced = ch.process_device_finish(shard.skip_chunks, dev_out_ptr, out_capacity_bytes, stream)
            mark()                                            # own scan + scale + convert
            return produced

    def rms_resume(self, shard: Shard, gathered_ptr: int, dev_out_ptr: int, out_capacity_bytes: int, stream: int = 0,
                   changed_ptr: int = 0) -> None:
        """One round of the RMS-AGC hand-over on this rank, after the all-gather: `gathered_ptr` holds every rank's end
        state ({g, y2'} float32 pairs in rank order, device memory); rank g >= 1 resumes from rank g-1's."""
        if shard.rank and shard.read_frames:
            self.chain.agc_rms_resume_device(shard.drop, gathered_ptr + 8 * (shard.rank - 1), dev_out_ptr,
                                             out_capacity_bytes, changed_ptr, stream)

    def _rms_rounds(self, shard: Shard, dev_out_ptr: int, out_capacity_bytes: int, stream: int, group, device) -> None:
        """The `world - 1` rounds of the RMS-AGC hand-over.  On a CUDA communication device everything is queued on the
        chain's stream without a host synchronisation (8-byte all-gathers over NCCL); otherwise the states travel through
        the host over any torch.distributed group.  A rank with an empty shard sends zeros (it is the last with data
        behind it) and takes part in every collective."""
        import torch
        import torch.distributed as dist

        ch, world = self.chain, shard.world
        if str(device).startswith("cuda"):
            key = (world, str(device))
            bufs = getattr(self, "_rms_bufs", None)
            if bufs is None or bufs[0] != key:
                bufs = (key, torch.zeros(2, dtype=torch.float32, device=device),
                        torch.zeros(2 * world, dtype=torch.float32, device=device))
                self._rms_bufs = bufs
            mine, gathered = bufs[1], bufs[2]
            with self._on_stream(stream):
                for _ in range(world - 1):
                    if shard.read_frames:
                        ch.agc_rms_state_device(mine.data_ptr(), stream)
                    else:
                        mine.zero_()
                    dist.all_gather_into_tensor(gathered, mine, group=group)
                    self.rms_resume(shard, gathered.data_ptr(), dev_out_ptr, out_capacity_bytes, stream)
            return
        for _ in range(world - 1):
            mine = torch.tensor(ch.get_agc_rms_state() if shard.read_frames else (0.0, 0.0), dtype=torch.float32)
            got = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(got, mine, group=group)
            # kept alive on the object: the resume reads it asynchronously on the chain's stream
            self._rms_host_state = torch.cat(got).to(torch.device("cuda", self.device))
            torch.cuda.synchronize(self.device)           # a copy from pageable memory may still be in flight on return
            self.rms_resume(shard, self._rms_host_state.data_ptr(), dev_out_ptr, out_capacity_bytes, stream)

    def process_device(self, shard: Shard, dev_in_ptr: int, dev_out_ptr: int, out_capacity_bytes: int,
                       stream: int = 0, group=None, comm_device="cpu") -> Tuple[int, int]:
        """Returns (frames written, frames to drop from the front)."""
        ch = self.chain
        out_lead = ch.seek(shard.lead)
        assert out_lead == shard.out_lead
        n = shard.read_frames
        if self.rms_agc and shard.world > 1:
            produced = ch.process_device(dev_in_ptr, n, dev_out_ptr, out_capacity_bytes, stream) if n else 0
            self._rms_rounds(shard, dev_out_ptr, out_capacity_bytes, stream, group, comm_device)
            return produced, shard.drop
        exchange = self.digital_agc and shard.world > 1
        plan = getattr(self, "_plans", {}).get((shard.world, shard.rank, shard.start, shard.frames))
        sizes = getattr(self, "_table_sizes", {}).get((shard.world, shard.rank, shard.start, shard.frames))
        on_device = exchange and plan is not None and str(comm_device).startswith("cuda")
        if n == 0:
            # an empty shard (more ranks than chunks) still takes part in the exchange, in the form its peers use
            if on_device:
                self._finish_device_exchange(shard, plan, dev_out_ptr, out_capacity_bytes, stream, group, comm_device)
            elif exchange:
                exchange_agc_state(np.zeros(0, np.float32), np.zeros(0, np.uint32), self.agc_target,
                                   self.target_rate, group, comm_device, sizes)
            return 0, 0
        if not exchange:
            return ch.process_device(dev_in_ptr, n, dev_out_ptr, out_capacity_bytes, stream), shard.drop
        ch.process_device_begin(dev_in_ptr, n, stream)
        if on_device:
            return self._finish_device_exchange(shard, plan, dev_out_ptr, out_capacity_bytes, stream, group, comm_device), shard.drop
        peaks, counts = ch.pending_chunk_peaks()
        state = exchange_agc_state(peaks[shard.skip_chunks:], counts[shard.skip_chunks:], self.agc_target,
                                   self.target_rate, group, comm_device, sizes)
        ch.set_agc_state(state)
        produced = ch.process_device_finish(shard.skip_chunks, dev_out_ptr, out_capacity_bytes, stream)
        return produced, shard.drop
