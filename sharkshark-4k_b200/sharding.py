"""Multi-GPU sharding of the hot path: one process per GPU, no collective inside the nets.

SURVEY.md section 8e: the upscalers are stateless per frame -> frames shard freely; the BSVD denoiser has a
temporal receptive field of exactly +-16 frames (16 BiBufferConvs, src/upscale/model/bsvd/model.py:582-588), so a
contiguous chunk plus a 16-frame halo on each side reproduces the single-stream result.  The only exchange step is
the gather of the finished uint8 frames to the encoder rank (the reference's streamer process,
src/stream/streamer.py:66-153), in stream order.
"""
from dataclasses import dataclass

import torch
import torch.distributed as dist

BSVD_HALO = 16


@dataclass
class Chunk:
    lo: int        # first owned frame
    hi: int        # one past the last owned frame
    load_lo: int   # first frame that has to be decoded / denoised (owned range + temporal halo, clipped to the clip)
    load_hi: int

    @property
    def owned(self):
        """slice of the locally denoised clip that holds the owned frames"""
        return slice(self.lo - self.load_lo, self.hi - self.load_lo)


def frame_shards(n_frames, world):
    """Contiguous, balanced frame ranges [lo, hi) per rank (sizes differ by at most one)."""
    base, rem = divmod(n_frames, world)
    out, lo = [], 0
    for r in range(world):
        hi = lo + base + (1 if r < rem else 0)
        out.append((lo, hi))
        lo = hi
    return out


def bsvd_chunks(n_frames, world, halo=BSVD_HALO):
    """Per-rank chunk with the temporal halo the denoiser needs on each side."""
    return [Chunk(lo, hi, max(0, lo - halo), min(n_frames, hi + halo)) for lo, hi in frame_shards(n_frames, world)]


def gather_frames(local, n_frames, dst=0, group=None):
    """Gather every rank's finished frames [n_local, ...] to ``dst`` in stream order.  Returns the full clip on
    ``dst`` and None elsewhere.  Ranks may own different frame counts: shards are padded to the largest.  Shape- and
    dtype-generic past the frame dimension: uint8 RGB [n, H, W, 3], packed NV12 [n, H*3/2, W] (half the bytes) or float
    frames gather the same way."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    shards = frame_shards(n_frames, world)
    biggest = max(hi - lo for lo, hi in shards)
    pad = torch.zeros((biggest,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[:local.shape[0]] = local
    bufs = [torch.empty_like(pad) for _ in range(world)] if rank == dst else None
    dist.gather(pad, bufs, dst=dst, group=group)
    if rank != dst:
        return None
    return torch.cat([bufs[r][:hi - lo] for r, (lo, hi) in enumerate(shards)], dim=0)


class StreamChunker:
    """Chunk + halo bookkeeping for a LIVE (unbounded) stream: frames arrive one batch after another, chunk k owns
    frames [k L, (k+1) L) and goes to GPU k % world; it can be dispatched as soon as its trailing halo has arrived
    (frame (k+1) L + halo - 1), i.e. the sharded denoiser adds L + halo frames of latency, not a whole clip.  At the
    end of the stream the last chunks are clipped to the frames that exist (zero features beyond the clip, like the
    reference's drain, src/upscale/model/bsvd/model.py:555-569)."""

    def __init__(self, world, chunk_len, halo=BSVD_HALO):
        assert world >= 1 and chunk_len >= 1 and halo >= 0
        self.world, self.chunk_len, self.halo = world, chunk_len, halo
        self.frames = 0        # frames received so far
        self.next_chunk = 0    # first chunk not dispatched yet
        self.closed = False

    def _chunk(self, k, total):
        lo, hi = k * self.chunk_len, min((k + 1) * self.chunk_len, total)
        return Chunk(lo, hi, max(0, lo - self.halo), min(total, hi + self.halo))

    def push(self, n_frames):
        """n_frames more frames arrived; returns the (rank, Chunk) pairs that became dispatchable."""
        assert not self.closed
        self.frames += n_frames
        out = []
        while (self.next_chunk + 1) * self.chunk_len + self.halo <= self.frames:
            out.append((self.next_chunk % self.world, self._chunk(self.next_chunk, 1 << 62)))
            self.next_chunk += 1
        return out

    def finish(self):
        """End of the stream: the remaining chunks, clipped to the clip length."""
        self.closed = True
        out = []
        while self.next_chunk * self.chunk_len < self.frames:
            out.append((self.next_chunk % self.world, self._chunk(self.next_chunk, self.frames)))
            self.next_chunk += 1
        return out

    def oldest_needed(self):
        """First frame a future chunk still needs: everything before it may be released by the frame store."""
        return max(0, self.next_chunk * self.chunk_len - self.halo)
