"""Multi-GPU plumbing: static block partition of the (HRTF set x orientation) batch over the
ranks of one node and the gather of the finished filter banks onto rank 0.

The path shards with no data-path collective (SURVEY.md 8-e): every filter set is independent.
NCCL (torch.distributed) is used once, after the solve, to gather the banks.
"""
from __future__ import annotations

import os

import torch
import torch.distributed as dist


def env_world():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def init(backend: str | None = None):
    """Initialise torch.distributed from the torchrun environment (no-op for world size 1)."""
    rank, local_rank, world = env_world()
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        backend = backend or ("nccl" if torch.cuda.is_available() else "gloo")
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
        dist.init_process_group(backend=backend, rank=rank, world_size=world)
    return rank, local_rank, world


def shard_range(n: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block [lo, hi) of n units owned by `rank`; sizes differ by at most one."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gather_banks(local: torch.Tensor, n_total: int, dst: int = 0):
    """Gather per-rank banks [n_local, ...] (unit index first) onto rank `dst`.

    Returns the [n_total, ...] tensor on rank dst and None elsewhere.  Shards may be ragged
    (see shard_range); they are padded to the largest shard for the collective.
    """
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return local
    world, rank = dist.get_world_size(), dist.get_rank()
    sizes = [shard_range(n_total, r, world) for r in range(world)]
    nmax = max(hi - lo for lo, hi in sizes)
    buf = local
    if local.shape[0] != nmax:
        buf = torch.zeros((nmax,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        buf[: local.shape[0]] = local
    buf = buf.contiguous()
    if rank == dst:
        parts = [torch.empty_like(buf) for _ in range(world)]
        dist.gather(buf, parts, dst=dst)
        return torch.cat([p[: hi - lo] for p, (lo, hi) in zip(parts, sizes)], 0)
    dist.gather(buf, None, dst=dst)
    return None


def gather_into(local: torch.Tensor, total: torch.Tensor | None, n_total: int, dst: int = 0):
    """Gather per-rank shards (unit index first) straight into the preallocated [n_total, ...] bank `total`
    of rank `dst`: grouped send/recv, no staging copies.  On rank dst, `local` may be the view
    total[lo:hi] of its own shard (then nothing is copied for it).  Returns `total` on dst, None elsewhere."""
    if not dist.is_initialized() or dist.get_world_size() == 1:
        if total is not None and total.data_ptr() != local.data_ptr():
            total[: local.shape[0]].copy_(local)
        return total if total is not None else local
    world, rank = dist.get_world_size(), dist.get_rank()
    if rank == dst:
        ops = []
        for r in range(world):
            lo, hi = shard_range(n_total, r, world)
            if r == dst:
                if total[lo:hi].data_ptr() != local.data_ptr():
                    total[lo:hi].copy_(local)
            elif hi > lo:
                ops.append(dist.P2POp(dist.irecv, total[lo:hi], r))
        for w in (dist.batch_isend_irecv(ops) if ops else []):
            w.wait()
        return total
    if local.shape[0] > 0:
        for w in dist.batch_isend_irecv([dist.P2POp(dist.isend, local.contiguous(), dst)]):
            w.wait()
    return None


class ShardedDesigner:
    """End-to-end eMagLS2 design of one orientation batch sharded over the ranks (SURVEY.md 8-e): host inputs
    in pinned memory -> H2D -> `emagls_design_emagls2_dev` on this rank's contiguous block of orientations ->
    D2H of this rank's shard into pinned host memory and NCCL gather of the banks into rank 0's device bank.
    No data-path collective; the gather is the only exchange.  All buffers are allocated once.

    The banks are double buffered: the transfers of step i (D2H + gather) run on a second stream while step i + 1
    is designed into the other buffer, so in steady state the exchange costs nothing but its bandwidth.  `step()`
    returns once the design has been enqueued; `wait()` returns when every transfer issued so far has finished."""

    def __init__(self, handle, hL, hR, az, ze, mic_radius, maz, mze, order, fs, length, rotations_total, config=None,
                 buffers: int = 2):
        import ctypes as C
        import numpy as np
        self.C, self.np, self.h = C, np, handle
        rank, local_rank, world = env_world()
        self.rank, self.world = rank, world
        self.dev = torch.device("cuda", handle.device if hasattr(handle, "device") else local_rank)
        self.cfg = config if config is not None else handle.default_config()
        self.stream = torch.cuda.ExternalStream(handle.stream, device=self.dev)
        self.xfer = torch.cuda.Stream(device=self.dev)
        R = np.ascontiguousarray(np.asarray(rotations_total, dtype=np.float64).reshape(-1, 9))
        self.n_total = R.shape[0]
        self.lo, self.hi = shard_range(self.n_total, rank, world)
        self.n_local = self.hi - self.lo
        self.T, self.D, self.M = hL.shape[0], hL.shape[1], int(np.asarray(maz).size)
        self.order, self.fs, self.len, self.r = int(order), float(fs), int(length), float(mic_radius)

        def pin(x):
            t = torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float64))).pin_memory()
            return t, torch.empty_like(t, device=self.dev)
        # [T, D] column-major == [D, T] row-major
        self.host_in = [pin(np.asarray(hL).T), pin(np.asarray(hR).T), pin(az), pin(ze), pin(maz), pin(mze),
                        pin(R[self.lo:self.hi])]
        self.h2d_bytes = sum(h.numel() * 8 for h, _ in self.host_in)
        shape = (max(self.n_local, 1), self.M, self.len)       # [len, M, B] column-major
        self.nbuf = max(1, int(buffers))
        self.totals, self.banks, self.host_outs = [], [], []
        for _ in range(self.nbuf):
            # rank 0 designs straight into its slice of the total bank [2 ears][n_total]
            total = (torch.empty((2, self.n_total, self.M, self.len), dtype=torch.float64, device=self.dev)
                     if rank == 0 else None)
            if rank == 0:
                bank = [total[e, self.lo:self.hi] for e in range(2)]
            else:
                bank = [torch.empty(shape, dtype=torch.float64, device=self.dev)[: self.n_local] for _ in range(2)]
            self.totals.append(total)
            self.banks.append(bank)
            self.host_outs.append([torch.empty((self.n_local, self.M, self.len), dtype=torch.float64).pin_memory()
                                   for _ in range(2)])
        self.designed = [torch.cuda.Event() for _ in range(self.nbuf)]
        self.moved = [None] * self.nbuf          # event: the transfers out of buffer b have finished
        self.cur = 0                             # buffer the next step designs into
        self.last = 0                            # buffer of the latest step
        self.d2h_bytes = 2 * self.n_local * self.M * self.len * 8

    # the buffers of the latest step (device bank of this rank, gathered bank on rank 0, pinned host shard)
    @property
    def bank(self):
        return self.banks[self.last]

    @property
    def total(self):
        return self.totals[self.last]

    @property
    def host_out(self):
        return self.host_outs[self.last]

    def step(self, gather: bool = True):
        C, h = self.C, self.h
        b = self.cur
        bank, total = self.banks[b], self.totals[b]
        with torch.cuda.stream(self.stream):
            if self.moved[b] is not None:
                self.stream.wait_event(self.moved[b])       # the previous contents of this buffer have left
            for hbuf, dbuf in self.host_in:
                dbuf.copy_(hbuf, non_blocking=True)
            d = [db for _, db in self.host_in]
            if self.n_local > 0:
                rc = h.lib.emagls_design_emagls2_dev(
                    h.ptr, C.byref(self.cfg), d[0].data_ptr(), d[1].data_ptr(), self.T, self.D, d[2].data_ptr(),
                    d[3].data_ptr(), self.r, d[4].data_ptr(), d[5].data_ptr(), self.M, self.order, self.fs, self.len,
                    1, self.n_local, d[6].data_ptr(), bank[0].data_ptr(), bank[1].data_ptr(), None)
                h.check(rc)
            self.designed[b].record(self.stream)
        with torch.cuda.stream(self.xfer):
            self.xfer.wait_event(self.designed[b])
            for e in range(2):
                self.host_outs[b][e].copy_(bank[e], non_blocking=True)
            if gather and self.world > 1:
                for e in range(2):
                    gather_into(bank[e], total[e] if total is not None else None, self.n_total, 0)
            ev = torch.cuda.Event()
            ev.record(self.xfer)
            self.moved[b] = ev
        self.last = b
        self.cur = (b + 1) % self.nbuf
        return total

    def wait(self):
        self.stream.synchronize()
        self.xfer.synchronize()


def render_shard(n_frames: int, taps: int, rank: int, world: int) -> tuple[int, int, int]:
    """Time-block sharding of the binaural render (SURVEY.md 8-e; dependencies/binauralDecode.m:39-42): rank r renders
    the output frames [lo, hi); an FIR of `taps` taps needs the `taps - 1` input frames before lo as a halo (zeros
    before frame 0).  Returns (lo, hi, halo) with halo = min(taps - 1, lo): the rank convolves in[lo - halo : hi] and
    drops the first `halo` output frames.  No exchange between ranks."""
    lo, hi = shard_range(n_frames, rank, world)
    return lo, hi, min(max(taps - 1, 0), lo)


class ShardedRenderer:
    """binauralDecode of one long multichannel signal sharded over the ranks by time blocks with a (taps - 1)-frame
    input halo: pinned host input block -> H2D -> emagls_binaural_decode_dev -> D2H of the block's two output
    channels.  Every rank keeps its block of the output (gather with torch.distributed if one host needs it all)."""

    def __init__(self, handle, block_host, wL, wR, halo: int, *, track=None, rotations=None, hop=None, fade=None,
                 first_sample=0):
        """block_host: [halo + frames of this rank, channels], the rank's input block with its halo in front.
        Head-tracked render (emagls_binaural_decode_tracked): wL, wR are a bank [taps, channels, pages], `track` the
        0-based page of every frame of `hop` samples of the whole signal, `fade` the crossfade (default hop) and
        `first_sample` the position of block_host[0] in the whole signal (lo - halo).
        Head-tracked render of a real SH signal (emagls_binaural_decode_sh_tracked): `rotations` [frames, 3, 3] is the
        head orientation of every frame of the whole signal, wL, wR one filter pair [taps, (order+1)^2]; `hop`, `fade`
        and `first_sample` as for `track`.  The track is uploaded once, here."""
        import ctypes as C
        import numpy as np
        if track is not None and rotations is not None:
            raise ValueError("track= (a filter bank) and rotations= (a rotated SH signal) exclude each other")
        self.C, self.h = C, handle
        self.dev = torch.device("cuda", handle.device)
        self.stream = torch.cuda.ExternalStream(handle.stream, device=self.dev)
        self.taps, self.ch = int(wL.shape[0]), int(wL.shape[1])
        self.pages = int(wL.shape[2]) if np.ndim(wL) == 3 else 1
        self.halo, self.n = int(halo), int(block_host.shape[0])
        self.track = None
        self.rot_d = None
        if track is not None or rotations is not None:
            self.hop = int(hop)
            self.fade = self.hop if fade is None else int(fade)
            self.first_sample = int(first_sample)
        if track is not None:
            self.track = np.ascontiguousarray(np.asarray(track), dtype=np.int32)
        if rotations is not None:
            self.order = int(round(self.ch ** 0.5)) - 1
            if (self.order + 1) ** 2 != self.ch or np.ndim(wL) != 2:
                raise ValueError("rotations= needs one filter pair [taps, (order+1)^2]")
            R = np.ascontiguousarray(np.asarray(rotations, dtype=np.float64).reshape(-1, 9))
            self.rot_d = torch.from_numpy(R).to(self.dev)
        # [frames, channels] column-major == [channels, frames] row-major
        blk = np.ascontiguousarray(np.asarray(block_host, dtype=np.float64).T)
        self.x_h = torch.from_numpy(blk).pin_memory()
        self.x_d = torch.empty_like(self.x_h, device=self.dev)
        self.w = [torch.from_numpy(np.ascontiguousarray(np.asarray(w, dtype=np.float64).T)).to(self.dev) for w in (wL, wR)]
        self.y_d = torch.empty((2, self.n), dtype=torch.float64, device=self.dev)
        self.y_h = torch.empty((2, self.n - self.halo), dtype=torch.float64).pin_memory()
        self.h2d_bytes = self.x_h.numel() * 8
        self.d2h_bytes = self.y_h.numel() * 8

    @classmethod
    def for_signal(cls, handle, x_host, wL, wR, *, track=None, rotations=None, hop=None, fade=None):
        """Shard the whole signal x_host [frames, channels] over the ranks of the process group (head-tracked with
        `track`, `hop`, `fade` and a bank wL, wR [taps, channels, pages], or with `rotations`, `hop`, `fade` and one
        filter pair for a real SH signal)."""
        rank, _, world = env_world()
        lo, hi, halo = render_shard(int(x_host.shape[0]), int(wL.shape[0]), rank, world)
        r = cls(handle, x_host[lo - halo:hi], wL, wR, halo, track=track, rotations=rotations, hop=hop, fade=fade,
                first_sample=lo - halo)
        r.lo, r.hi = lo, hi
        return r

    def step(self):
        h = self.h
        with torch.cuda.stream(self.stream):
            self.x_d.copy_(self.x_h, non_blocking=True)
            if self.rot_d is not None:
                h.check(h.lib.emagls_binaural_decode_sh_tracked_dev(
                    h.ptr, self.x_d.data_ptr(), self.n, self.order, self.w[0].data_ptr(), self.w[1].data_ptr(),
                    self.taps, self.rot_d.data_ptr(), self.rot_d.shape[0], self.hop, self.fade, self.first_sample, 0,
                    self.y_d.data_ptr()))
            elif self.track is None:
                h.check(h.lib.emagls_binaural_decode_dev(h.ptr, self.x_d.data_ptr(), self.n, self.ch,
                                                         self.w[0].data_ptr(), self.w[1].data_ptr(), self.taps, 0,
                                                         self.y_d.data_ptr()))
            else:
                h.check(h.lib.emagls_binaural_decode_tracked_dev(
                    h.ptr, self.x_d.data_ptr(), self.n, self.ch, self.w[0].data_ptr(), self.w[1].data_ptr(), self.taps,
                    self.pages, self.track.ctypes.data_as(self.C.c_void_p), self.track.size, self.hop, self.fade,
                    self.first_sample, 0, self.y_d.data_ptr()))
            self.y_h.copy_(self.y_d[:, self.halo:], non_blocking=True)

    def wait(self):
        self.stream.synchronize()
        return self.y_h.numpy().T        # [frames of this block, 2]


def max_over_ranks(value: float, device=None) -> float:
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device or ("cuda" if dist.get_backend() == "nccl" else "cpu"))
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier():
    if dist.is_initialized() and dist.get_world_size() > 1:
        dist.barrier()
