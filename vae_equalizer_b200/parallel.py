"""Multi-GPU plumbing (one process per GPU, torch.distributed): SURVEY.md §8e.

* Sweep sharding: the cells of the reference's parameter sweep (Eval_run_DP.py:68-95: nu x batch_len x lr x M x
  theta_diff x symb_rate x flex_step x theta x SNR x iter) are independent `processing()` calls.  `shard_cells`
  deals them round-robin to the ranks, `gather_cell_results` reassembles the per-cell result tensors on rank 0, NaN entries
  included.  No data-path collective.
* Batch-split of ONE long minibatch (VAE-flex with large batch_len): `BatchSplitDP` gives every rank a contiguous
  symbol range of the window and all-reduces (a) the ELBO partial sums (8 + 2(M-1) doubles) before the backward scale
  kappa = (L-Mh)/C is known and (b) the 16*M tap-gradient floats before the replicated Adam step.  Both messages are
  latency-bound (< 1 KB); NCCL over NVLink carries them on the step's stream.
CMA does not shard (per-symbol tap recurrence): replicas only.
"""
from __future__ import annotations

import itertools

import torch
import torch.distributed as dist

TILE = 496                      # owned symbols per tile of the fast kernels (csrc/dp_fast.cu FT_T = 4 * 128 - 16)


KEEP_COST = 0.04                # extra cost of a tile whose q / out columns are WRITTEN, relative to the whole step of a tile that writes none
                                # (forward 279 vs 259 us of a ~500 us step at N = 8, profiles/r02_batch_split.txt)


def split_ranges(B: int, world: int, align: int = TILE, keep=None, keep_cost: float = KEEP_COST):
    """Contiguous symbol ranges [lo, hi) covering [0, B), multiples of 4, sized in whole tiles where possible.

    keep = (keep_lo, keep_n): the window is stepped by a frame loop that writes q / out for the kept section only (VAEflex_DP:64-65), so a
    tile inside it costs 1 + keep_cost and one outside 1; the ranges then carry equal COST instead of equal length (the ranks inside
    the kept section get ~keep_cost/2 fewer symbols), which removes the wait of the other ranks at the first exchange of every step."""
    if B % 4:
        raise ValueError("batch-split needs batch_len % 4 == 0")
    units = (B + align - 1) // align
    if units < world:
        raise ValueError(f"batch_len={B} is too short to split {world} ways in tiles of {align} symbols")
    if keep is None or keep_cost <= 0.0 or world == 1:
        counts = [units // world + (1 if r < units % world else 0) for r in range(world)]
    else:
        klo, khi = int(keep[0]), int(keep[0]) + int(keep[1])

        def cost_upto(u):                                   # cost of tiles [0, u): u + keep_cost * (kept symbols below u * align) / align
            kept = max(0, min(u * align, khi, B) - klo)
            return u + keep_cost * kept / align

        total, bounds = cost_upto(units), [0]
        for r in range(1, world):
            target, lo_u, hi_u = total * r / world, bounds[-1] + 1, units - (world - r)
            a, b = lo_u, hi_u                                # smallest u in [lo_u, hi_u] with cost_upto(u) >= target (cost_upto is monotone)
            while a < b:
                mid = (a + b) // 2
                if cost_upto(mid) >= target:
                    b = mid
                else:
                    a = mid + 1
            if a > lo_u and target - cost_upto(a - 1) < cost_upto(a) - target:
                a -= 1
            bounds.append(a)
        bounds.append(units)
        counts = [bounds[r + 1] - bounds[r] for r in range(world)]
        equal, eb = [units // world + (1 if r < units % world else 0) for r in range(world)], [0]
        for n in equal:
            eb.append(eb[-1] + n)
        if max(cost_upto(eb[r + 1]) - cost_upto(eb[r]) for r in range(world)) <= max(cost_upto(bounds[r + 1]) - cost_upto(bounds[r]) for r in range(world)):
            counts = equal                                   # tile granularity: the equal split is at least as good (short windows)
    out, lo = [], 0
    for r in range(world):
        hi = min(B, lo + counts[r] * align)
        if r == world - 1:
            hi = B
        out.append((lo, hi))
        lo = hi
    if any(hi <= lo for lo, hi in out):
        raise ValueError(f"batch_len={B} is too short to split {world} ways in tiles of {align} symbols")
    return out


def shard_cells(cells, rank: int, world: int):
    """Round-robin assignment of sweep cells (any sequence) to `rank`; returns [(global_index, cell), ...]."""
    return [(i, c) for i, c in enumerate(cells) if i % world == rank]


def sweep_cells(**axes):
    """Cartesian product of named parameter lists in the reference's loop order -> list of dicts."""
    names = list(axes)
    return [dict(zip(names, vals)) for vals in itertools.product(*(axes[n] for n in names))]


def gather_cell_results(local, n_cells: int, shape, rank: int, world: int, group=None, device="cpu"):
    """`local` = {global_index: tensor(shape)} computed by this rank.  Returns the (n_cells, *shape) tensor on rank 0
    (None elsewhere).  One all_reduce of a dense, zero-padded block per rank; cells are disjoint so a sum suffices.  NaN entries
    (unscored frames) survive it: the block carries the values with NaN as 0 next to a NaN mask, so values of either sign are kept."""
    block = torch.zeros((n_cells,) + tuple(shape), dtype=torch.float32, device=device)
    for i, t in local.items():
        block[i] = t.to(device=device, dtype=torch.float32)
    nan = torch.isnan(block)
    block = torch.stack((block.masked_fill(nan, 0.0), nan.to(torch.float32)))
    if world > 1:
        dist.all_reduce(block, op=dist.ReduceOp.SUM, group=group)
    return block[0].masked_fill(block[1] > 0, float("nan")) if rank == 0 else None


def allreduce_sum_(t: torch.Tensor, group=None):
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def kept_owner_ranges(B: int, world: int, keep_lo: int, keep_n: int, weighted: bool = False):
    """Per rank: the part [a, b) of the kept section [keep_lo, keep_lo + keep_n) of a window that this rank's symbol range covers, as
    offsets INSIDE the kept section (empty ranges have a == b).  The ranges of all ranks tile [0, keep_n).  weighted: the cost-balanced
    ranges of a frame loop that writes the kept section only (split_ranges(keep=...))."""
    out = []
    for lo, hi in split_ranges(B, world, keep=(keep_lo, keep_n) if weighted else None):
        a, b = max(lo, keep_lo), min(hi, keep_lo + keep_n)
        out.append((a - keep_lo, b - keep_lo) if b > a else (0, 0))
    return out


class BatchSplitDP:
    """One DP VAE-LE/VAE-flex run whose minibatch is split over the ranks of `group` (all ranks call in lockstep).

    Every rank keeps the full rx window (an input, replicated once per frame outside the step) and an identical
    copy of W / h / Adam state; the update is replicated and bit-identical because both reductions return the same
    bits on every rank.  Summation order differs from the single-GPU run, so parity with it is ~1e-6, not bitwise.

    transport: "peer" = both reductions inside the library over NVLink peer memory (vaeq_dp_split_step_peer: slots in
    torch symmetric memory, epoch flags, partials added in rank order; no host-issued collective in the step), "nccl" = two
    NCCL all-reduces between the three phase calls, "auto" = peer when symmetric memory can be set up for the group."""

    def __init__(self, eq, group=None, transport="auto", balance_keep=True):
        self.eq, self.group = eq, group
        self.balance_keep = bool(balance_keep)   # steps that write the kept section only split the window by cost, not by length
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.transport, self.comm, self._graphs, self._local, self._warm = "nccl", None, {}, {}, set()
        if transport not in ("auto", "peer", "nccl"):
            raise ValueError(f"unknown transport {transport!r}")
        if transport != "nccl" and self.world > 1:
            try:
                self._setup_peer()
                self.transport = "peer"
            except Exception as e:              # no symmetric memory on this box / build: NCCL carries the two messages
                if transport == "peer":
                    raise
                self.peer_error = repr(e)
            if transport == "auto":             # every rank must take the same path
                ok = torch.tensor([1 if self.transport == "peer" else 0], device=eq.device)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
                if int(ok.item()) == 0:
                    self.transport = "nccl"

    def _setup_peer(self):
        import torch.distributed._symmetric_memory as symm
        from . import _lib
        if self.world > 8:
            raise _lib.VaeqError("peer transport: at most 8 ranks (one NVSwitch domain)")
        nbytes = int(self.eq.lib.vaeq_peer_slot_bytes(self.eq.M))
        self._slot = symm.empty(nbytes, dtype=torch.uint8, device=self.eq.device)
        self._slot.zero_()
        hdl = symm.rendezvous(self._slot, self.group if self.group is not None else dist.group.WORLD)
        ptrs = [int(x) for x in hdl.buffer_ptrs]
        if len(ptrs) != self.world or int(hdl.rank) != self.rank:
            raise _lib.VaeqError("symmetric-memory rendezvous does not match the process group")
        self._epoch = torch.zeros(2, dtype=torch.int32, device=self.eq.device)
        comm = _lib.PeerComm()
        comm.rank, comm.world, comm.epoch = self.rank, self.world, self._epoch.data_ptr()
        for r, ptr in enumerate(ptrs):
            comm.slot[r] = ptr
        torch.cuda.synchronize(self.eq.device)
        dist.barrier(group=self.group)          # every slot is zeroed before anyone publishes into it
        self.comm, self._symm_handle = comm, hdl

    # -- per-rank buffers ------------------------------------------------------------------------------------------------------
    def local_columns(self, B: int):
        """(lo, hi, col0, n_cols): this rank's symbol range of a batch_len-B window and the q / out columns it writes."""
        lo, hi = split_ranges(B, self.world)[self.rank]
        col0, col1 = max(0, lo - 16), min(B, hi + 16)
        return lo, hi, col0, col1 - col0

    def alloc_local(self, B: int):
        """q / out buffers holding only this rank's columns of a window (pass them with col0 = local_columns(B)[2])."""
        if B not in self._local:
            lo, hi, col0, n = self.local_columns(B)
            dev = self.eq.device
            self._local[B] = (torch.empty(2, 2 * self.eq.n_lev, n, dtype=torch.float32, device=dev),
                              torch.empty(2, 2, n, dtype=torch.float32, device=dev), col0)
        return self._local[B]

    # -- one step ----------------------------------------------------------------------------------------------------------------
    def train_step(self, rx, lr_w, lr_h, q=None, out=None, col0=0, q_keep=None, out_keep=None, keep_lo=0, keep_n=0):
        """One optimizer step on the window rx (2,2,sps*B).  q / out: full-width (col0 = 0) or this rank's columns only
        (alloc_local); q_keep / out_keep receive the kept columns this rank counts."""
        B = rx.shape[-1] // self.eq.sps
        if q is None and q_keep is None:
            q, out, col0 = self.alloc_local(B)
        keep_only = self.balance_keep and q is None and q_keep is not None and keep_n > 0
        lo, hi = split_ranges(B, self.world, keep=(keep_lo, keep_n) if keep_only else None)[self.rank]
        if self.transport == "peer":
            self.eq.split_step_peer(rx, lo, hi, q, out, self.comm, lr_w, lr_h, col0, q_keep, out_keep, keep_lo, keep_n)
        else:
            stats = self.eq.split_forward(rx, lo, hi, q, out, col0, q_keep, out_keep, keep_lo, keep_n)
            allreduce_sum_(stats, self.group)
            grads = self.eq.split_backward(rx, lo, hi, q, out, col0)
            allreduce_sum_(grads, self.group)
            self.eq.split_update(rx, q, out, lr_w, lr_h, col0)
        return self.eq.loss, self.eq.var_est, (lo, hi)

    # -- one frame of sliding windows (func_VAEflex_DP_MQAM_shaping.py:59-70) -------------------------------------------------------
    def train_frame(self, rx_frame, batch_len, stride_sym, n_steps, lr_w, lr_h, out_train, out_const, keep_lo, keep_n, graph=True):
        """Step m trains on symbols [m*stride_sym, m*stride_sym + batch_len) of the frame, every window split over the ranks; the kept
        columns of step m that THIS rank counts land at column m*stride_sym + (u - keep_lo) of out_train / out_const (call
        gather_kept to assemble them on one rank).  graph=True replays the whole frame loop from a CUDA graph (one capture per
        (buffers, shapes, learning rates)); the rx / out tensors must then be the same objects frame after frame.
        Returns (loss_steps (n_steps,), var_est_steps (2, n_steps))."""
        eq, sps, B = self.eq, self.eq.sps, int(batch_len)
        dev = eq.device
        q = out = None                           # the frame loop wants the kept section of every window only: no per-window q / out is written
        col0 = 0
        key = (rx_frame.data_ptr(), out_train.data_ptr(), out_const.data_ptr(), B, int(stride_sym), int(n_steps), float(lr_w), float(lr_h),
               int(keep_lo), int(keep_n))

        def run(loss_steps, var_steps):
            for m in range(n_steps):
                s0 = m * stride_sym
                win = rx_frame[:, :, s0 * sps:(s0 + B) * sps]
                self.train_step(win, lr_w, lr_h, q, out, col0, out_train[:, :, s0:], out_const[:, :, s0:], keep_lo, keep_n)
                loss_steps[m:m + 1].copy_(eq.loss)
                var_steps[:, m].copy_(eq.var_est)

        if not graph:
            loss_steps = torch.empty(n_steps, dtype=torch.float32, device=dev)
            var_steps = torch.empty(2, n_steps, dtype=torch.float32, device=dev)
            run(loss_steps, var_steps)
            return loss_steps, var_steps
        if key not in self._graphs:
            loss_steps = torch.empty(n_steps, dtype=torch.float32, device=dev)
            var_steps = torch.empty(2, n_steps, dtype=torch.float32, device=dev)
            if B not in self._warm:              # first frame of this batch_len: a plain step allocates the workspaces and sets the kernel
                saved = (eq.W.clone(), eq.h.clone(), eq.adam.clone())              # attributes; it must not count as training: state restored
                self.train_step(rx_frame[:, :, :B * sps], lr_w, lr_h, None, None, 0, out_train, out_const, keep_lo, keep_n)
                eq.W.copy_(saved[0]); eq.h.copy_(saved[1]); eq.adam.copy_(saved[2])
                self._warm.add(B)                # (the peer epoch counters stay advanced: every rank made the same extra call)
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize(dev)
            with torch.cuda.graph(g):
                run(loss_steps, var_steps)
            self._graphs[key] = (g, loss_steps, var_steps, (rx_frame, out_train, out_const))
        g, loss_steps, var_steps, _ = self._graphs[key]
        g.replay()
        return loss_steps, var_steps

    def gather_kept(self, B, stride_sym, n_steps, out_train, out_const, keep_lo, keep_n, dst=0):
        """Assemble the kept columns of a frame on rank `dst`: every rank sends the columns it counted (its part of the kept section
        of every step, packed) point to point; nothing is sent for empty parts.  keep_n must equal stride_sym (VAE-flex keeps
        the middle flex_step symbols of every window, VAEflex_DP:64-65)."""
        if self.world == 1:
            return
        if keep_n != stride_sym:
            raise ValueError("gather_kept needs keep_n == stride_sym")
        parts = kept_owner_ranges(B, self.world, keep_lo, keep_n, weighted=self.balance_keep)
        views = [t[:, :, :n_steps * stride_sym].unflatten(2, (n_steps, stride_sym)) for t in (out_train, out_const)]
        ops, bufs = [], []
        if self.rank == dst:
            for r, (a, b) in enumerate(parts):
                if r == dst or b <= a:
                    continue
                for v in views:
                    buf = torch.empty(v.shape[:3] + (b - a,), dtype=v.dtype, device=v.device)
                    ops.append(dist.P2POp(dist.irecv, buf, dist.get_global_rank(self.group, r) if self.group is not None else r, self.group))
                    bufs.append((v, a, b, buf))
        else:
            a, b = parts[self.rank]
            if b > a:
                for v in views:
                    buf = v[:, :, :, a:b].contiguous()
                    ops.append(dist.P2POp(dist.isend, buf, dist.get_global_rank(self.group, dst) if self.group is not None else dst, self.group))
                    bufs.append(buf)
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
        if self.rank == dst:
            for v, a, b, buf in bufs:
                v[:, :, :, a:b].copy_(buf)
