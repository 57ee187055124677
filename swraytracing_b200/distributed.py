"""Multi-GPU layer: packets shard, the flow replicates, only histograms / diagnostics reduce.

One process per GPU (torchrun); ``torch.distributed`` is plumbing only.  The step has NO data-path
collective (packets are independent, SURVEY.md 8e); the collectives are an integer SUM all-reduce
of the omega / energy histogram (analysis/load_data.m:39-49) and of a handful of diagnostic
scalars, once per diagnostic interval.  Integer histograms are bit-exact under any sharding.
"""
from __future__ import annotations

import numpy as np


def shard_range(n, rank, world):
    """contiguous packet slice [lo, hi) owned by ``rank`` (SURVEY.md 8e)."""
    return (rank * n) // world, ((rank + 1) * n) // world


class _DeviceI64:
    """__cuda_array_interface__ view of n int64 at a raw device pointer (the engine's histogram counts;
    u64 counts reinterpreted as i64 -- identical bits for counts < 2^63)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": "<i8", "data": (int(ptr), False), "version": 3}


class HistPipeline:
    """Histogram diagnostics pipelined against the packet kernel (the only collective of the path).

    Per diagnostic interval the caller does
        engine.step(...)          # asynchronous launch of the interval's packet kernel
        done = pipe.rotate()      # host work hidden under that kernel (see below)
        pipe.launch(alpha)        # local histogram kernel queued behind the packet kernel, no host wait
    ``rotate`` takes the histogram launched in the PREVIOUS interval (its kernel has long finished), snapshots the
    counts with a device-to-device copy, issues the SUM all-reduce asynchronously, and returns the globally reduced
    counts of the interval before that (or None while the pipeline fills).  No rank ever blocks on another inside an
    interval; ``drain()`` returns the results still in flight.  Without a process group (1 GPU, or the CPU stand-in
    engines of the gloo tests) the same calls degrade to local / synchronous reductions."""

    def __init__(self, ens, edges, kind=0):
        self.ens, self.edges, self.kind = ens, np.ascontiguousarray(edges, dtype=np.float64), kind
        self.nccl = (ens.dist is not None and ens.world > 1 and ens.device is not None
                     and getattr(ens.device, "type", "cpu") == "cuda")
        self.device_side = hasattr(ens.engine, "hist_omega_launch")
        self._launched = None      # (ptr, nbins) of a histogram kernel in flight
        self._reducing = None      # (work, tensor) of an all-reduce in flight
        self._ready = []           # finished results not yet handed out (non-NCCL paths)

    def launch(self, alpha=0.0):
        if self.device_side:
            self._launched = self.ens.engine.hist_omega_launch(self.edges, self.kind, alpha)
        else:
            self._ready.append(self.ens.hist_omega(self.edges, self.kind, alpha))

    def _collect(self):
        if self._reducing is None:
            return None
        work, t = self._reducing
        self._reducing = None
        if work is not None:
            work.wait()
        return t.cpu().numpy().astype(np.uint64)

    def rotate(self):
        out = self._collect()
        if self._launched is not None:
            import torch
            ptr, nb = self._launched
            self._launched = None
            self.ens.engine.hist_omega_wait()                         # that kernel only, not the work queued after it
            dev = self.ens.device if self.ens.device is not None else torch.device("cuda", self.ens.engine.device)
            t = torch.empty(nb, dtype=torch.int64, device=dev)
            t.copy_(torch.as_tensor(_DeviceI64(ptr, nb), device=dev))   # D2D snapshot: the engine reuses its buffer
            torch.cuda.current_stream(dev).synchronize()
            work = self.ens.dist.all_reduce(t, op=self.ens.dist.ReduceOp.SUM, async_op=True) if self.nccl else None
            self._reducing = (work, t)
        if out is None and self._ready:
            out = self._ready.pop(0)
        return out

    def drain(self):
        """results still in flight, oldest first"""
        outs = []
        for _ in range(3):
            r = self.rotate()
            if r is not None:
                outs.append(r)
        return outs


class ShardedEnsemble:
    """A rank-local engine holding this rank's packet shard.

    ``engine`` is any object with the Engine methods used here (set_packets/get_packets/step/
    hist_omega/diag); tests on CPU (gloo) pass an oracle-backed stand-in, production passes
    ``swraytracing_b200.Engine`` bound to the local CUDA device."""

    def __init__(self, engine, n_total, rank=0, world=1, dist=None, device=None):
        self.engine, self.n_total, self.rank, self.world = engine, int(n_total), int(rank), int(world)
        self.lo, self.hi = shard_range(self.n_total, self.rank, self.world)
        self.dist = dist
        self.device = device

    # -- packets --
    def set_packets_global(self, x, y, k, l, a=None):
        s = slice(self.lo, self.hi)
        self.engine.set_packets(x[s], y[s], k[s], l[s], None if a is None else a[s])

    def step(self, scheme, dt, nsteps, alpha0=0.0, dalpha=0.0):
        self.engine.step(scheme, dt, nsteps, alpha0, dalpha)

    def ode23(self, tspan, tmax, rtol=1e-3, atol=1e-6, per_packet=False, events=None, ev_cap=4):
        """the reference's per-flow-step ode23 solve over ALL shards: the error norm is MAX-all-reduced so
        that every rank accepts/rejects the same steps (the reference's norm couples all packets).
        ``per_packet=True``: every packet under its own controller (``Engine.ode23_packets``) on the local shard, with no
        collective; the returned counts are this rank's, and so are the event records with ``events`` (per-packet only).
        A 2-D ``tspan`` (per-packet only) is the global ``(ntspan, n_total)`` matrix: this rank solves its columns [lo, hi)."""
        from .reference_api import ode23
        if events is not None and not per_packet:
            raise ValueError("ode23: events need per_packet=True (the coupled solve has no events)")
        if per_packet and np.ndim(tspan) == 2:
            tspan = np.asarray(tspan, dtype=np.float64)
            if tspan.shape[1] != self.n_total:
                raise ValueError(f"ode23: a per-packet tspan must have n_total = {self.n_total} columns, got {tspan.shape}")
            tspan = tspan[:, self.lo:self.hi]
        if per_packet:
            return ode23(self.engine, tspan, tmax, rtol, atol, per_packet=True, events=events, ev_cap=ev_cap)
        return ode23(self.engine, tspan, tmax, rtol, atol, reduce_max=self._allreduce_max)

    def ode23_packets_tspans_events(self, tspan, tmax, events, rtol=1e-3, atol=1e-6, ev_cap=4):
        """``Engine.ode23_packets_tspans_events`` on the local shard, with no collective: a 2-D ``tspan`` is the global
        ``(ntspan, n_total)`` matrix and this rank solves its columns [lo, hi); a 1-D one is shared by every packet.  The
        returned counts and event records are this rank's."""
        tspan = np.asarray(tspan, dtype=np.float64)
        if tspan.ndim == 2:
            if tspan.shape[1] != self.n_total:
                raise ValueError(f"ode23_packets_tspans_events: tspan must have n_total = {self.n_total} columns, got {tspan.shape}")
            tspan = tspan[:, self.lo:self.hi]
        return self.engine.ode23_packets_tspans_events(tspan, tmax, events, rtol, atol, ev_cap)

    def _allreduce_max(self, v):
        if self.dist is None or self.world == 1:
            return v
        import torch
        t = torch.tensor([v], dtype=torch.float64)
        if self.device is not None:
            t = t.to(self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.cpu()[0])

    # -- reductions --
    def _allreduce_sum(self, arr_i64):
        if self.dist is None or self.world == 1:
            return arr_i64
        import torch
        t = torch.from_numpy(arr_i64.copy())
        if self.device is not None:
            t = t.to(self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t.cpu().numpy()

    def hist_omega(self, edges, kind=0, alpha=0.0):
        """global histcounts over all shards: local u64 counts -> SUM all-reduce (bit-exact).
        With NCCL the counts are reduced in place in the engine's device buffer (no host round trip)."""
        on_gpu = (self.dist is not None and self.world > 1 and self.device is not None
                  and getattr(self.device, "type", "cpu") == "cuda" and hasattr(self.engine, "hist_omega_dev"))
        if on_gpu:
            import torch
            ptr, nb = self.engine.hist_omega_dev(edges, kind, alpha)
            t = torch.as_tensor(_DeviceI64(ptr, nb), device=self.device)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
            return t.cpu().numpy().astype(np.uint64)
        local = self.engine.hist_omega(edges, kind, alpha)
        return self._allreduce_sum(local.astype(np.int64)).astype(np.uint64)

    def hist2(self, qx, xedges, qy, yedges, alpha=0.0):
        """global histcounts2 of two packet quantities (``Engine.hist2``) over all shards: each rank's local u64 counts,
        SUM-all-reduced (bit-exact under any world size)"""
        local = np.asarray(self.engine.hist2(qx, xedges, qy, yedges, alpha))
        return self._allreduce_sum(local.astype(np.int64)).astype(np.uint64)

    def hist2_sums(self, qx, xedges, qy, yedges, weights, alpha=0.0):
        """``Engine.hist2_sums`` over all shards, bit-identical under any world size: every rank's scale exponents
        MAX-all-reduced, each rank's int64 accumulators with those exponents SUM-all-reduced, then rounded once on the host
        (``fixed_sums_to_double``).  Returns ``(sums, counts)``."""
        from .engine import fixed_sums_to_double
        e = np.asarray(self.engine.weight_scale(weights, alpha), dtype=np.int32)
        if self.dist is not None and self.world > 1:
            import torch
            t = torch.from_numpy(e.copy())
            if self.device is not None:
                t = t.to(self.device)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            e = t.cpu().numpy()
        _, counts, acc = self.engine.hist2_sums(qx, xedges, qy, yedges, weights, alpha, scale_exp=e, return_acc=True)
        acc = self._allreduce_sum(np.ascontiguousarray(acc))
        counts = self._allreduce_sum(np.asarray(counts).astype(np.int64)).astype(np.uint64)
        return fixed_sums_to_double(acc, e), counts

    def hist_pipeline(self, edges, kind=0):
        return HistPipeline(self, edges, kind)

    def ideal_omega_hist(self, x, y, kvx, kvy, omega0, edges, alpha=0.0):
        """theoretical omega pdf (ideal_omega_distribution.m:3-11) over ALL grid points, sharded: each rank bins
        omega0 + U(x_i).k_j for its contiguous slice of the points, then the same integer SUM all-reduce as the packet
        histogram (SURVEY.md 8f-4).  Every rank passes the full point list; counts are bit-exact under any sharding."""
        x = np.asarray(x, dtype=np.float64).ravel(); y = np.asarray(y, dtype=np.float64).ravel()
        lo, hi = shard_range(x.size, self.rank, self.world)
        local = self.engine.ideal_omega_hist(x[lo:hi], y[lo:hi], kvx, kvy, omega0, edges, alpha)
        return self._allreduce_sum(np.asarray(local).astype(np.int64)).astype(np.uint64)

    def energy_vs_omega(self, edges, kind=0, alpha=0.0):
        """energy = centre .* counts (analysis/load_data.m:40,49)"""
        counts = self.hist_omega(edges, kind, alpha)
        edges = np.asarray(edges, dtype=np.float64)
        centre = (edges[1:] + edges[:-1]) / 2
        return centre, centre * counts.astype(np.float64), counts

    def diag(self, alpha=0.0):
        """sum/max/min diagnostics all-reduced: sums add, extrema reduce with max/min."""
        d = np.asarray(self.engine.diag(alpha), dtype=np.float64)
        if self.dist is None or self.world == 1:
            return d
        import torch
        sums = torch.tensor([d[0], d[1], d[4], d[5], d[6], d[7]], dtype=torch.float64)
        mx = torch.tensor([d[2]], dtype=torch.float64)
        mn = torch.tensor([d[3]], dtype=torch.float64)
        if self.device is not None:
            sums, mx, mn = sums.to(self.device), mx.to(self.device), mn.to(self.device)
        self.dist.all_reduce(sums, op=self.dist.ReduceOp.SUM)
        self.dist.all_reduce(mx, op=self.dist.ReduceOp.MAX)
        self.dist.all_reduce(mn, op=self.dist.ReduceOp.MIN)
        s = sums.cpu().numpy()
        return np.array([s[0], s[1], float(mx.cpu()[0]), float(mn.cpu()[0]), s[2], s[3], s[4], s[5]])

    def gather_packets(self):
        """all shards' packets on every rank (for tests / small runs)."""
        loc = self.engine.get_packets()
        if self.dist is None or self.world == 1:
            return loc
        import torch
        out = []
        for arr in loc:
            pieces = [None] * self.world
            self.dist.all_gather_object(pieces, arr)
            out.append(np.concatenate(pieces))
        return tuple(out)
