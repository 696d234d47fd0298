"""Multi-GPU reconstruct: one process per GPU, `torch.distributed` (NCCL over NVLink on GPUs, gloo in the CPU tests)
for the plumbing, the C ABI for every kernel.

The reference parallelises over subdomains (dense_subdomains.rs:521-526, :1581-1598); subdomains are independent once
each one has its ghost particles.  Across ranks the subdomain grid is cut into slabs along its longest axis, balanced
by particle count.  One exchange step (variable all-to-all) gives every rank the particles that are members of its
slab's subdomains plus one halo layer of subdomains that is processed for particle densities only -- so ghost
particles get bit-identical densities without a second exchange.  Global particle order (rank r holds the global
indices [offset_r, offset_{r+1})) is preserved by the exchange, because the reference's per-grid-point summation
order is ascending particle index.  There is no data-path collective besides that halo exchange, two tiny
reductions (bounding box, slab histogram + max subdomain population) and the optional mesh gather to rank 0.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional

import numpy as np
import torch
import torch.distributed as dist


# fixed cost of one occupied subdomain tile in the slab balance, in "particle equivalents" (measured: a 64^3-cell tile of
# bulk fluid holds 4096 particles; a nearly empty tile still costs about as much level-set + marching-cubes time)
TILE_COST_PARTICLES = 4096.0

# ---------------------------------------------------------------------------- partition plan (pure host logic) ----
@dataclass
class SlabPlan:
    axis: int                  # partition axis of the subdomain grid
    nsub_axis: int             # subdomains along that axis
    cuts: List[int]            # world+1 cut positions: rank r owns subdomain indices [cuts[r], cuts[r+1])
    srad: int                  # ghost reach in subdomains (ceil(margin / subdomain size))
    halo: int                  # density-only subdomain layers kept around a slab (= srad)
    margin: float = 0.0        # ghost particle margin (dense_subdomains.rs:120-121)
    sub_size: float = 0.0      # edge length of a subdomain
    gmin_axis: Optional[float] = None   # subdomain grid aabb.min along `axis` (set by plan_partition)

    def own(self, r: int):
        return self.cuts[r], self.cuts[r + 1]

    def recv_range(self, r: int):
        """Owner-subdomain index range (along the axis) of the particles rank r needs: members of the subdomains in
        [own_lo - halo, own_hi + halo) are owned by subdomains at most srad further out (+1 for rounding slack)."""
        lo, hi = self.own(r)
        if hi <= lo:
            return 0, 0
        reach = self.halo + self.srad + 1
        return lo - reach, hi + reach

    def recv_interval(self, r: int):
        """Coordinate interval (along the axis) of the particles rank r needs: the members -- owned or ghost -- of the
        subdomain layers [own_lo - halo, own_hi + halo) lie within the ghost margin of that range of layers.  A little slack
        (0.2 % of the margin plus a few float32 ulps of the coordinate) makes it a superset of what the library's f32
        classifier keeps; the library filters exactly.  Far tighter than `recv_range`'s whole layers."""
        lo, hi = self.own(r)
        if hi <= lo or self.gmin_axis is None:
            return 0.0, 0.0
        a = self.gmin_axis + (lo - self.halo) * self.sub_size
        b = self.gmin_axis + (hi + self.halo) * self.sub_size
        slack = self.margin * 1.002 + 1e-5 * (abs(a) + abs(b) + self.sub_size)
        return a - slack, b + slack


def balanced_cuts(hist: np.ndarray, world: int) -> List[int]:
    """Cut positions so that every rank owns a contiguous run of subdomain layers: the partition that MINIMISES THE MAXIMUM load of
    a rank (the step time is the slowest rank's), ties broken towards equal loads.  Layers are coarse -- the 50 M dam break has 21
    dense layers for 8 ranks -- so cutting at the cumulative targets r / world can miss the optimum by a whole layer; this is the
    exact optimum by dynamic programming over (ranks, layers), O(world * n^2) on a few hundred layers."""
    w = np.asarray(hist, dtype=np.float64)
    n = len(w)
    if n == 0 or world <= 1:
        return [0] + [n] * max(world, 1)
    csum = np.concatenate([[0.0], np.cumsum(w)])
    seg = csum[None, :] - csum[:, None]                       # seg[j, i] = load of layers [j, i)
    INF = float("inf")
    seg = np.where(np.arange(n + 1)[:, None] <= np.arange(n + 1)[None, :], seg, INF)
    best_max = seg[0].copy()                                  # one rank owns [0, i)
    best_sq = seg[0] ** 2
    choice = np.zeros((world, n + 1), dtype=np.int64)
    for r in range(1, world):
        cand_max = np.maximum(best_max[:, None], seg)         # [j, i]: ranks < r own [0, j), rank r owns [j, i)
        cand_sq = best_sq[:, None] + np.where(np.isfinite(seg), seg, 0.0) ** 2
        cand_sq = np.where(np.isfinite(cand_max), cand_sq, INF)
        m = cand_max.min(axis=0)
        # among the j that reach the minimum (up to rounding), the most even split
        tie = cand_max <= m[None, :] * (1.0 + 1e-12) + 1e-300
        sq = np.where(tie, cand_sq, INF)
        j = sq.argmin(axis=0)
        choice[r] = j
        best_max, best_sq = m, sq[j, np.arange(n + 1)]
    cuts = [n]
    i = n
    for r in range(world - 1, 0, -1):
        i = int(choice[r][i])
        cuts.append(i)
    cuts.append(0)
    return cuts[::-1]


def make_plan(grid_ncells, subdomain_cubes: int, cube_size: float, compact_support: float, hist_axis=None, world: int = 1,
              axis: Optional[int] = None) -> SlabPlan:
    S = int(subdomain_cubes)
    nsd = [(int(n) + S - 1) // S for n in grid_ncells]
    ax = int(np.argmax(nsd)) if axis is None else int(axis)
    # ghost margin = ceil(h / c) * c * 1.01 (dense_subdomains.rs:120-121); reach in subdomains (:1827)
    c32, h32 = np.float32(cube_size), np.float32(compact_support)
    margin = np.float32(np.float32(np.ceil(h32 / c32) * c32) * np.float32(1.01))
    srad = int(np.ceil(margin / np.float32(c32 * np.float32(S))))
    hist = np.zeros(nsd[ax]) if hist_axis is None else np.asarray(hist_axis)
    return SlabPlan(ax, nsd[ax], balanced_cuts(hist, world), srad, srad, float(margin), float(np.float32(c32 * np.float32(S))))


def plan_partition(x: torch.Tensor, grid_min, grid_ncells, S: int, cube_size: float, compact_support: float, world: int, group=None):
    """Collective: every rank passes its local particles (any device) and gets the same SlabPlan plus its particles' owner
    layers.  Work model per layer of subdomains: particles + a fixed cost per occupied subdomain tile (every tile pays for
    its bricks and 65^3 grid points even when it only holds a thin sheet of fluid)."""
    plan0 = make_plan(grid_ncells, S, cube_size, compact_support, None, world)
    ax = plan0.axis
    sub_size = float(np.float32(np.float32(cube_size) * np.float32(S)))
    nsd = [(int(nc) + S - 1) // S for nc in grid_ncells]
    o = [owner_layer(x[:, d], float(grid_min[d]), sub_size).clamp(0, nsd[d] - 1) for d in range(3)]
    layer = owner_layer(x[:, ax], float(grid_min[ax]), sub_size)
    hist = torch.bincount(o[ax], minlength=nsd[ax]).to(torch.float64)
    dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=group)
    occ = torch.zeros(nsd[0] * nsd[1] * nsd[2], dtype=torch.int32, device=x.device)
    occ[(o[0] * nsd[1] + o[1]) * nsd[2] + o[2]] = 1
    dist.all_reduce(occ, op=dist.ReduceOp.MAX, group=group)
    other = tuple(d for d in range(3) if d != ax)
    tiles = occ.view(nsd[0], nsd[1], nsd[2]).sum(dim=other).to(torch.float64)
    work = hist + TILE_COST_PARTICLES * tiles
    plan = make_plan(grid_ncells, S, cube_size, compact_support, work.cpu().numpy(), world, axis=ax)
    plan.gmin_axis = float(grid_min[ax])
    return plan, layer


def owner_layer(x_axis: torch.Tensor, gmin: float, sub_size: float) -> torch.Tensor:
    """Subdomain layer index of each particle along the partition axis (float64 on purpose: only used to route
    particles conservatively, +-1 slack is added by SlabPlan.recv_range)."""
    return torch.floor((x_axis.to(torch.float64) - float(gmin)) / float(sub_size)).to(torch.int64)


def exchange_particles(x_local: torch.Tensor, layer: torch.Tensor, plan: SlabPlan, world: int, group=None, payload: Optional[torch.Tensor] = None):
    """Variable all-to-all: returns (particles for this rank in ascending global order, counts received per source).
    A particle goes to every rank whose kept layers it can be a member of: by coordinate interval (`recv_interval`) when the
    plan knows the grid origin, else by whole owner layers (`recv_range`).  `payload` ((n, 3) rows, default: the particles
    themselves) is what travels; the routing always comes from `x_local`."""
    if plan.gmin_axis is not None and x_local.shape[1] >= 3:
        coord = x_local[:, plan.axis].to(torch.float64)
        los = torch.tensor([plan.recv_interval(r)[0] for r in range(world)], dtype=torch.float64, device=x_local.device)
        his = torch.tensor([plan.recv_interval(r)[1] for r in range(world)], dtype=torch.float64, device=x_local.device)
        masks = (coord[None, :] >= los[:, None]) & (coord[None, :] < his[:, None])      # (world, n)
    else:
        los = torch.tensor([plan.recv_range(r)[0] for r in range(world)], dtype=torch.int64, device=x_local.device)
        his = torch.tensor([plan.recv_range(r)[1] for r in range(world)], dtype=torch.int64, device=x_local.device)
        masks = (layer[None, :] >= los[:, None]) & (layer[None, :] < his[:, None])      # (world, n)
    idx = torch.nonzero(masks)                                                           # row-major: by rank, then ascending index
    data = x_local if payload is None else payload
    send = data[idx[:, 1]].contiguous()
    counts = [int(v) for v in masks.sum(dim=1).tolist()]
    cnt_in = torch.tensor(counts, dtype=torch.int64, device=x_local.device)
    cnt_out = torch.empty(world, dtype=torch.int64, device=x_local.device)
    dist.all_to_all_single(cnt_out, cnt_in, group=group)
    out_counts = [int(v) for v in cnt_out.tolist()]
    recv = torch.empty((sum(out_counts), 3), dtype=data.dtype, device=x_local.device)
    dist.all_to_all_single(recv.view(-1), send.view(-1), output_split_sizes=[3 * v for v in out_counts],
                           input_split_sizes=[3 * v for v in counts], group=group)
    return recv, out_counts


# ---------------------------------------------------------------------------- device helpers ----
class _CudaView:
    """Zero-copy torch view of device memory owned by the C library (via __cuda_array_interface__)."""

    def __init__(self, ptr: int, shape, typestr: str):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def _view(ptr, shape, typestr, device):
    if not ptr or int(np.prod(shape)) == 0:
        dt = {"<f4": torch.float32, "<u4": torch.int32, "<i4": torch.int32, "<i8": torch.int64, "<u8": torch.int64}[typestr]
        return torch.empty(tuple(shape), dtype=dt, device=device)
    typestr = typestr.replace("<u4", "<i4").replace("<u8", "<i8")
    if device.type != "cuda":        # host memory: only when the runner is driven by the tests' CPU executor of the CUDA sources
        dt = np.dtype(typestr)
        buf = (C.c_char * (int(np.prod(shape)) * dt.itemsize)).from_address(int(ptr))
        return torch.from_numpy(np.frombuffer(buf, dtype=dt).reshape(tuple(shape)))
    return torch.as_tensor(_CudaView(ptr, shape, typestr), device=device)


class _HostEvent:
    """Stands in for torch.cuda.Event when the runner works on host memory (tests only)."""

    def record(self):
        import time
        self.t = time.perf_counter()

    def elapsed_time(self, other) -> float:
        return (other.t - self.t) * 1e3


def _event(device):
    return torch.cuda.Event(enable_timing=True) if device.type == "cuda" else _HostEvent()


def _sync(device):
    if device.type == "cuda":
        torch.cuda.synchronize()


def _pinned(t: torch.Tensor, device) -> torch.Tensor:
    return t.pin_memory() if device.type == "cuda" else t


class Runner:
    """Drives one reconstruct step on this rank's GPU (world == 1: plain C-ABI call)."""

    def __init__(self, ctx, params, world: int, rank: int, local_rank: int, group=None, device=None, protocol: str = "stats"):
        self.ctx, self.params, self.world, self.rank, self.local_rank, self.group = ctx, params, world, rank, local_rank, group
        # how the global maximum subdomain population (sparse rule) reaches the library: "stats" (default) = the plan statistics
        # count the members of every subdomain with the exact classifier (ss_partition_members_f32), their all-reduced maximum
        # is passed to ONE library call; "two_call" = decomposition pre-pass, all-reduce, full call (3.9 of 66 ms per step at 2 GPUs);
        # "callback" = one call, the library calls back for the all-reduce after its decomposition
        if protocol not in ("stats", "two_call", "callback"):
            raise ValueError("protocol must be 'stats', 'two_call' or 'callback'")
        self.protocol = protocol
        self._out_v = self._out_t = self._out_n = None
        self._seg = None; self._seg_path = None; self._seg_gen = 0; self._seg_registered = False; self._layout = None
        self.want_keys = False           # also publish the MC edge keys of the assembled vertices (parity tools)
        self.ctx_normals = False         # set by the caller when ss_context_set_compute_sph_normals is on: normals join the assembled mesh
        # parameters that carry a particle AABB: the GRID comes from that box (lib.rs:476-516) while `params` (no box) drive the
        # partitioned calls on particles the caller has already filtered
        self.grid_params = None
        self.balance_feedback = True     # slab cuts learn from the measured per-rank time of earlier frames
        self._layer_scale = None; self._layer_key = None
        # ... for a few frames; then the best cuts seen are kept (a plan that keeps moving keeps re-allocating: one 150 ms step in
        # twenty was measured at 8 GPUs) until the slowest rank drifts 15 % above the time they were chosen for
        self.explore_frames = 4
        self._explore_left = self.explore_frames; self._best_t = float("inf"); self._best_cuts = None; self._frozen_cuts = None; self._drift = 0
        # `device` is only overridden by the tests that drive the runner over gloo with the CPU executor of the CUDA sources
        self.device = torch.device("cuda", local_rank) if device is None else torch.device(device)
        self.last_plan: Optional[SlabPlan] = None

    def gathered_normals(self):
        """Host copy of the SPH normals of the last assembled mesh (None when they were not computed / not gathered)."""
        lay = getattr(self, "_layout", None)
        if lay is None:                                      # single-GPU / small-domain path
            return getattr(self, "_out_n", None)
        if not lay[3] or self.device.type != "cuda":
            return None
        nvg, ntg, want_keys, _ = lay
        nbase = ((nvg * 12 + ntg * 12 + 7) // 8 * 8) + (nvg * 8 if want_keys else 0)
        return self._seg[nbase:nbase + nvg * 12].view(torch.float32).view(-1, 3).numpy().copy()

    @property
    def plan_settled(self) -> bool:
        """True once the slab cuts no longer move from frame to frame (single rank, feedback off, or the exploration frames are over).
        The same on every rank: the decision is taken from all-reduced step times."""
        return self.world == 1 or not self.balance_feedback or self._frozen_cuts is not None

    # -- input sharding used by the bench: rank r holds a contiguous range of global particle indices
    def take_local(self, particles: np.ndarray) -> np.ndarray:
        if self.world == 1:
            return particles
        n = len(particles)
        lo, hi = (n * self.rank) // self.world, (n * (self.rank + 1)) // self.world
        return np.ascontiguousarray(particles[lo:hi])

    # -- single GPU
    def _step_single(self, xyz_ptr: int, n: int, copy_out: bool, params=None, force_copy: bool = False) -> dict:
        L = self.ctx._L
        s = self.ctx.reconstruct_raw(xyz_ptr, n, self.params if params is None else params)
        try:
            return self._collect(s, copy_out, n_local=n, force_copy=force_copy)
        finally:
            self.ctx.free_surface(s)

    def _collect(self, s, copy_out: bool, n_local: int, extra_ms: float = 0.0, force_copy: bool = False) -> dict:
        L = self.ctx._L
        tm = self.ctx.timings(s)
        nv, nt = L.ss_surface_num_vertices(s), L.ss_surface_num_triangles(s)
        out = {"timings": tm, "device_ms": tm["upload"] + tm["total_device"] + extra_ms, "launches": int(tm["kernel_launches"]), "nv": nv,
               "nt": nt, "nsub": L.ss_surface_num_subdomains(s), "d2h_bytes": 0}
        cnt = np.zeros(out["nsub"], np.uint64)
        owned = np.ones(out["nsub"], np.uint8)
        if out["nsub"]:
            L.ss_surface_copy_subdomains(s, None, cnt.ctypes.data, None)
            L.ss_surface_copy_subdomain_owned(s, owned.ctypes.data)
        out["memberships"] = float(cnt[owned.astype(bool)].sum())
        out["nsub_owned"] = int(owned.sum())
        if copy_out and (self.world == 1 or force_copy):          # (force_copy: the small-domain path of a multi-rank run, rank 0 holds the mesh)
            self._layout = None
            if self._out_v is None or self._out_v.numel() < nv * 3:
                self._out_v = _pinned(torch.empty(max(nv * 3, 1), dtype=torch.float32), self.device)
            if self._out_t is None or self._out_t.numel() < nt * 3:
                self._out_t = _pinned(torch.empty(max(nt * 3, 1), dtype=torch.int32), self.device)
            rc = L.ss_surface_copy_vertices(s, C.c_void_p(self._out_v.data_ptr()))
            rc |= L.ss_surface_copy_triangles_u32(s, C.c_void_p(self._out_t.data_ptr()))
            if rc:
                raise RuntimeError("mesh copy-out failed")
            out["d2h_bytes"] = nv * 12 + nt * 12
            self._out_n = None
            if force_copy and self.ctx_normals and L.ss_surface_device_normals(s):      # (the bench's single-GPU e2e reading stays as measured)
                self._out_n = np.empty((nv, 3), dtype=np.float32)
                if nv and L.ss_surface_copy_normals(s, C.c_void_p(self._out_n.ctypes.data)):
                    raise RuntimeError("normal copy-out failed")
                out["d2h_bytes"] += nv * 12
        return out

    # -- public step: `x` is this rank's (n, 3) float32 tensor (cuda, or pinned host for the end-to-end path)
    def step(self, x, n: Optional[int] = None, copy_out: bool = False) -> dict:
        if self.world == 1:
            if isinstance(x, int):
                return self._step_single(x, int(n), copy_out)
            return self._step_single(x.data_ptr(), x.shape[0], copy_out)
        return self._step_multi(x, copy_out)

    def _step_multi(self, x: torch.Tensor, copy_out: bool) -> dict:
        L, p, world, rank, dev = self.ctx._L, self.params, self.world, self.rank, self.device
        from . import _Grid
        import time
        t_ev = [_event(dev) for _ in range(3)]
        t_ev[0].record()
        t_host = [time.perf_counter()]          # host clock after each phase (every phase ends in a host sync): where the runner's time goes
        xd = x.to(dev, non_blocking=True) if x.device.type != dev.type else x
        n = int(xd.shape[0])
        S = int(p.subdomain_num_cubes_per_dim)
        # 1. global bounding box with ONE all-reduce (MAX over [-min, max]) -> the grid of ALL particles (lib.rs:476-516)
        if n:
            mn, mx = torch.aminmax(xd, dim=0)
            box = torch.cat([-mn, mx])
        else:
            box = torch.full((6,), float("-inf"), device=dev)
        dist.all_reduce(box, op=dist.ReduceOp.MAX, group=self.group)
        b = box.cpu().numpy().astype(np.float32)                    # host sync: also orders the upload before the library calls
        corners = np.ascontiguousarray(np.stack([-b[:3], b[3:]]))
        t_host.append(time.perf_counter())      # 1: bounding box
        grid = _Grid()
        gp = self.grid_params if self.grid_params is not None else p
        rc = L.ss_grid_for_reconstruction_f32(self.ctx._h, C.c_void_p(corners.ctypes.data), C.c_uint64(2), C.byref(gp), C.byref(grid))
        if rc:
            raise RuntimeError((L.ss_last_error() or b"").decode())
        ncells = [int(v) for v in grid.cells_per_dim]
        if int(p.spatial_decomposition) == 1 and int(p.auto_disable) and max(ncells) <= int(1.2 * S):
            # lib.rs:421-440: small domains take the global (non-decomposed) arithmetic -> one rank does it, the others idle
            return self._step_small_domain(xd, copy_out, t_ev)
        # 2. slab plan from the library's statistics kernel (particles per layer + occupied tiles), summed over ranks
        nsd = [(nc + S - 1) // S for nc in ncells]
        ax = int(np.argmax(nsd))
        stats = torch.empty(nsd[ax] + nsd[0] * nsd[1] * nsd[2], dtype=torch.int32, device=dev)
        if self.protocol == "stats":
            # members of every subdomain slot by the exact classifier: occupied tiles AND the global maximum population in one go
            rc = L.ss_partition_members_f32(self.ctx._h, C.c_void_p(xd.data_ptr()), C.c_uint64(n), C.byref(p), C.byref(grid), ax,
                                            C.c_void_p(stats.data_ptr()), C.c_void_p(stats.data_ptr() + 4 * nsd[ax]))
        else:
            rc = L.ss_partition_stats_f32(self.ctx._h, C.c_void_p(xd.data_ptr()), C.c_uint64(n), C.byref(grid), C.c_uint32(S), ax,
                                          C.c_void_p(stats.data_ptr()), C.c_void_p(stats.data_ptr() + 4 * nsd[ax]))
        # a failing rank still takes part in the all-reduce (and raises afterwards): nobody is left waiting
        stats_msg = (L.ss_last_error() or b"").decode() if rc else ""
        if rc:
            stats.fill_(-(1 << 20))
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=self.group)
        h = stats.cpu().numpy()
        if rc or int(h.min()) < 0:
            raise RuntimeError(f"rank {rank}: {stats_msg}" if rc else f"rank {rank}: another rank failed in the plan statistics")
        occ = (h[nsd[ax]:] > 0).reshape(nsd)
        stats_gmax = int(h[nsd[ax]:].max()) if self.protocol == "stats" else 0
        tiles = occ.sum(axis=tuple(d for d in range(3) if d != ax)).astype(np.float64)
        work = h[:nsd[ax]].astype(np.float64) + TILE_COST_PARTICLES * tiles
        # feedback from earlier frames: layers whose rank took longer than the mean weigh more (frames are temporally coherent)
        if self.balance_feedback and self._layer_scale is not None and self._layer_key == (ax, nsd[ax]):
            work = work * self._layer_scale
        else:
            self._layer_scale, self._layer_key = np.ones(nsd[ax]), (ax, nsd[ax])
            self._explore_left, self._best_t, self._best_cuts, self._frozen_cuts = self.explore_frames, float("inf"), None, None
        plan = make_plan(ncells, S, float(p.cube_size), float(p.compact_support_radius), work, world, axis=ax)
        if self.balance_feedback and self._frozen_cuts is not None:
            plan.cuts = list(self._frozen_cuts)                     # settled: same slabs as the best frame so far
        plan.gmin_axis = float(grid.aabb_min[ax])
        self.last_plan = plan
        t_host.append(time.perf_counter())      # 2: statistics + plan
        # 3. halo exchange: the library packs per destination (stable), NCCL moves it; ascending global particle order is kept
        iv = [plan.recv_interval(r) for r in range(world)]
        lo = (C.c_double * world)(*[v[0] for v in iv]); hi = (C.c_double * world)(*[v[1] for v in iv])
        counts = (C.c_uint64 * world)()
        rc = L.ss_partition_pack_f32(self.ctx._h, C.c_void_p(xd.data_ptr()), C.c_uint64(n), ax, lo, hi, C.c_uint32(world), counts, None)
        if rc:
            raise RuntimeError((L.ss_last_error() or b"").decode())
        counts = [int(v) for v in counts]
        send = torch.empty((sum(counts), 3), dtype=torch.float32, device=dev)
        if n:
            rc = L.ss_partition_pack_f32(self.ctx._h, C.c_void_p(xd.data_ptr()), C.c_uint64(n), ax, lo, hi, C.c_uint32(world), (C.c_uint64 * world)(),
                                         C.c_void_p(send.data_ptr()))
            if rc:
                raise RuntimeError((L.ss_last_error() or b"").decode())
        cnt_in = torch.tensor(counts, dtype=torch.int64, device=dev)
        cnt_out = torch.empty(world, dtype=torch.int64, device=dev)
        dist.all_to_all_single(cnt_out, cnt_in, group=self.group)
        out_counts = [int(v) for v in cnt_out.tolist()]
        recv = torch.empty((sum(out_counts), 3), dtype=torch.float32, device=dev)
        dist.all_to_all_single(recv.view(-1), send.view(-1), output_split_sizes=[3 * v for v in out_counts],
                               input_split_sizes=[3 * v for v in counts], group=self.group)
        t_ev[1].record()
        own_lo, own_hi = plan.own(rank)
        _sync(dev)                                                  # the exchange has landed before the library (own stream) reads it
        t_host.append(time.perf_counter())      # 3: pack + exchange
        # 4. this rank's slab.  The global maximum subdomain population (sparse rule, dense_subdomains.rs:1242-1251) is max-reduced
        #    from inside the call ("callback") or by a decomposition pre-pass ("two_call"); every rank issues the same collectives.
        s = C.c_void_p()
        pre_launches = 0
        failure = []
        recv_ptr = C.c_void_p(recv.data_ptr())
        if getattr(self, "_test_fail_rank", None) == rank:          # fault injection for tests/test_distributed_cpu.py: a NULL particle pointer
            recv_ptr = C.c_void_p(None)
        if self.protocol == "stats":
            rc = L.ss_reconstruct_partition_f32(self.ctx._h, recv_ptr, C.c_uint64(recv.shape[0]), C.byref(p),
                                                C.byref(grid), ax, own_lo, own_hi, plan.halo, C.c_uint64(stats_gmax), 0, C.byref(s))
        elif self.protocol == "callback":
            def _reduce(local_max, _user):
                try:
                    t = torch.tensor([int(local_max)], dtype=torch.int64, device=dev)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
                    return int(t.item())
                except BaseException as exc:                      # ctypes would swallow it: remember and re-raise after the call
                    failure.append(exc)
                    return int(local_max)
            cb = C.CFUNCTYPE(C.c_uint64, C.c_uint64, C.c_void_p)(_reduce)
            rc = L.ss_reconstruct_partition_cb_f32(self.ctx._h, recv_ptr, C.c_uint64(recv.shape[0]), C.byref(p),
                                                   C.byref(grid), ax, own_lo, own_hi, plan.halo, cb, None, C.byref(s))
        else:
            rc = L.ss_reconstruct_partition_f32(self.ctx._h, recv_ptr, C.c_uint64(recv.shape[0]), C.byref(p),
                                                C.byref(grid), ax, own_lo, own_hi, plan.halo, C.c_uint64(0), 1, C.byref(s))
            local_max = 0
            if not rc:
                local_max = L.ss_surface_max_subdomain_particles(s)
                pre_launches = int(self.ctx.timings(s)["kernel_launches"])
                self.ctx.free_surface(s)
            gmax = torch.tensor([local_max], dtype=torch.int64, device=dev)
            dist.all_reduce(gmax, op=dist.ReduceOp.MAX, group=self.group)       # issued on every rank, also after a failed pre-pass
            gmax_i = int(gmax.item())
            t_host.append(time.perf_counter())  # 4: decomposition pre-pass + max-reduce (two_call only)
            if not rc:
                s = C.c_void_p()
                rc = L.ss_reconstruct_partition_f32(self.ctx._h, C.c_void_p(recv.data_ptr()), C.c_uint64(recv.shape[0]), C.byref(p),
                                                    C.byref(grid), ax, own_lo, own_hi, plan.halo, C.c_uint64(gmax_i), 0, C.byref(s))
        # 5. the status is part of the protocol: every rank learns whether any rank failed and raises together (no rank is
        #    left waiting in a later collective)
        msg = (L.ss_last_error() or b"").decode() if rc else ""
        t_host.append(time.perf_counter())      # 5 (4 with the callback protocol): the library call
        status = torch.zeros(1 + world, dtype=torch.float64, device=dev)       # [worst return code, library ms of every rank]
        status[0] = float(int(rc) if not failure else 255)
        if not rc and not failure:
            tm = self.ctx.timings(s)      # kernel time of the stages (event-bracketed; allocation stalls of a changing plan stay out)
            status[1 + rank] = float(sum(tm[k] for k in ("decomposition", "density", "binning", "levelset", "marching_cubes", "stitching")))
        dist.all_reduce(status, op=dist.ReduceOp.MAX, group=self.group)
        status = status.cpu().numpy()
        if failure:
            raise failure[0]
        if int(status[0]):
            if s and not rc:
                self.ctx.free_surface(s)
            raise RuntimeError(f"rank {rank}: {msg}" if rc else f"rank {rank}: another rank failed (code {int(status[0])})")
        if self.balance_feedback:
            t_r = status[1:]
            busy = [r for r in range(world) if plan.own(r)[1] > plan.own(r)[0]]
            mean = float(np.mean([t_r[r] for r in busy])) if busy else 0.0
            worst = max(float(t_r[r]) for r in busy) if busy else 0.0
            if self._frozen_cuts is not None:
                # the cloud has moved on (three frames in a row 15 % slower than when the cuts were chosen; one slow frame is noise):
                # explore again
                self._drift = self._drift + 1 if worst > 1.15 * self._best_t else 0
                if self._drift >= 3:
                    self._explore_left, self._best_t, self._best_cuts, self._frozen_cuts, self._drift = max(self.explore_frames - 1, 1), float("inf"), None, None, 0
            elif mean > 0:
                if worst < self._best_t:
                    self._best_t, self._best_cuts = worst, list(plan.cuts)
                # adapt only while the slowest rank is more than 4 % above the mean
                if worst > 1.04 * mean:
                    for r in busy:
                        a, bnd = plan.own(r)
                        self._layer_scale[a:bnd] *= float(np.clip(t_r[r] / mean, 0.6, 1.6))
                    self._layer_scale = np.clip(self._layer_scale / self._layer_scale.mean(), 0.2, 5.0)
                self._explore_left -= 1
                if self._explore_left <= 0:
                    self._frozen_cuts = list(self._best_cuts)
        try:
            t_ev[2].record()
            _sync(dev)
            out = self._collect(s, False, n_local=n)
            # events on torch's stream bracket the whole step: exchange (NCCL) + the host-synchronous library calls
            out["device_ms"] = t_ev[0].elapsed_time(t_ev[2])
            out["launches"] += pre_launches
            out["recv_particles"] = int(recv.shape[0])
            out["exchange_ms"] = t_ev[0].elapsed_time(t_ev[1])
            out["plan"] = plan
            t_host.append(time.perf_counter())
            names = ["bbox", "stats_plan", "pack_exchange"] + (["prepass_maxreduce"] if self.protocol == "two_call" else []) + ["library", "status_collect"]   # noqa: E501
            out["phase_ms"] = {k: round(1e3 * (t_host[i + 1] - t_host[i]), 3) for i, k in enumerate(names) if i + 1 < len(t_host)}
            if copy_out:
                out.update(self._assemble_mesh(s, plan))
            return out
        finally:
            self.ctx.free_surface(s)

    # -- domains at most 1.2 subdomains wide (auto_disable rule): all particles go to rank 0, which takes the single-GPU entry
    def _step_small_domain(self, xd: torch.Tensor, copy_out: bool, t_ev) -> dict:
        world, rank, dev = self.world, self.rank, self.device
        sizes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([xd.shape[0]], dtype=torch.int64, device=dev), group=self.group)
        sizes = [int(v.item()) for v in sizes]
        parts = [torch.empty((m, 3), dtype=torch.float32, device=dev) for m in sizes]
        pad = max(sizes + [1])
        buf = torch.zeros((pad, 3), dtype=torch.float32, device=dev)
        buf[:xd.shape[0]] = xd
        bufs = [torch.empty_like(buf) for _ in range(world)]
        dist.all_gather(bufs, buf, group=self.group)
        allp = torch.cat([bufs[r][:sizes[r]] for r in range(world)]).contiguous()
        _sync(dev)
        out = self._step_single(allp.data_ptr(), allp.shape[0] if rank == 0 else 0, copy_out and rank == 0, params=self.grid_params,
                                force_copy=True)
        t_ev[2].record(); _sync(dev)
        out["device_ms"] = t_ev[0].elapsed_time(t_ev[2])
        out["recv_particles"] = int(allp.shape[0]) if rank == 0 else 0
        out["plan"] = SlabPlan(0, 1, [0] + [1] * world, 0, 0)
        if rank != 0:
            out.update(nv=0, nt=0, nsub=0, nsub_owned=0, memberships=0.0)
        if copy_out:
            nvnt = torch.tensor([out["nv"], out["nt"]], dtype=torch.int64, device=dev)
            dist.broadcast(nvnt, 0, group=self.group)
            out["nv_global"], out["nt_global"] = (int(nvnt[0]), int(nvnt[1])) if rank == 0 else (None, None)
            out["small_domain"] = True
        return out

    # -- shared host segment for the assembled mesh: every rank copies its part device -> host over its own PCIe link
    def _host_segment(self, nbytes: int):
        if self._seg is not None and self._seg.numel() >= nbytes:
            return self._seg
        import os
        want = int(nbytes * 1.25) + (1 << 20)
        if self.device.type != "cuda":
            self._seg = torch.empty(want, dtype=torch.uint8)       # tests on host memory: private buffer, parts gathered through gloo
            return self._seg
        self._release_segment()
        name = [f"/dev/shm/ss_b200_mesh_{os.getpid()}_{id(self) & 0xffffff:x}_{self._seg_gen}"]
        self._seg_gen += 1
        dist.broadcast_object_list(name, src=0, group=self.group)  # rank 0 names the segment
        name = name[0]
        if self.rank == 0:
            with open(name, "wb") as f:
                f.truncate(want)
        dist.barrier(group=self.group)
        self._seg = torch.from_file(name, shared=True, size=want, dtype=torch.uint8)
        # page-locked: asynchronous device -> host copies at link speed, all ranks in parallel
        err = torch.cuda.cudart().cudaHostRegister(self._seg.data_ptr(), want, 0)
        self._seg_registered = (int(err) == 0) if err is not None else True
        dist.barrier(group=self.group)
        if self.rank == 0:
            os.unlink(name)                                        # the mappings keep the segment alive
        return self._seg

    def _release_segment(self):
        if self._seg is not None and self._seg_registered and self.device.type == "cuda":
            torch.cuda.synchronize()
            torch.cuda.cudart().cudaHostUnregister(self._seg.data_ptr())
        self._seg = None; self._seg_registered = False; self._layout = None

    def close(self):
        """Releases the shared host segment (unregisters it before the mapping goes away)."""
        self._release_segment()

    def __del__(self):
        try:
            self._release_segment()
        except Exception:
            pass

    # -- mesh assembly: duplicates on the faces between slabs are resolved against the LOWER neighbour by MC edge key (the copy
    #    of the lowest subdomain wins, as in the single-GPU weld), global vertex ids are rank-major, and every rank writes its own
    #    vertices / triangles into the shared host segment.  Only face keys and a few counters travel between GPUs.
    def _assemble_mesh(self, s, plan: SlabPlan) -> dict:
        L, world, rank, dev = self.ctx._L, self.world, self.rank, self.device
        nv, nt = L.ss_surface_num_vertices(s), L.ss_surface_num_triangles(s)
        v = _view(L.ss_surface_device_vertices(s), (nv, 3), "<f4", dev)
        t = _view(L.ss_surface_device_triangles(s), (nt, 3), "<u4", dev)
        k = _view(L.ss_surface_device_vertex_keys(s), (nv,), "<u8", dev)
        S = int(self.params.subdomain_num_cubes_per_dim)
        shift = (42, 22, 2)[plan.axis]
        own_lo, own_hi = plan.own(rank)
        coord = (k >> shift) & 0xFFFFF
        onface = (k & 3) != plan.axis
        up_idx = torch.nonzero(onface & (coord == own_hi * S)).view(-1)        # my vertices a higher rank may duplicate
        lo_idx = torch.nonzero(onface & (coord == own_lo * S)).view(-1) if own_lo > 0 else up_idx[:0]
        # round 1: sizes
        sz = torch.tensor([nv, nt, up_idx.numel()], dtype=torch.int64, device=dev)
        all_sz = [torch.empty_like(sz) for _ in range(world)]
        dist.all_gather(all_sz, sz, group=self.group)
        all_sz = torch.stack(all_sz).cpu().numpy()
        fmax = max(int(all_sz[:, 2].max()), 1)
        # round 2: upper-face keys of every rank
        mine = torch.full((fmax,), -1, dtype=torch.int64, device=dev)
        mine[:up_idx.numel()] = k[up_idx]
        allk = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allk, mine, group=self.group)
        # my duplicates: lower-face vertices whose key a lower rank published
        keep = torch.ones(nv, dtype=torch.bool, device=dev)
        dup_src_rank = dup_src_pos = None
        if rank > 0 and lo_idx.numel():
            lower = torch.cat([allk[q][:int(all_sz[q, 2])] for q in range(rank)])
            owner = torch.cat([torch.full((int(all_sz[q, 2]),), q, dtype=torch.int64, device=dev) for q in range(rank)])
            posin = torch.cat([torch.arange(int(all_sz[q, 2]), dtype=torch.int64, device=dev) for q in range(rank)])
            if lower.numel():
                sk, order = torch.sort(lower)
                mykeys = k[lo_idx]
                pos = torch.searchsorted(sk, mykeys).clamp(max=sk.numel() - 1)
                hit = sk[pos] == mykeys
                dup_v = lo_idx[hit]
                keep[dup_v] = False
                dup_src_rank, dup_src_pos = owner[order[pos[hit]]], posin[order[pos[hit]]]
        newid = torch.cumsum(keep, 0, dtype=torch.int64) - 1                     # compacted local ids
        nkeep = int(newid[-1].item()) + 1 if nv else 0
        # round 3: kept counts + compacted ids of my upper-face vertices (they are never dropped: different plane)
        pub = torch.full((fmax + 1,), -1, dtype=torch.int64, device=dev)
        pub[0] = nkeep
        pub[1:1 + up_idx.numel()] = newid[up_idx]
        allp = [torch.empty_like(pub) for _ in range(world)]
        dist.all_gather(allp, pub, group=self.group)
        nkeeps = [int(a[0].item()) for a in allp]
        voff = [0]
        for q in range(world):
            voff.append(voff[-1] + nkeeps[q])
        toff = [0]
        for q in range(world):
            toff.append(toff[-1] + int(all_sz[q, 1]))
        nvg, ntg = voff[-1], toff[-1]
        gid = newid + voff[rank]
        if dup_src_rank is not None and dup_src_rank.numel():
            table = torch.stack([a[1:] for a in allp])                            # (world, fmax) compacted local ids of upper-face vertices
            offs = torch.tensor(voff[:-1], dtype=torch.int64, device=dev)
            gid[dup_v] = table[dup_src_rank, dup_src_pos] + offs[dup_src_rank]
        tg = gid[t.to(torch.int64).view(-1)].to(torch.int32) if nt else torch.empty(0, dtype=torch.int32, device=dev)
        vk = v[keep].contiguous()
        want_keys = self.want_keys
        nptr = L.ss_surface_device_normals(s)                                     # SPH normals travel with the vertices when they were computed
        has_n = torch.tensor([1 if (nptr or nv == 0) else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(has_n, op=dist.ReduceOp.MIN, group=self.group)
        has_n = bool(int(has_n.item())) and bool(self.ctx_normals)
        nbytes = nvg * 12 + ntg * 12 + (nvg * 8 if want_keys else 0) + 8 + (nvg * 12 if has_n else 0)
        seg = self._host_segment(nbytes + 64)
        self._layout = (nvg, ntg, want_keys, has_n)
        sv = seg[:nvg * 12].view(torch.float32)
        st = seg[nvg * 12:nvg * 12 + ntg * 12].view(torch.int32)
        if dev.type == "cuda":
            sv[voff[rank] * 3:voff[rank + 1] * 3].copy_(vk.view(-1), non_blocking=True)
            st[toff[rank] * 3:toff[rank + 1] * 3].copy_(tg, non_blocking=True)
            if want_keys:
                base = (nvg * 12 + ntg * 12 + 7) // 8 * 8
                seg[base:base + nvg * 8].view(torch.int64)[voff[rank]:voff[rank + 1]].copy_(k[keep], non_blocking=True)
            if has_n:
                nbase = ((nvg * 12 + ntg * 12 + 7) // 8 * 8) + (nvg * 8 if want_keys else 0)
                nk = _view(nptr, (nv, 3), "<f4", dev)[keep].contiguous() if nv else torch.empty((0, 3), dtype=torch.float32, device=dev)
                seg[nbase:nbase + nvg * 12].view(torch.float32)[voff[rank] * 3:voff[rank + 1] * 3].copy_(nk.view(-1), non_blocking=True)
            _sync(dev)
            dist.barrier(group=self.group)                                        # every part has landed in the shared segment
        else:
            # host-memory runs (tests): no shared segment, rank 0 gathers the parts through the process group
            parts_v = [torch.empty(nkeeps[q] * 3, dtype=torch.float32) for q in range(world)]
            parts_t = [torch.empty(int(all_sz[q, 1]) * 3, dtype=torch.int32) for q in range(world)]
            parts_k = [torch.empty(nkeeps[q], dtype=torch.int64) for q in range(world)]
            pad_v, pad_t = max(nkeeps + [1]) * 3, max(int(all_sz[:, 1].max()), 1) * 3
            bv = torch.zeros(pad_v, dtype=torch.float32); bv[:nkeep * 3] = vk.view(-1)
            bt = torch.zeros(pad_t, dtype=torch.int32); bt[:nt * 3] = tg
            bk = torch.zeros(pad_v // 3, dtype=torch.int64); bk[:nkeep] = k[keep]
            gv = [torch.empty_like(bv) for _ in range(world)]; gt = [torch.empty_like(bt) for _ in range(world)]; gk = [torch.empty_like(bk) for _ in range(world)]
            dist.all_gather(gv, bv, group=self.group); dist.all_gather(gt, bt, group=self.group); dist.all_gather(gk, bk, group=self.group)
            for q in range(world):
                sv[voff[q] * 3:voff[q + 1] * 3] = gv[q][:nkeeps[q] * 3]
                st[toff[q] * 3:toff[q + 1] * 3] = gt[q][:int(all_sz[q, 1]) * 3]
            if want_keys:
                base = (nvg * 12 + ntg * 12 + 7) // 8 * 8
                sk8 = seg[base:base + nvg * 8].view(torch.int64)
                for q in range(world):
                    sk8[voff[q]:voff[q + 1]] = gk[q][:nkeeps[q]]
        res = {"d2h_bytes": nkeep * 12 + nt * 12 + (nkeep * 12 if has_n else 0), "has_normals": has_n, "nv_global": nvg if rank == 0 else None, "nt_global": ntg if rank == 0 else None,
               "nv_total": nvg, "nt_total": ntg}
        if want_keys and rank == 0:
            base = (nvg * 12 + ntg * 12 + 7) // 8 * 8
            res["keys_global"] = seg[base:base + nvg * 8].view(torch.int64).clone()
        return res

    def gathered_mesh(self, nv: int, nt: int):
        """Host copies of the last assembled mesh (any rank can read the shared segment; tests: rank 0)."""
        if getattr(self, "_layout", None) is None:              # single-GPU / small-domain path
            return self._out_v[:nv * 3].view(-1, 3).numpy().copy(), self._out_t[:nt * 3].view(-1, 3).numpy().copy()
        seg = self._seg
        return seg[:nv * 12].view(torch.float32).view(-1, 3).numpy().copy(), seg[nv * 12:nv * 12 + nt * 12].view(torch.int32).view(-1, 3).numpy().copy()



# ------------------------------------------------------------------------------------ user-facing call (one frame, N GPUs) ----
class DistributedReconstructor:
    """`reconstruct_surface` for ONE particle cloud spread over the ranks of a process group (one process per GPU).

    Every rank passes the particles it holds -- any split of the cloud into contiguous index ranges in rank order (the order matters
    for bit-identical results: the reference sums in ascending particle index); empty parts are fine.  The call is collective.  Rank 0
    gets the assembled mesh (vertices, triangles, SPH normals when `sph_normals`), identical to the single-GPU result; the other ranks
    get None.  Keep the object for a frame sequence: the slab plan settles after a few frames and the buffers are reused.

    The reference has no counterpart (it parallelises over subdomains with rayon inside one process, dense_subdomains.rs:521-526);
    parameters are those of `pysplashsurf.reconstruct_surface`.  A particle AABB (`aabb_min` / `aabb_max`) defines the grid like in the
    reference (lib.rs:476-516) and filters every rank's particles before the exchange; the mesh post-processing of
    `reconstruction_pipeline` is a single-GPU step."""

    def __init__(self, *, sph_normals: bool = False, group=None, device=None, protocol: str = "stats", local_rank: Optional[int] = None,
                 anisotropic: bool = False, **params):
        import os
        import splashsurf_b200 as ss
        if anisotropic:
            # each rank would need its ghost particles' kernel centres, which the one-exchange halo does not carry
            raise ValueError("anisotropic kernels are not available in distributed reconstructions")
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed is not initialised: launch one process per GPU (torchrun) and call init_process_group first")
        self._ss, self._kw = ss, dict(params)
        self._aabb = None
        if params.get("aabb_min") is not None and params.get("aabb_max") is not None:
            self._aabb = (np.asarray(params["aabb_min"], np.float64).astype(np.float32), np.asarray(params["aabb_max"], np.float64).astype(np.float32))
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        lr = int(os.environ.get("LOCAL_RANK", "0")) if local_rank is None else int(local_rank)
        self.ctx = ss.Context(lr if device is None else 0)
        self.sph_normals = bool(sph_normals)
        if self.sph_normals:
            ss._check(self.ctx._L, self.ctx._L.ss_context_set_compute_sph_normals(self.ctx._h, 1))
        no_box = {k: v for k, v in params.items() if k not in ("aabb_min", "aabb_max")}
        self.runner = Runner(self.ctx, ss.make_params(**no_box), self.world, self.rank, lr, group=group, device=device, protocol=protocol)
        self.runner.ctx_normals = self.sph_normals
        if self._aabb is not None:
            self.runner.grid_params = ss.make_params(**params)

    def __call__(self, particles_local: np.ndarray):
        ss = self._ss
        p = np.ascontiguousarray(particles_local, dtype=np.float32).reshape(-1, 3)
        if self.world == 1:
            r = ss.reconstruct_surface(p, context=self.ctx, sph_normals=self.sph_normals, **self._kw)
            return ss.MeshWithData(r.mesh, {"normals": r.normals} if self.sph_normals and r.normals is not None else {}, {})
        if self._aabb is not None:                    # lib.rs:369-406: particles outside the half-open box take no part
            p = np.ascontiguousarray(p[np.all(p >= self._aabb[0], axis=1) & np.all(p < self._aabb[1], axis=1)])
        total = torch.tensor([len(p)], dtype=torch.int64, device=self.runner.device)
        dist.all_reduce(total, group=self.runner.group)
        if int(total.item()) == 0:                    # no particle anywhere: an empty mesh, like the single-device call returns
            return ss.MeshWithData(ss.TriMesh3d(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint64)), {}, {}) if self.rank == 0 else None
        x = torch.from_numpy(p)                       # pageable: the runner's upload stages it (a page-locked tensor is taken as it is)
        out = self.runner.step(x, copy_out=True)
        if self.rank != 0:
            return None
        v, t = self.runner.gathered_mesh(out["nv_global"], out["nt_global"])
        attrs = {}
        n = self.runner.gathered_normals()
        if n is not None:
            attrs["normals"] = n
        return ss.MeshWithData(ss.TriMesh3d(v, t.view(np.uint32).astype(np.uint64)), attrs, {})

    def close(self):
        self.runner.close()
        self.ctx.close()
