"""View-sharded densification: one process per GPU, views in contiguous blocks.

Stage 1 is independent per view and stage 2 per pixel; stage 3 needs read-only access to the refined
depth of each source view's K neighbours, stage 4 is a global group-by on the voxel key
(SURVEY.md §8e).  So there are exactly two exchange steps:

* halo exchange of refined depth: a rank receives only the neighbour views its own rows of the
  neighbour table reference (with ring-ordered cameras that is <= K maps per shard boundary instead
  of the all-gather of all V maps);
* voxel exchange: every rank fuses its own points into per-voxel PARTIAL SUMS (integer fixed point,
  so the result does not depend on how points are split over ranks); the grid's tiles are cut into R
  contiguous ranges that balance the global record count - each rank owns one disjoint key range, so a
  destination's share of a rank's sorted records is one contiguous slice and needs no pack kernel - and
  the owner adds up what the R ranks hold for its range.

Two implementations of the same steps:

* the DEVICE path (CUDA): no host round trip anywhere in a step.  The grid is derived on the device from
  the bounding boxes the alignment kernels produce (all ranks' boxes are read through NVLink peer
  memory), the consistency kernel marks the occupancy of the points it keeps, and the owner-side merge
  pulls its share of every rank's partial records straight out of their HBM inside its own kernels
  (ddn_fuse_merge_peers: coalesced NVLink loads, peers visited in rotated order) - no host-side plan;
* the COLLECTIVE path (all-to-all-v over torch.distributed; host-side grid and plan): what the gloo tests
  drive on CPU with a stand-in backend, and the fallback when symmetric memory cannot be set up.

With world == 1 both exchanges vanish and this is the single-GPU pipeline.
"""

from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import torch

from . import ops
from .engine import DensifyConfig, DensifyResult, max_sparse_count


def shard_bounds(n_views: int, world: int) -> list[tuple[int, int]]:
    """Contiguous equal shards [lo, hi) per rank (the last ranks may be short or empty)."""
    per = (n_views + world - 1) // world
    return [(min(r * per, n_views), min((r + 1) * per, n_views)) for r in range(world)]


@dataclass
class HaloPlan:
    """Who sends which refined-depth maps to whom; computed identically on every rank from the
    replicated neighbour table, so no communication is needed to build it."""

    slots: np.ndarray  # global view id of every local slot: own views first, then halo views
    nbr_slots: np.ndarray  # [n_local, K] neighbour table in slot space (-1 = unused)
    send_views: list[np.ndarray]  # per peer: LOCAL indices of own views to send
    recv_counts: list[int]  # per peer: number of halo views received (stored in slot order)

    @property
    def n_local(self) -> int:
        return self.nbr_slots.shape[0]


def needed_views(nbr: np.ndarray, lo: int, hi: int) -> np.ndarray:
    need = np.unique(nbr[lo:hi])
    return need[need >= 0]


def make_halo_plan(nbr: np.ndarray, bounds: list[tuple[int, int]], rank: int) -> HaloPlan:
    lo, hi = bounds[rank]
    world = len(bounds)

    def owner(v: int) -> int:
        for r, (a, b) in enumerate(bounds):
            if a <= v < b:
                return r
        raise ValueError(f"view {v} has no owner")

    need = needed_views(nbr, lo, hi)
    halo = [int(v) for v in need if not (lo <= v < hi)]
    halo_by_peer: list[list[int]] = [[] for _ in range(world)]
    for v in halo:
        halo_by_peer[owner(v)].append(v)
    halo_sorted = [v for q in range(world) for v in sorted(halo_by_peer[q])]
    slots = np.array(list(range(lo, hi)) + halo_sorted, dtype=np.int64)
    slot_of = {int(v): i for i, v in enumerate(slots)}
    nbr_slots = np.full((hi - lo, nbr.shape[1]), -1, dtype=np.int32)
    for i in range(hi - lo):
        for k, t in enumerate(nbr[lo + i]):
            if t >= 0:
                nbr_slots[i, k] = slot_of[int(t)]
    send_views = []
    for q in range(world):
        qlo, qhi = bounds[q]
        if q == rank or qhi <= qlo:
            send_views.append(np.zeros(0, dtype=np.int64))
            continue
        qneed = needed_views(nbr, qlo, qhi)
        mine = np.array(sorted(int(v) for v in qneed if lo <= v < hi), dtype=np.int64)
        send_views.append(mine - lo)
    return HaloPlan(slots=slots, nbr_slots=nbr_slots, send_views=send_views, recv_counts=[len(h) for h in halo_by_peer])


@dataclass
class ShardResult(DensifyResult):
    events: dict = field(default_factory=dict)


class PeerMemory:
    """NVLink peer access through torch symmetric memory: every rank allocates the same buffer, the
    rendezvous maps all of them into every process, and a rank then READS what it needs straight out of
    its peers' HBM with copy-engine transfers bracketed by device-side barriers.  On 2 x B200 a 178 MB
    exchange runs at 665 GB/s this way against 309 GB/s for NCCL all_to_all_single
    (scripts/experiments/a2a_probe.py), and there is no send-side packing at all."""

    def __init__(self, group, device):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm

        self._symm, self.group, self.device = symm, group if group is not None else dist.group.WORLD, device
        self.world = dist.get_world_size(self.group)
        self.bufs = {}

    def buffer(self, name: str, shape, dtype):
        """The local symmetric buffer `name` (allocated collectively on first use) and the peers' views."""
        key = (name, tuple(shape), dtype)
        if key not in self.bufs:
            t = self._symm.empty(*shape, dtype=dtype, device=self.device)
            hdl = self._symm.rendezvous(t, self.group)
            views = [hdl.get_buffer(q, tuple(shape), dtype) for q in range(self.world)]
            self.bufs[key] = (t, hdl, views)
        return self.bufs[key]


class ShardedDensifier:
    """Pipeline of one rank.  ``cam_from_world`` / ``intr`` cover ALL views (replicated, tiny);
    the per-view maps passed to ``run`` cover the rank's own views [lo, hi)."""

    def __init__(self, cfg: DensifyConfig, device, rank: int, world: int, n_views_total: int, lo: int, hi: int,
                 cam_from_world: torch.Tensor, intr: torch.Tensor, nbr: np.ndarray, height: int, width: int, group=None,
                 backend=None):
        # `backend` is the module providing the device ops; the product always uses `ops` (CUDA, no CPU
        # fallback).  Tests inject an object with the same functions to exercise the exchange logic on
        # CPU with the gloo backend.
        if backend is None:
            if not torch.cuda.is_available():
                raise ops.DDNError("ShardedDensifier needs a CUDA device: depthdensifier_b200 has no CPU fallback")
            backend = ops
        self.ops = backend
        self.cfg = cfg
        self.device = torch.device(device)
        self.rank, self.world, self.group = rank, world, group
        self.V, self.lo, self.hi, self.H, self.W = n_views_total, lo, hi, height, width
        self.K = nbr.shape[1]
        self.thr = cfg.vote_threshold_for(self.K)
        self.fthr = ops.fusion_threshold(self.thr, cfg.min_support is not None)  # what fusion tests the vote bytes with
        bounds = shard_bounds(n_views_total, world) if world > 1 else [(lo, hi)]
        if world > 1 and bounds[rank] != (lo, hi):
            raise ValueError(f"rank {rank}: shard {(lo, hi)} does not match the contiguous layout {bounds[rank]}")
        self.plan = make_halo_plan(nbr, bounds, rank if world > 1 else 0)
        slots = torch.from_numpy(self.plan.slots).to(self.device)
        self.poses_slots = cam_from_world.to(self.device)[slots].contiguous()
        self.intr_slots = intr.to(self.device)[slots].contiguous()
        self.nbr_slots = torch.from_numpy(self.plan.nbr_slots).to(self.device).contiguous()
        self.n_local = hi - lo
        self.n_slots = len(self.plan.slots)
        self.kmat = ops.intrinsics_matrix(self.intr_slots[: self.n_local])
        self._max_sparse = None
        self._host_out = None
        # NVLink peer reads for the two exchange steps (CUDA, world > 1); the collective path (all-to-all-v)
        # remains for the gloo tests and as the fallback when symmetric memory cannot be set up
        self.peer = None
        self.bounds = bounds
        self.device_path = self.device.type == "cuda" and backend is ops  # sync-free fusion sessions
        self.session = None
        self._tables = None
        s0 = cfg.filter.stride
        self.Hs, self.Ws = (height + s0 - 1) // s0, (width + s0 - 1) // s0
        self._local_max = max(b - a for a, b in bounds)
        if world > 1 and self.device_path:
            try:
                self.peer = PeerMemory(group, self.device)
                plans = [make_halo_plan(nbr, bounds, q) for q in range(world)]
                self._slots_max = max(len(pl.slots) for pl in plans)
                self._local_max = max(b - a for a, b in bounds)
                # which peer owns each of my halo slots, and its index there
                self._halo_src = []
                for j, v in enumerate(self.plan.slots[self.n_local:]):
                    q = next(i for i, (a, b) in enumerate(bounds) if a <= v < b)
                    self._halo_src.append((self.n_local + j, q, int(v) - bounds[q][0]))
                self._side = torch.cuda.Stream(device=self.device)
                # allocate and map both exchange buffers now (collective): a platform without symmetric memory
                # fails here, on every rank alike, and the collectives take over
                s_ = cfg.filter.stride
                self.peer_records_shape = (self._local_max * ((height + s_ - 1) // s_) * ((width + s_ - 1) // s_), 6)
                # refined maps and bounding boxes are double-buffered (step parity): a rank may start aligning step i+1
                # while a peer still pulls its step-i maps, so a step needs no barrier at its start
                self._parity = 0
                for par in (0, 1):
                    self.peer.buffer(f"refined{par}", (self._slots_max, self.H, self.W), torch.float32)
                    self.peer.buffer(f"bbox{par}", (64,), torch.int32)
                if cfg.voxel is not None:
                    self.peer.buffer("records", self.peer_records_shape, torch.int64)
                    self._make_session()
            except Exception as e:  # pragma: no cover - depends on the platform
                print(f"[depthdensifier_b200] symmetric memory unavailable ({e!r}); using NCCL collectives")
                self.peer = None
                self.session = None
            if self.peer is None:
                self.device_path = False
        elif self.device_path and cfg.voxel is not None:
            self._make_session()

    def _make_session(self) -> None:
        """Fusion session of this rank; with peers its tile prefix (and the partial records) live in symmetric memory
        so the owner-side merge of every other rank can read them over NVLink."""
        cfg = self.cfg
        if self.peer is None:
            self.session = ops.FuseSession(self.device, cfg.max_grid_cells)
            return

        def alloc(name, nbytes):
            if name == "tile_prefix":
                return self.peer.buffer("fuse_" + name, (nbytes,), torch.uint8)[0]
            return None

        self.session = ops.FuseSession(self.device, cfg.max_grid_cells, tile_prefix=True, alloc=alloc)
        ptrs = lambda name, shape, dt: [int(v.data_ptr()) for v in self.peer.buffer(name, shape, dt)[2]]
        self._peer_prefix = ptrs("fuse_tile_prefix", (self.session.tile_prefix.numel(),), torch.uint8)
        self._peer_records = ptrs("records", tuple(self.peer_records_shape), torch.int64)
        self._peer_samples = ptrs("hash_samples", (ops._lib.HASH_SAMPLES + 1,), torch.int64)
        self._peer_bbox = [ptrs(f"bbox{par}", (64,), torch.int32) for par in (0, 1)]
        self._plan = torch.zeros(64, dtype=torch.int64, device=self.device)
        # a rank's share of the merged voxels: the cuts balance the global record count, up to one tile per rank
        # (the hashed merge: its sampled splitters balance the global record count up to hashed_merge_capacity)
        n_max = self._local_max * self.Hs * self.Ws
        self._cap_merge = max(n_max + 24576 * self.world + 1024, ops.hashed_merge_capacity(n_max, self.world))
        self._merge_out = [ops.new_voxel_outputs(self._cap_merge, self.device), None]  # second set: pipelined host calls
        self.session.merge_scratch(self.world, self._cap_merge)

    # -- exchange steps -------------------------------------------------------------------------------
    def _exchange_halo(self, refined_slots: torch.Tensor) -> None:
        """Fill refined_slots[n_local:] with the neighbour maps owned by other ranks (all-to-all-v)."""
        if self.world == 1:
            return
        import torch.distributed as dist

        hw = self.H * self.W
        send_idx = np.concatenate(self.plan.send_views) if self.plan.send_views else np.zeros(0, np.int64)
        if len(send_idx):
            send = refined_slots[torch.from_numpy(send_idx).to(self.device)].reshape(-1)
        else:
            send = refined_slots.new_empty(0)
        recv = refined_slots[self.n_local:].reshape(-1)
        dist.all_to_all_single(recv, send, output_split_sizes=[c * hw for c in self.plan.recv_counts],
                               input_split_sizes=[len(s) * hw for s in self.plan.send_views], group=self.group)

    def _interior_range(self) -> tuple[int, int]:
        """Longest run [i0, i1) of own source views whose neighbours are all own views (no halo needed)."""
        if getattr(self, "_interior", None) is None:
            self._interior = self._find_interior_range()
        return self._interior

    def _find_interior_range(self) -> tuple[int, int]:
        local = ((self.plan.nbr_slots < self.n_local)).all(axis=1)
        best, i = (0, 0), 0
        n = self.n_local
        while i < n:
            if local[i]:
                j = i
                while j < n and local[j]:
                    j += 1
                if j - i > best[1] - best[0]:
                    best = (i, j)
                i = j
            else:
                i += 1
        return best

    def _pull_halo_async(self, refined_slots):
        """Halo exchange over peer memory: after a device-side barrier (every rank's refined maps are in
        place) the neighbour maps are pulled from the peers' HBM on a side stream, so the caller can keep
        the main stream busy with the source views that need no halo.  Returns the join function."""
        _, hdl, views = self.peer.buffer(f"refined{self._parity}", (self._slots_max, self.H, self.W), torch.float32)
        cur = torch.cuda.current_stream(self.device)
        hdl.barrier()  # every rank's refined maps and bounding box of this step are in place
        if self.cfg.overlap_align:
            self._ev_stage1_may_start = torch.cuda.Event()
            self._ev_stage1_may_start.record(cur)
        self._side.wait_stream(cur)
        with torch.cuda.stream(self._side):
            for slot, q, j in self._halo_src:
                refined_slots[slot].copy_(views[q][j], non_blocking=True)
        return lambda: cur.wait_stream(self._side)

    def _global_bbox(self, bbox: torch.Tensor) -> np.ndarray:
        bb = self.ops.decode_bbox(bbox) if self.world == 1 else None
        if self.world > 1:
            import torch.distributed as dist

            # order-preserving int encoding: min/max of the encodings == encodings of the min/max; ~x reverses
            # the order without overflow, so ONE all-reduce(MIN) over (lo, ~hi) does both
            both = torch.cat([bbox[:3], ~bbox[3:]])
            dist.all_reduce(both, op=dist.ReduceOp.MIN, group=self.group)
            bb = self.ops.decode_bbox(torch.cat([both[:3], ~both[3:]]))
        return bb

    # -- pipeline ---------------------------------------------------------------------------------------
    def run(self, depth, normal, mask, rgb, sparse_xyz, sparse_offsets, record_events: bool = False, grid=None) -> ShardResult:
        """One step on device-resident inputs of the rank's own views.  On the device path nothing in here waits
        for the GPU: validate with ``ShardResult.check()`` (or read ``counts``) when the results are needed."""
        cfg = self.cfg
        ev = {}

        def mark(name, fn):
            if not record_events or self.device.type != "cuda":
                return fn()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = fn()
            b.record()
            ev[name] = (a, b)
            return out

        if self._max_sparse is None:
            self._max_sparse = max_sparse_count(sparse_offsets)
        fuse = cfg.voxel is not None

        def stage1():
            refined_slots = self._new_refined_slots()
            pair, src = mark("pair_tables", self._pair_tables)
            box = self._new_box() if (self.device_path and fuse and grid is None) else None
            _, stats = mark("align", lambda: self.ops.align_views(
                depth, mask, self.poses_slots[: self.n_local].contiguous(), self.kmat, sparse_xyz, sparse_offsets,
                self._max_sparse, cfg.align, out=refined_slots[: self.n_local], **self._box_args(src, box)))
            return refined_slots, pair, src, box, stats

        if self.device_path and cfg.overlap_align:
            # Stage 1 on its own stream.  It may start as soon as the PREVIOUS step has passed its halo barrier (one
            # rank: has launched its K4) - from then on nobody reads the buffers it writes (the other parity's maps
            # and box) - and then fills whatever the main stream leaves idle.  (Holding it back until the previous
            # step starts its merge was measured on 8 GPUs: strong cfg 3 3.38 instead of 3.42 ms, but weak cfg 2 11.5
            # instead of 9.9 ms - a whole K3 beside the record pull slows the pull, and every rank then waits.)
            main = torch.cuda.current_stream(self.device)
            if getattr(self, "_align_stream", None) is None:
                self._align_stream, self._ev_stage1_may_start = torch.cuda.Stream(device=self.device), None
            side = self._align_stream
            if self._ev_stage1_may_start is None:
                side.wait_stream(main)
            else:
                side.wait_event(self._ev_stage1_may_start)
            with torch.cuda.stream(side):
                refined_slots, pair, src, box, stats = stage1()
                done = torch.cuda.Event()
                done.record(side)
            main.wait_event(done)
            for t in (refined_slots, pair, src, box, stats):
                if t is not None and t.is_cuda:
                    t.record_stream(main)
        else:
            refined_slots, pair, src, box, stats = stage1()
        xyz, votes, bbox, support = self._halo_and_filter(refined_slots, normal, mark, pair, src, box=box, grid=grid)
        res = ShardResult(refined=refined_slots[: self.n_local], stats=stats, xyz=xyz, votes=votes, vote_threshold=self.thr,
                          bbox=bbox, events=ev, support=support, min_support=cfg.min_support)
        if not fuse:
            return res
        s = cfg.filter.stride
        rgb_s = rgb if s == 1 else rgb[:, ::s, ::s].contiguous()
        if self.device_path:
            drop = self._sparse_for_dedup(sparse_xyz) if cfg.dedup_sparse else None
            k, x, c, n, counts = mark("voxel_fuse", lambda: self._fuse_device(xyz, rgb_s, votes, mark, drop))
            res.session, res.grid, res.hash = self.session, grid, self._hash
            res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count, res.counts = k, x, c, n, counts
            return res
        # collective path: the grid is made on the host from the (all-reduced) box of the kept points
        if grid is None:
            bb = mark("bbox_sync", lambda: self._global_bbox(bbox))
            if not np.all(np.isfinite(bb)):
                res.counts = torch.zeros(2, dtype=torch.int64, device=self.device)
                return res
            grid = self.ops.make_grid(bb[:3], bb[3:], cfg.voxel)
        if self.world == 1:
            k, x, c, n, counts = mark("voxel_fuse", lambda: self.ops.voxel_fuse(
                xyz.view(-1, 3), rgb_s.view(-1, 3), votes.view(-1), self.fthr, grid, trim=False, row_len=xyz.shape[2]))
        else:
            k, x, c, n, counts = mark("voxel_fuse", lambda: self._fuse_sharded(xyz, rgb_s, votes, grid, mark))
        res.grid, res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count, res.counts = grid, k, x, c, n, counts
        return res

    def _pair_tables(self):
        return self.ops.build_pair_tables(self.poses_slots, self.intr_slots, self._nbr_full(), 0, self.n_local, self.H, self.W)

    def _new_box(self) -> torch.Tensor:
        """Bounding box of this rank's back-projected pixels (filled by the alignment kernel); in peer-visible
        memory when there are peers, whose boxes the grid kernel reads directly."""
        if self.peer is not None:
            buf = self.peer.buffer(f"bbox{self._parity}", (64,), torch.int32)[0]
            return ops.init_bbox(buf[:6])
        return self.ops.new_bbox(self.device)

    @staticmethod
    def _box_args(src, box, c0=None, c1=None):
        if box is None:
            return {}
        return {"src_table": src if c0 is None else src[c0:c1], "bbox": box}

    def _begin_session(self, box, grid) -> None:
        """Opens the fusion step (stream-ordered after the barrier that made every rank's box visible)."""
        if grid is not None:
            self.session.begin_grid(grid)
        elif self.peer is not None:
            self.session.begin(self._peer_bbox[self._parity], self.cfg.voxel)
        else:
            self.session.begin([box], self.cfg.voxel)

    def _new_refined_slots(self) -> torch.Tensor:
        """[n_slots,H,W] buffer for own + halo refined maps; NVLink-visible when peer memory is in use."""
        if self.peer is not None:
            # No barrier at the start of a step.  The maps and the box written now belong to the OTHER parity than
            # the ones peers may still be reading (they were last used two steps ago, and every peer has since passed
            # the halo barrier of the previous step, which it reaches only after it is done with them); the occupancy
            # units and partial records are only overwritten after THIS step's halo barrier, which a peer reaches
            # only after its merge of the previous step has finished.  The returned maps stay valid for two steps.
            self._parity ^= 1
            buf = self.peer.buffer(f"refined{self._parity}", (self._slots_max, self.H, self.W), torch.float32)[0]
            return buf[: self.n_slots]
        return torch.empty((self.n_slots, self.H, self.W), dtype=torch.float32, device=self.device)

    def _halo_and_filter(self, refined_slots, normal, mark, pair, src, wait_normal=None, box=None, grid=None):
        """Halo exchange + stages 2-3.  With peer memory the halo maps are pulled on a side stream while K4
        already runs on the source views whose neighbours are all local.  On the device path the fusion step is
        opened in between (the grid needs every rank's box: same barrier as the halo) and K4 marks the occupancy
        of the points it keeps."""
        cfg = self.cfg
        join_halo = None
        if self.peer is not None:
            join_halo = mark("halo_exchange", lambda: self._pull_halo_async(refined_slots))
        else:
            mark("halo_exchange", lambda: self._exchange_halo(refined_slots))
        sess = None
        if self.device_path and cfg.voxel is not None:
            mark("fuse_begin", lambda: self._begin_session(box, grid))
            sess = self.session
        bbox = self.ops.new_bbox(self.device) if not self.device_path or sess is None else None
        xyz = torch.empty((self.n_local, self.Hs, self.Ws, 3), dtype=torch.float32, device=self.device)
        votes = torch.empty((self.n_local, self.Hs, self.Ws), dtype=torch.uint8, device=self.device)
        support = None if cfg.min_support is None else torch.empty_like(votes)
        if wait_normal is not None:
            wait_normal()
        extra = {"mark": sess} if self.device_path else {}

        def k4(c0, c1):
            if c1 <= c0:
                return
            whole = c0 == 0 and c1 == self.n_local
            sup = {} if support is None else {"support": cfg.support(), "support_out": support[c0:c1]}
            self.ops.backproject_filter(refined_slots, normal if whole else normal[c0:c1], self.nbr_slots,
                                        pair if whole else pair[c0:c1], src if whole else src[c0:c1], c0, self.thr, cfg.filter,
                                        bbox=bbox, xyz_out=xyz[c0:c1], votes_out=votes[c0:c1], **extra, **sup)

        if join_halo is not None:
            i0, i1 = self._interior_range()
            mark("backproject_filter", lambda: k4(i0, i1))
            join_halo()
            mark("backproject_filter_boundary", lambda: (k4(0, i0), k4(i1, self.n_local)))
        else:
            mark("backproject_filter", lambda: k4(0, self.n_local))
            if self.device_path and cfg.overlap_align and self.peer is None:
                self._ev_stage1_may_start = torch.cuda.Event()
                self._ev_stage1_may_start.record(torch.cuda.current_stream(self.device))
        return xyz, votes, bbox, support

    def _merge_outputs(self, slot: int):
        if self._merge_out[slot] is None:
            self._merge_out[slot] = ops.new_voxel_outputs(self._cap_merge, self.device)
        return self._merge_out[slot]

    def _sparse_for_dedup(self, sparse_xyz):
        """N5: float32 sparse points of ALL ranks (padded with NaN, which falls into no cell).  The per-rank
        capacity is agreed once (the only host wait, first call)."""
        mine = sparse_xyz.float().contiguous()
        if self.peer is None:
            return mine
        import torch.distributed as dist

        if getattr(self, "_sparse_cap", None) is None or self._sparse_cap < mine.shape[0]:
            cap = torch.tensor([mine.shape[0]], dtype=torch.int64, device=self.device)
            dist.all_reduce(cap, op=dist.ReduceOp.MAX, group=self.group)
            self._sparse_cap = int(cap.item())
        pad = torch.full((self._sparse_cap, 3), float("nan"), dtype=torch.float32, device=self.device)
        pad[: mine.shape[0]] = mine
        allp = torch.empty((self.world * self._sparse_cap, 3), dtype=torch.float32, device=self.device)
        dist.all_gather_into_tensor(allp, pad, group=self.group)
        return allp

    def hash_fuse(self, n_points: int) -> ops.HashFuse:
        """The hashed fusion path's buffers, grown when a step has more points (+ dedup points) than they hold; with peers
        also large enough for the owner's share of the merge."""
        need = max(int(n_points), self._cap_merge if self.peer is not None else 0)
        if getattr(self, "_hash", None) is None or self._hash.cap_voxels < need:
            self._hash = None  # free the old buffers first
            self._hash = ops.HashFuse(self.device, need)
        return self._hash

    def _fuse_device(self, xyz, rgb, votes, mark=None, drop=None, out_slot: int = 0):
        """Stage 4 on the device path.  One rank: rank + accumulate + finalise.  R ranks: partial records into
        peer-visible memory, one barrier, then the owner-side merge that reads the peers' units and records over
        NVLink.  Both the dense and the hashed form of each half are enqueued on the same outputs; the device grid
        decides which one runs (the hashed path takes a grid too large for the session's bitmap), so nothing is read
        back.  Returns persistent output buffers (valid until the next step) and a snapshot of the counts."""
        if mark is None:
            mark = lambda name, fn: fn()
        sess = self.session
        flat = (xyz.view(-1, 3), rgb.view(-1, 3), votes.view(-1))
        if drop is not None and drop.shape[0] == 0:
            drop = None
        hf = self.hash_fuse(flat[0].shape[0] + (0 if drop is None else drop.shape[0]))
        if self.peer is None:
            if drop is not None:
                sess.unmark_points(drop)
            out = self.ops.fuse_finish(sess, *flat, self.fthr, row_len=xyz.shape[2])[:4]
            k, x, c, n, counts = self.ops.fuse_finish_hashed(sess, hf, *flat, self.fthr, row_len=xyz.shape[2], dedup_xyz=drop, out=out)
            return k, x, c, n, counts.clone()
        rec, hdl, _ = self.peer.buffer("records", tuple(self.peer_records_shape), torch.int64)
        samples = self.peer.buffer("hash_samples", (ops._lib.HASH_SAMPLES + 1,), torch.int64)[0]

        def partials():
            self.ops.fuse_finish_partial(sess, *flat, self.fthr, rec, row_len=xyz.shape[2])
            # N5 on the hashed path: every rank tombstones the cells of all ranks' sparse points, so their points are
            # never sent
            self.ops.fuse_finish_hashed_partial(sess, hf, *flat, self.fthr, rec, samples, row_len=xyz.shape[2], dedup_xyz=drop)

        def merge():
            out = self.ops.fuse_merge_peers(sess, self.rank, self.world, self._peer_records, self._peer_prefix, self._plan, self._cap_merge,
                                            out=self._merge_outputs(out_slot), drop_xyz=drop)[:4]
            return self.ops.fuse_merge_hashed_peers(sess, hf, self.rank, self.world, self._peer_records, self._peer_samples, self._plan,
                                                    self._cap_merge, out=out)

        mark("fuse_partials", partials)
        hdl.barrier()  # every rank's units, tile prefix, records and samples are complete
        k, x, c, n, counts = mark("fuse_merge", merge)
        return k, x, c, n, counts.clone()

    def _nbr_full(self) -> torch.Tensor:
        """Neighbour table padded to n_slots rows (build_pair_tables indexes it by global slot)."""
        if self.n_slots == self.n_local:
            return self.nbr_slots
        if getattr(self, "_nbr_padded", None) is None:
            pad = torch.full((self.n_slots - self.n_local, self.K), -1, dtype=torch.int32, device=self.device)
            self._nbr_padded = torch.cat([self.nbr_slots, pad], 0).contiguous()
        return self._nbr_padded

    def _fuse_sharded(self, xyz, rgb, votes, grid, mark=None):
        if mark is None:
            mark = lambda name, fn: fn()
        n_tiles, _ = self.ops.fuse_tile_info(grid)
        tile_prefix = torch.empty(n_tiles + 1, dtype=torch.int32, device=self.device) if n_tiles > 0 else None
        rec, counts = mark("fuse_partials", lambda: self.ops.voxel_fuse_partial(
            xyz.view(-1, 3), rgb.view(-1, 3), votes.view(-1), self.fthr, grid, row_len=xyz.shape[2], tile_prefix=tile_prefix))
        return mark("fuse_exchange_merge", lambda: self._exchange_and_merge(rec, counts, grid, mark, tile_prefix))

    def _plan_by_tiles(self, tile_prefix):
        """Ownership by tile ranges.  Every rank all-gathers the [n_tiles + 1] record prefix of its sorted
        partial records; the R-1 cut tiles that balance the GLOBAL record count follow from the summed
        prefixes, and the same table gives what every rank sends to and receives from every other - no key
        sampling, no search, no separate count exchange.  One small collective, one readback."""
        import torch.distributed as dist

        R, r = self.world, self.rank
        flat = torch.empty(R * tile_prefix.numel(), dtype=torch.int32, device=self.device)
        dist.all_gather_into_tensor(flat, tile_prefix.contiguous(), group=self.group)
        allp = flat.view(R, -1).long()
        cum = allp.sum(0)  # global number of records in tiles [0, t)
        total = cum[-1]
        targets = (total * torch.arange(1, R, device=self.device)) // R
        cuts = torch.searchsorted(cum, targets, right=False).clamp_(0, cum.numel() - 1)
        bnd = torch.cat([cuts.new_zeros(1), cuts, cuts.new_full((1,), cum.numel() - 1)])  # R + 1 tile boundaries
        bnd = torch.cummax(bnd, 0).values
        at = allp[:, bnd]  # [R, R + 1] record index of every rank at every boundary
        send = at[r, 1:] - at[r, :-1]
        recv = at[:, r + 1] - at[:, r]
        host = torch.cat([send, recv, bnd[r:r + 2], at[r, -1:]]).cpu().tolist()  # the one readback
        return host[:R], host[R:2 * R], (host[2 * R], host[2 * R + 1]), host[2 * R + 2]

    def _plan_by_samples(self, rec, mv):
        """Grids too large for tiles: R-1 sampled splitter keys."""
        import torch.distributed as dist

        R = self.world
        pk = rec[:mv, 0]
        if mv > 0:
            q = torch.linspace(0, mv - 1, R + 1, device=self.device)[1:-1].round().long()
            samples = pk[q]
        else:
            samples = torch.full((R - 1,), torch.iinfo(torch.int64).max, dtype=torch.int64, device=self.device)
        allsamp = torch.empty(R * (R - 1), dtype=torch.int64, device=self.device)
        dist.all_gather_into_tensor(allsamp, samples.contiguous(), group=self.group)
        allsamp, _ = torch.sort(allsamp)
        splitters = allsamp[torch.arange(1, R, device=self.device) * (R - 1) - 1]
        cuts = torch.searchsorted(pk.contiguous(), splitters)  # local sorted keys: slice r = [cuts[r-1], cuts[r])
        bnd = torch.cat([torch.zeros(1, dtype=torch.int64, device=self.device), cuts, torch.tensor([mv], device=self.device)])
        send_counts = (bnd[1:] - bnd[:-1]).contiguous()
        recv_counts = torch.empty_like(send_counts)
        dist.all_to_all_single(recv_counts, send_counts, group=self.group)
        sc, rc = torch.stack([send_counts, recv_counts]).cpu().tolist()
        return sc, rc, (0, 0), mv

    def _exchange_and_merge(self, rec, counts, grid, mark, tile_prefix=None):
        import torch.distributed as dist

        if tile_prefix is not None:
            sc, rc, tile_range, mv = self._plan_by_tiles(tile_prefix)
        else:
            mv = int(counts[1].item())
            sc, rc, tile_range, mv = self._plan_by_samples(rec, mv)
        rec = rec[:mv]
        n_recv = int(sum(rc))
        W = rec.shape[1]

        def exchange():
            # the sorted records of one destination are one contiguous slice: no pack kernel
            out = torch.empty((n_recv, W), dtype=rec.dtype, device=self.device)
            dist.all_to_all_single(out.view(-1), rec.reshape(-1), output_split_sizes=[c * W for c in rc],
                                   input_split_sizes=[c * W for c in sc], group=self.group)
            return out

        got = mark("fuse_alltoall", exchange)
        k, x, c, n, mcounts = mark("fuse_merge", lambda: self.ops.voxel_merge_partials(got, grid, tile_range=tile_range))
        # (points fused locally, voxels owned); the owner's colour-sum overflow flag (-1) is kept
        counts2 = torch.stack([torch.where(mcounts[0] < 0, mcounts[0], counts[0]), mcounts[1]])
        return k, x, c, n, counts2

    # -- end-to-end with host buffers -----------------------------------------------------------------
    def pin_host_inputs(self, depth, normal, mask, rgb, sparse_xyz, sparse_offsets, pack_mask: bool = False):
        """Pinned copies of the host inputs.  ``pack_mask``: the mask goes up as one bit per pixel (ops.pack_mask)."""
        if pack_mask:
            mask = ops.pack_mask(mask)
        return tuple(t.contiguous().pin_memory() for t in (depth, normal, mask, rgb, sparse_xyz, sparse_offsets))

    def _host_state(self, sparse_xyz, sparse_offsets):
        """Copy streams and TWO sets of device staging / pinned result buffers (a call uses the set its predecessor
        did not), created once: the uploads of one call overlap the kernels and the downloads of the previous one."""
        if self._host_out is None:
            n, H, W, dev = self.n_local, self.H, self.W, self.device

            def slot():
                return {"depth": torch.empty((n, H, W), dtype=torch.float32, device=dev),
                        "mask": None,  # bool [n,H,W] or bit-packed uint8 [n, ceil(HW/8)], allocated on first use
                        "rgb": torch.empty((n, H, W, 3), dtype=torch.uint8, device=dev),
                        "normal": None,
                        "sparse_xyz": torch.empty(tuple(sparse_xyz.shape), dtype=torch.float64, device=dev),
                        "sparse_offsets": torch.empty(tuple(sparse_offsets.shape), dtype=torch.int64, device=dev),
                        "small": torch.zeros(32, dtype=torch.int64).pin_memory(),  # counts [2] + grid state [8 x i64]
                        "free": None,  # event: the kernels that read this set's staging buffers have finished
                        "out": None}

            self._host_out = {"copy": torch.cuda.Stream(device=dev), "d2h": torch.cuda.Stream(device=dev), "slots": [slot(), slot()],
                              "next": 0}
        return self._host_out

    def _pinned_out(self, st, mv):
        out = st["out"]
        if out is None or out["keys"].shape[0] < mv:
            cap = int(mv * 1.25) + 1024
            out = {"keys": torch.empty(cap, dtype=torch.int64).pin_memory(),
                   "xyz": torch.empty((cap, 3), dtype=torch.float32).pin_memory(),
                   "rgb": torch.empty((cap, 3), dtype=torch.uint8).pin_memory(),
                   "count": torch.empty(cap, dtype=torch.int32).pin_memory()}
            st["out"] = out
        return out

    def run_host(self, depth, normal, mask, rgb, sparse_xyz, sparse_offsets, normals_in_place: bool = True,
                 chunk_views: int = 16):
        """Public end-to-end call: host arrays of the rank's own views in, fused cloud back on the host
        (= ``collect_host(submit_host(...))``; a stream of scenes should call the two halves itself, submitting
        scene i+1 before collecting scene i, so that uploads, kernels and downloads of neighbouring scenes overlap).

        Inputs should be pinned (``pin_host_inputs``).  The copy engine and the kernels overlap: depth and
        mask travel in chunks of ``chunk_views`` views and each chunk is aligned as soon as it has landed;
        colours follow while the consistency kernel runs.  With ``normals_in_place`` the normal maps stay
        in pinned host memory and the consistency kernel reads, over PCIe, only the normals of its vote
        candidates (a few percent of the pixels) instead of moving 12 B/pixel to the device.  The fused
        cloud returns through pinned buffers (views into them: valid until the call after the next)."""
        return self.collect_host(self.submit_host(depth, normal, mask, rgb, sparse_xyz, sparse_offsets, normals_in_place, chunk_views))

    def submit_host(self, depth, normal, mask, rgb, sparse_xyz, sparse_offsets, normals_in_place: bool = True,
                    chunk_views: int = 16) -> dict:
        """First half of ``run_host``: enqueues the uploads and every kernel of the step and returns a ticket without
        waiting for anything."""
        cfg = self.cfg
        if self.device.type != "cuda":
            raise ops.DDNError("run_host needs a CUDA device")
        hs = self._host_state(sparse_xyz, sparse_offsets)
        st = hs["slots"][hs["next"]]
        hs["next"] ^= 1
        comp = torch.cuda.current_stream(self.device)
        copy = hs["copy"]
        if st["free"] is not None:
            copy.wait_event(st["free"])  # the call before the previous one is done with this set's staging buffers
        n = self.n_local
        if self._max_sparse is None:
            self._max_sparse = max_sparse_count(sparse_offsets)
        h2d = 0

        def upload(dst, src):
            nonlocal h2d
            dst.copy_(src, non_blocking=True)
            h2d += src.numel() * src.element_size()

        with torch.cuda.stream(copy):
            upload(st["sparse_xyz"], sparse_xyz)
            upload(st["sparse_offsets"], sparse_offsets)
        refined_slots = self._new_refined_slots()
        poses_local = self.poses_slots[:n]
        fuse = cfg.voxel is not None
        pair, src = self._pair_tables()
        box = self._new_box() if (self.device_path and fuse) else None
        stats = []
        for c0 in range(0, n, max(int(chunk_views), 1)):
            c1 = min(c0 + max(int(chunk_views), 1), n)
            if st["mask"] is None or st["mask"].shape != mask.shape or st["mask"].dtype != mask.dtype:
                st["mask"] = torch.empty(tuple(mask.shape), dtype=mask.dtype, device=self.device)
            with torch.cuda.stream(copy):
                upload(st["depth"][c0:c1], depth[c0:c1])
                upload(st["mask"][c0:c1], mask[c0:c1])
                ev = torch.cuda.Event()
                ev.record(copy)
            comp.wait_event(ev)
            _, s_c = self.ops.align_views(st["depth"][c0:c1], st["mask"][c0:c1], poses_local[c0:c1].contiguous(),
                                          self.kmat[c0:c1].contiguous(), st["sparse_xyz"], st["sparse_offsets"][c0:c1 + 1].contiguous(),
                                          self._max_sparse, cfg.align, out=refined_slots[c0:c1], **self._box_args(src, box, c0, c1))
            stats.append(s_c)
        with torch.cuda.stream(copy):
            if normals_in_place and normal.is_pinned():
                normal_arg = normal
            else:
                if st["normal"] is None:
                    st["normal"] = torch.empty((n, self.H, self.W, 3), dtype=torch.float32, device=self.device)
                upload(st["normal"], normal)
                normal_arg = st["normal"]
            ev_n = torch.cuda.Event()
            ev_n.record(copy)
            upload(st["rgb"], rgb)
            ev_rgb = torch.cuda.Event()
            ev_rgb.record(copy)
        xyz, votes, bbox, _ = self._halo_and_filter(refined_slots, normal_arg, lambda name, fn: fn(), pair, src,
                                                    wait_normal=lambda: comp.wait_event(ev_n), box=box)
        ticket = {"slot": st, "h2d_bytes": h2d, "stats": torch.cat(stats) if stats else None, "fused": None, "host_grid": None}
        s = cfg.filter.stride
        if fuse and self.device_path:
            comp.wait_event(ev_rgb)
            rgb_s = st["rgb"] if s == 1 else st["rgb"][:, ::s, ::s].contiguous()
            drop = self._sparse_for_dedup(st["sparse_xyz"]) if cfg.dedup_sparse else None
            # (with peers the merge writes into persistent buffers: each staging set has its own)
            k, x, c, m, counts = self._fuse_device(xyz, rgb_s, votes, drop=drop, out_slot=hs["next"] ^ 1)
            st["small"][:2].copy_(counts, non_blocking=True)
            st["small"][2:10].copy_(self.session.grid.view(torch.int64), non_blocking=True)
            st["small"][10:12].copy_(self._hash.state[:2], non_blocking=True)
            ticket["fused"] = (k, x, c, m)
        elif fuse:
            # collective fallback (host-side grid and plan: it waits for the device on its way)
            bb = self._global_bbox(bbox)
            if np.all(np.isfinite(bb)):
                grid = self.ops.make_grid(bb[:3], bb[3:], cfg.voxel)
                comp.wait_event(ev_rgb)
                rgb_s = st["rgb"] if s == 1 else st["rgb"][:, ::s, ::s].contiguous()
                if self.world == 1:
                    k, x, c, m, counts = self.ops.voxel_fuse(xyz.view(-1, 3), rgb_s.view(-1, 3), votes.view(-1), self.fthr, grid,
                                                             trim=False, row_len=xyz.shape[2])
                else:
                    k, x, c, m, counts = self._fuse_sharded(xyz, rgb_s, votes, grid)
                st["small"][:2].copy_(counts, non_blocking=True)
                ticket["fused"], ticket["host_grid"] = (k, x, c, m), grid
        done = torch.cuda.Event()
        done.record(comp)
        st["free"] = done
        ticket["done"] = done
        return ticket

    def collect_host(self, ticket: dict) -> dict:
        """Second half of ``run_host``: waits for the step's kernels, reads the voxel count, downloads exactly that many
        voxels on the download stream and returns the host views."""
        hs, st = self._host_out, ticket["slot"]
        out = {"h2d_bytes": ticket["h2d_bytes"], "d2h_bytes": 0, "num_points": 0, "stats": ticket["stats"]}
        ticket["done"].synchronize()  # the one wait: the host needs the voxel count to size the download
        if ticket["fused"] is None:
            return out
        k, x, c, m = ticket["fused"]
        small = st["small"]
        n_pts, mv = int(small[0]), int(small[1])
        out["d2h_bytes"] += 16
        grid = ticket["host_grid"]
        if grid is None:
            gs = ops._lib.GridState.from_buffer_copy(small[2:10].numpy().tobytes())
            out["d2h_bytes"] += 64
            if gs.status == ops._lib.GRID_EMPTY:
                return out
            ops.check_hash_state(small[10:12].tolist())
            if gs.status not in (ops._lib.GRID_OK, ops._lib.GRID_HASHED):
                raise ops.DDNError(f"fusion grid: {ops.GRID_STATUS.get(gs.status, gs.status)} (dims {list(gs.dims)}); raise "
                                   "max_grid_cells or use a larger voxel")
            grid = ops._lib.VoxelGrid()
            grid.voxel = gs.voxel
            for i in range(3):
                grid.origin[i], grid.bits[i], grid.dims[i] = gs.origin[i], gs.bits[i], gs.dims[i]
        if n_pts < 0:
            raise ops.DDNError("voxel fusion: a voxel collected 2^24 or more points (32-bit colour sums); use a smaller voxel")
        if mv > k.shape[0]:
            raise ops.DDNError(f"voxel fusion: {mv} voxels exceed the output capacity {k.shape[0]}")
        po = self._pinned_out(st, mv)
        d2h = hs["d2h"]
        with torch.cuda.stream(d2h):
            for name, t in (("keys", k), ("xyz", x), ("rgb", c), ("count", m)):
                po[name][:mv].copy_(t[:mv], non_blocking=True)
                t.record_stream(d2h)
                out[name] = po[name][:mv]
                out["d2h_bytes"] += out[name].numel() * out[name].element_size()
        d2h.synchronize()
        out["num_points"] = n_pts
        out["grid"] = grid
        return out
