"""Per-scene runner: reference views sharded round-robin over ranks (one process per GPU), no
collective during depth inference, ONE all-gather of the final depth maps before fusion
(SURVEY.md section 8(e); upstream hands depth maps over through PFM files, test_tank.py:304-373).
"""
from __future__ import annotations

from typing import Callable, Dict, List, Sequence, Tuple

import torch
import torch.distributed as dist


def block_start(n_views: int, rank: int, world: int) -> int:
    """First view of rank's block under balanced block sharding (rank == world gives n_views)."""
    q, r = divmod(n_views, world)
    return rank * q + min(rank, r)


def shard_views(n_views: int, rank: int, world: int, mode: str = "round_robin") -> List[int]:
    """Reference views owned by `rank`.  "round_robin": rank, rank+world, ... ; "block": a contiguous run --
    neighbouring reference views share their source images, so a rank that caches encoded features (section 8(f)
    row 1) encodes each image at most once.  Both are balanced: every rank owns floor(n/world) views and the first
    n % world ranks one more, so a rank is empty only when n_views < world (49 views on 8 ranks: 7,6,6,6,6,6,6,6)."""
    if mode == "block":
        return list(range(block_start(n_views, rank, world), block_start(n_views, rank + 1, world)))
    return list(range(rank, n_views, world))


def slots_per_rank(n_views: int, world: int) -> int:
    return (n_views + world - 1) // world


def view_slot(i: int, n_views: int, world: int, mode: str = "round_robin"):
    """(owner rank, slot inside the owner's all-gather block) of reference view i."""
    if mode != "block":
        return i % world, i // world
    q, r = divmod(n_views, world)
    owner = i // (q + 1) if i < r * (q + 1) else r + (i - r * (q + 1)) // max(q, 1)
    return owner, i - block_start(n_views, owner, world)


def view_groups(views: Sequence, k: int) -> List[Tuple[list, int]]:
    """`views` in order as consecutive groups of k, each with the number of its real entries: a short last group is padded
    to k entries with copies of its last entry (whose results the caller drops).  No views give no groups."""
    if k < 1:
        raise ValueError("groups of at least one view, got k = {}".format(k))
    views = list(views)
    out = []
    for a in range(0, len(views), k):
        g = views[a:a + k]
        out.append((g + [g[-1]] * (k - len(g)), len(g)))
    return out


def gather_depths(local: Dict[int, torch.Tensor], n_views: int, rank: int, world: int, h: int, w: int, device,
                  mode: str = "round_robin") -> torch.Tensor:
    """All-gather of the per-rank depth maps into one (n_views,h,w) tensor on every rank.

    Each rank contributes a (slots,h,w) block, zero padded where it owns fewer than `slots` views (a rank that owns
    none still contributes its zero block: every rank must enter the collective); view i lives at
    view_slot(i) = (owner, slot) of the rank-major concatenation."""
    slots = slots_per_rank(n_views, world)
    mine = torch.zeros(slots, h, w, device=device, dtype=torch.float32)
    for i, d in local.items():
        owner, slot = view_slot(i, n_views, world, mode)
        if owner != rank:
            raise ValueError("view {} belongs to rank {}, not {} ({} sharding)".format(i, owner, rank, mode))
        mine[slot] = d
    if world == 1 or not (dist.is_available() and dist.is_initialized()):
        flat = mine
    else:
        flat = torch.empty(world * slots, h, w, device=device, dtype=torch.float32)   # rank-major concatenation
        dist.all_gather_into_tensor(flat, mine)
    index = [o * slots + s for o, s in (view_slot(i, n_views, world, mode) for i in range(n_views))]
    if index == list(range(n_views)):
        return flat[:n_views]
    return flat.index_select(0, torch.as_tensor(index, device=flat.device))


def agree_on_size(local_hw, n_views: int, world: int, device):
    """(h, w) of the depth maps on every rank.  Only when n_views < world can a rank own no view and not know the
    size; then (and only then -- the condition is the same on all ranks) one 2-element MAX all-reduce tells it."""
    if n_views >= world or world == 1 or not (dist.is_available() and dist.is_initialized()):
        if local_hw is None:
            raise ValueError("no depth map on this rank and no peer to learn its size from")
        return local_hw
    t = torch.tensor(list(local_hw or (0, 0)), device=device, dtype=torch.int64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return int(t[0]), int(t[1])


@torch.no_grad()
def run_scene(infer: Callable, fuse: Callable, n_views: int, pairs: Sequence[Sequence[int]], rank: int = 0, world: int = 1,
              device="cuda", fuse_pairs: Sequence[Sequence[int]] = None, timings: dict = None, sharding: str = "round_robin",
              views_per_batch: int = None):
    """infer(ref_view, src_views) -> (depth (h,w), conf (hc,wc)) on `device`;
    fuse(ref_view, ref_depth (1,1,h,w), conf (1,hc,wc), src_views, src_depths (1,v,1,h,w)) -> dict with
    'final' (1,1,h,w) bool and 'points' (1,3,h,w).
    pairs[i]: source views used for the depth map of view i; fuse_pairs[i] (default: pairs[i]): source
    views whose depth maps the consistency filter of view i reads (upstream: 4 and up to 10).
    When infer has `batch` (infer.batch([(ref_view, src_views), ...]) -> [(depth, conf), ...]), the rank's views go to
    it in view order, in groups of at most views_per_batch (default: infer.views_per_batch, else 1).
    Returns {ref_view: (points (k,3), depth (h,w))} for the views this rank owns."""
    fuse_pairs = pairs if fuse_pairs is None else fuse_pairs
    mine = shard_views(n_views, rank, world, sharding)
    batch = getattr(infer, "batch", None)
    k = views_per_batch if views_per_batch is not None else getattr(infer, "views_per_batch", 1)
    if batch is None and k != 1:
        raise ValueError("views_per_batch = {} needs an infer with a `batch` method".format(k))
    depths, confs = {}, {}
    timed = timings is not None and torch.cuda.is_available() and str(device).startswith("cuda")
    if timed:
        ev_start = torch.cuda.Event(enable_timing=True)
        ev_start.record()
    if batch is None:
        for i in mine:
            depths[i], confs[i] = infer(i, list(pairs[i]))
    else:
        for group, n in view_groups(mine, k):
            real = group[:n]
            for i, (d, c) in zip(real, batch([(i, list(pairs[i])) for i in real])):
                depths[i], confs[i] = d, c
    # a rank without a view (n_views < world) still enters the collective below with a zero block
    h, w = agree_on_size(tuple(next(iter(depths.values())).shape[-2:]) if depths else None, n_views, world, device)
    ev = None
    if timed:
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
    all_depths = gather_depths(depths, n_views, rank, world, h, w, device, sharding)
    if ev:
        ev[1].record()
    out = {}
    flat = [j for i in mine for j in fuse_pairs[i]]
    flat_dev = torch.as_tensor(flat, device=all_depths.device, dtype=torch.long) if flat else None      # ONE host -> device copy
    at = 0
    for i in mine:
        src = list(fuse_pairs[i])
        sel = flat_dev[at:at + len(src)]
        at += len(src)
        res = fuse(i, depths[i].reshape(1, 1, h, w), confs[i].unsqueeze(0), src, all_depths.index_select(0, sel).reshape(1, len(src), 1, h, w))
        m = res["final"][0, 0]
        out[i] = (res["points"][0][:, m].t().contiguous(), depths[i])
    if ev:
        ev[2].record()
        torch.cuda.synchronize()
        timings["depth_maps_ms"] = ev_start.elapsed_time(ev[0])
        timings["all_gather_ms"] = ev[0].elapsed_time(ev[1])
        timings["fusion_ms"] = ev[1].elapsed_time(ev[2])
    return out


def _as_words(*ts):
    """contiguous (N, ...) tensors as (N, row) matrices of 16-byte complex128 words when every row allows it, else of their
    own elements: index_select / index_copy_ along dim 0 then move 16 bytes per element instead of 4 (with 4-byte elements
    the 49-view DTU scene at one view per replay was 1.4 % slower than plain per-view copies).  The bits are copied, never
    computed on."""
    flat = [t.view(t.shape[0], -1) for t in ts]
    if all((f.shape[1] * f.element_size()) % 16 == 0 and f.data_ptr() % 16 == 0 for f in flat):
        return [f.view(torch.complex128) for f in flat]
    return flat


class GraphedViewRunner:
    """Depth inference of reference views from a per-scene feature cache as two CUDA graphs: `encode` (one image through
    the FPN into its rows of the cache) and `forward` (the cascade for `views_per_replay` = K reference views at once).
    The hot path has no host synchronisation, so both capture; per K views the host issues one device-to-device index
    copy and one replay instead of ~320 launches per view (section 8(f) row 1 + SURVEY section 8(e) "CUDA-graph the
    forward").  Batching fills the launches of the 1/8-resolution stage, which one view leaves mostly idle.

    The cache is one preallocated tensor per stage, (N_images, h, w, C) in memory: row j read through
    ``permute(0, 3, 1, 2)`` is image j's channels-last (C, h, w) map, and every row is 32-byte aligned (C >= 8 floats),
    which the TMA tile kernels of effimvs_warp_corr_agg_f32 need.  At DTU's 1600x1184 that is 26.5 MB per image: about
    1.3 GB for a 49-image scene, plus 26.5 * K * (n_src + 1) MB for the gathered features of one replay.

    The forward graph starts with the gathers, all driven by one static (K, 1 + n_src) index buffer (reference view,
    then sources, per batch row): features from the cache, reference images from `imgs`, cameras from `cams`."""

    def __init__(self, model, imgs: torch.Tensor, cams: Dict[str, torch.Tensor], depth_values: torch.Tensor, n_src: int,
                 views_per_replay: int = 1):
        if views_per_replay < 1:
            raise ValueError("views_per_replay must be at least 1, got {}".format(views_per_replay))
        imgs = imgs.contiguous()
        self.model, self.imgs, self.cams = model, imgs, cams
        self.stages = [k for k in ("stage1", "stage2", "stage3") if k in cams]
        K, V = views_per_replay, n_src + 1
        self.views_per_replay, self.n_src = K, n_src
        dev = imgs.device
        self.encoded_images = set()                  # images whose cache rows hold their features
        self._sel: Dict[tuple, torch.Tensor] = {}
        self.stream = torch.cuda.Stream(dev)
        self.slot = torch.zeros(1, device=dev, dtype=torch.long)        # the image `encode` reads = the cache row it writes
        self.idx = torch.zeros(K, V, device=dev, dtype=torch.long)      # the views `forward` reads
        self.img_in = imgs[:1].clone()
        self.ref_in = torch.empty(K, *imgs.shape[1:], device=dev, dtype=imgs.dtype)
        self.cam_in = {k: torch.empty(K, V, *cams[k].shape[1:], device=dev, dtype=cams[k].dtype) for k in self.stages}
        self.dv = depth_values.reshape(1, -1).repeat(K, 1)
        with torch.no_grad():
            torch.cuda.synchronize(dev)
            with torch.cuda.stream(self.stream):
                enc = [st[0] for st in model.encode(self.img_in.unsqueeze(1))]
                self.cache = [torch.empty(imgs.shape[0], *e.shape[2:], e.shape[1], device=dev, dtype=e.dtype) for e in enc]
                self.gathered = [torch.empty(V * K, *c.shape[1:], device=dev, dtype=c.dtype) for c in self.cache]
                # warm-up (cuDNN autotune, lazy init, workspace sizes) on image 0's features in every view of every row
                for _ in range(2):
                    self._encode()
                for _ in range(2):
                    self._forward()
            self.stream.synchronize()
            self.g_enc = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.g_enc, stream=self.stream):
                self._encode()
            self.g_fwd = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.g_fwd, stream=self.stream):
                out = self._forward()
            self.out = (out["depth"][-1], out["photometric_confidence"])

    def _encode(self):
        """image `slot` through the FPN into row `slot` of the cache"""
        src, dst = _as_words(self.imgs, self.img_in)
        torch.index_select(src, 0, self.slot, out=dst)
        for c, e in zip(self.cache, self.model.encode(self.img_in.unsqueeze(1))):
            dst, src = _as_words(c, e[0].permute(0, 2, 3, 1).contiguous())
            dst.index_copy_(0, self.slot, src)

    def _forward(self):
        """the cascade on the K rows of `idx`.  Features are gathered view-major: view v of all K rows is the
        contiguous channels-last (K, C, h, w) slice v * K .. v * K + K - 1 of the gathered tensor."""
        K, V = self.idx.shape
        flat = self.idx.t().reshape(-1)
        self.feat_in = []
        for c, g in zip(self.cache, self.gathered):
            src, dst = _as_words(c, g)
            torch.index_select(src, 0, flat, out=dst)
            self.feat_in.append([g[v * K:(v + 1) * K].permute(0, 3, 1, 2) for v in range(V)])
        src, dst = _as_words(self.imgs, self.ref_in)
        torch.index_select(src, 0, self.idx[:, 0].contiguous(), out=dst)
        rows = self.idx.reshape(-1)
        for k in self.stages:
            torch.index_select(self.cams[k], 0, rows, out=self.cam_in[k].view(K * V, *self.cams[k].shape[1:]))
        return self.model.forward_from_features(self.feat_in, self.ref_in, self.cam_in, self.dv)

    def _index(self, idx):
        """device tensor of an index list, built once per distinct list: a host list -> device copy is a stream
        synchronisation, and one per replay would serialise the host's enqueue work with the previous replay"""
        key = tuple(map(tuple, idx)) if idx and isinstance(idx[0], (list, tuple)) else tuple(idx)
        if key not in self._sel:
            self._sel[key] = torch.as_tensor(idx, device=self.imgs.device, dtype=torch.long)
        return self._sel[key]

    def clear_cache(self):
        """forget which images are encoded: the next replays encode them again"""
        self.encoded_images.clear()

    @torch.no_grad()
    def infer_batch(self, items: Sequence):
        """items: up to K (reference view, source views) pairs -> [(depth (H,W), conf (hc,wc))] in the same order.
        A short batch is padded with its last view; the padded rows' outputs are dropped."""
        if not 0 < len(items) <= self.views_per_replay:
            raise ValueError("GraphedViewRunner takes 1 to {} views per replay, got {}".format(self.views_per_replay, len(items)))
        for _, srcs in items:
            if len(srcs) != self.n_src:
                raise ValueError("GraphedViewRunner was captured for {} source views, got {}".format(self.n_src, len(srcs)))
        (rows, n), = view_groups([[i] + list(srcs) for i, srcs in items], self.views_per_replay)
        with torch.cuda.stream(self.stream):
            for j in (j for row in rows[:n] for j in row):
                if j not in self.encoded_images:
                    self.slot.copy_(self._index([j]))
                    self.g_enc.replay()
                    self.encoded_images.add(j)
            self.idx.copy_(self._index(rows))
            self.g_fwd.replay()
            depth, conf = self.out[0][:n].clone(), self.out[1][:n].clone()     # before the next replay overwrites them
        torch.cuda.current_stream().wait_stream(self.stream)
        return [(depth[b], conf[b]) for b in range(n)]


def cuda_scene_callables(model, imgs: torch.Tensor, cams: Dict[str, torch.Tensor], depth_values: torch.Tensor,
                         dist_base: float, rel_diff_base: float, thres_view: int, prob_threshold: float,
                         feature_cache: bool = False, graphed_src_views: int = 0, views_per_replay: int = 1):
    """infer / fuse callables for `run_scene` on the CUDA path.
    imgs (Nv,3,H,W) on the device; cams {"stage1".."stage4": (Nv,2,4,4)}; depth_values (Dv).
    feature_cache: encode every image once per rank and reuse its feature pyramid for each reference view
    that lists it as a source (section 8(f) row 1; eval-mode results are those of re-encoding it).
    graphed_src_views > 0: run encode / cascade as CUDA graphs captured for that many source views (implies the
    feature cache); then infer.batch([(ref_view, src_views), ...]) runs up to views_per_replay views per replay of the
    cascade, and run_scene groups the views accordingly.  views_per_replay > 1 needs the graphs."""
    from . import fusion
    if views_per_replay != 1 and graphed_src_views <= 0:
        raise ValueError("views_per_replay = {} needs graphed_src_views > 0 (views are batched inside the CUDA graph)".format(views_per_replay))
    cache: Dict[int, list] = {}
    runner = GraphedViewRunner(model, imgs, cams, depth_values, graphed_src_views, views_per_replay) if graphed_src_views > 0 else None

    def encoded(j):
        if j not in cache:
            cache[j] = [stage[0] for stage in model.encode(imgs[j].reshape(1, 1, *imgs.shape[1:]))]
        return cache[j]

    def infer(i, srcs):
        if runner is not None:
            return runner.infer_batch([(i, srcs)])[0]
        idx = [i] + list(srcs)
        stage_cams = {k: v[idx].unsqueeze(0) for k, v in cams.items() if k != "stage4"}
        if feature_cache:
            per_view = [encoded(j) for j in idx]
            feats = [[pv[s] for pv in per_view] for s in range(3)]
            out = model.forward_from_features(feats, imgs[i].unsqueeze(0), stage_cams, depth_values.unsqueeze(0))
        else:
            out = model(imgs[idx].unsqueeze(0), stage_cams, depth_values.unsqueeze(0))
        return out["depth"][-1][0], out["photometric_confidence"][0]

    if runner is not None:
        infer.batch = runner.infer_batch
        infer.views_per_batch = views_per_replay

    def clear_cache():
        """forget the encoded feature pyramids (a new scene, or a benchmark pass that must encode again)"""
        cache.clear()
        if runner is not None:
            runner.clear_cache()
    infer.clear_cache = clear_cache

    sel_cache: Dict[tuple, torch.Tensor] = {}

    def fuse(i, ref_depth, conf, srcs, src_depths):
        full = cams["stage4"]
        key = tuple(srcs)
        if key not in sel_cache:        # one host -> device copy (a synchronisation) per distinct source list, not per call
            sel_cache[key] = torch.as_tensor(list(srcs), device=full.device)
        return fusion.filter_view(ref_depth, conf, src_depths, full[i].unsqueeze(0), full.index_select(0, sel_cache[key]).unsqueeze(0),
                                  dist_base, rel_diff_base, thres_view, prob_threshold, torch_inverse=False)
    return infer, fuse
