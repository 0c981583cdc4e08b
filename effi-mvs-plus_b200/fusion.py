"""Geometric-consistency fusion on the CUDA path, with upstream's function names where a call
site exists (misc/fusion.py:117-181; driver arithmetic of test_tank.py:470-515)."""
from __future__ import annotations

import torch

from . import ops


def inverse_cameras(ref_cam: torch.Tensor, srcs_cam: torch.Tensor) -> torch.Tensor:
    """(n,2,4,4), (n,v,2,4,4) -> (n,1+v,2,4,4) holding inverse(E) and inverse(K) (padded to 4x4),
    taken with torch's LU like upstream's ``.inverse()`` calls (fusion.py:24,32) but without the
    host synchronisation of the error check."""
    cams = torch.cat([ref_cam.unsqueeze(1), srcs_cam], dim=1)
    out = torch.zeros_like(cams)
    out[:, :, 0] = torch.linalg.inv_ex(cams[:, :, 0])[0]
    out[:, :, 1, :3, :3] = torch.linalg.inv_ex(cams[:, :, 1, :3, :3])[0]
    return out.contiguous()


def get_reproj_dynamic(ref_depth, srcs_depth, ref_cam, srcs_cam, torch_inverse: bool = True):
    """Drop-in for misc/fusion.py:117 ``get_reproj_dynamic``.  Returns (reproj_xyd (n,v,3,h,w), None, None):
    the two camera-space tensors upstream also returns are never read by its own caller's
    arithmetic (vis_filter_dynamic only reshapes them, fusion.py:161-162) and are not materialised."""
    inv = inverse_cameras(ref_cam, srcs_cam) if torch_inverse else ops.fusion_invert_cameras(ref_cam, srcs_cam)
    return ops.fusion_reproject(ref_depth, srcs_depth, ref_cam, srcs_cam, inv), None, None


def vis_filter_dynamic(ref_depth, reproj_xyd, ref_idx_world=None, src2ref_idx_cam=None, dist_base=4, rel_diff_base=1300,
                       thres_view=2, relative=False):
    """Drop-in for misc/fusion.py:157 ``vis_filter_dynamic``: (masks (n,v,K,h,w) bool, mask (n,v,1,h,w) bool).
    The two camera-space arguments are accepted and ignored, as upstream's own arithmetic ignores them."""
    masks = ops.fusion_masks(ref_depth, reproj_xyd, float(dist_base), float(rel_diff_base), int(thres_view), bool(relative)).bool()
    return masks, masks[:, :, -1:]


def filter_view(ref_depth, ref_conf, srcs_depth, ref_cam, srcs_cam, dist_base, rel_diff_base, thres_view,
                prob_threshold, relative: bool = False, want_masks: bool = False, torch_inverse: bool = True):
    """One reference view of ``dynamic_filter_depth`` (test_tank.py:470-515) in a single kernel.

    ref_depth (n,1,h,w), ref_conf (n,hc,wc), srcs_depth (n,v,1,h,w), cams as upstream.
    -> dict(final (n,1,h,w) bool, depth_avg (n,1,h,w), points (n,3,h,w)[, masks (n,v,K,h,w) bool])."""
    inv = inverse_cameras(ref_cam, srcs_cam) if torch_inverse else ops.fusion_invert_cameras(ref_cam, srcs_cam)
    final, avg, pts, masks = ops.fusion_filter(ref_depth, srcs_depth, ref_conf, ref_cam, srcs_cam, inv, float(dist_base),
                                               float(rel_diff_base), int(thres_view), float(prob_threshold), bool(relative),
                                               bool(want_masks))
    out = {"final": final.bool(), "depth_avg": avg, "points": pts}
    if want_masks:
        out["masks"] = masks.bool()
    return out


# ---- the same filter for a whole scene: all of a rank's reference views in one launch -----------------------------
MAX_SOURCES = 16              # EFFIMVS_MAX_SRC_VIEWS: the camera records a block keeps in shared memory


class DynamicSceneCameras:
    """The dynamic filter's cameras of every view of a scene (see dynamic_scene_cameras).

    cams (N,2,4,4) float32 on the device; inv (N,2,4,4): inverse(E) and inverse(K) (padded to 4x4) of every camera, as
    effimvs_fusion_invert_cameras_f32 forms them; pairs[i]: the source views of view i (host lists)."""

    def __init__(self, cams: torch.Tensor, inv: torch.Tensor, pairs):
        self.cams, self.inv = cams, inv
        self.pairs = [[int(j) for j in p] for p in pairs]
        self.n_views = len(self.pairs)
        self.vmax = max(len(p) for p in self.pairs)
        self._rows = {}

    def check(self, views, thres_view: int):
        """ValueError naming the first of `views` that is outside the scene or has fewer than thres_view sources"""
        for i in views:
            if not 0 <= i < self.n_views:
                raise ValueError("view {} is outside the scene's {} views".format(i, self.n_views))
            if len(self.pairs[i]) < thres_view:
                raise ValueError("view {} has {} source views, fewer than thres_view = {}".format(i, len(self.pairs[i]), thres_view))

    def rows(self, views, device, stack_rows=None, n_stack=None):
        """the device arrays of effimvs_fusion_filter_views_f32 for reference views `views` (in that order):
        (ref_idx (n,), src_idx (n,vmax), src_count (n,) int32, cams (N,2,4,4), inv (N,2,4,4)).  Indices are scene view
        numbers, or stack_rows[view] where the depth stack (n_stack maps) holds the scene's maps in another order; then
        cams / inv are gathered into the stack's order.  Built and uploaded in one host -> device copy the first time a
        list is asked for, then cached: a host -> device copy synchronises the host with the stream and cannot be
        captured in a CUDA graph, so the first call for a list comes before a capture."""
        views = [int(i) for i in views]
        key = (tuple(views), str(device), None if stack_rows is None else (tuple(sorted(stack_rows.items())), n_stack))
        if key not in self._rows:
            self.check(views, 0)
            row = (lambda j: j) if stack_rows is None else (lambda j: int(stack_rows[j]))   # noqa: E731
            n, vmax = len(views), self.vmax
            host = [row(i) for i in views]
            for i in views:
                host += [row(j) for j in self.pairs[i]] + [0] * (vmax - len(self.pairs[i]))
            host += [len(self.pairs[i]) for i in views]
            if stack_rows is not None:          # the scene view of every stack row this launch reads (others: view 0)
                perm = [0] * n_stack
                for i in views:
                    for j in [i] + self.pairs[i]:
                        perm[row(j)] = j
                host += perm
            dev = torch.as_tensor(host, dtype=torch.int32).to(device)
            a, b, c = n, n + n * vmax, 2 * n + n * vmax
            cams, inv = self.cams, self.inv
            if stack_rows is not None:
                cams, inv = cams.index_select(0, dev[c:]), inv.index_select(0, dev[c:])
            self._rows[key] = (dev[:a], dev[a:b].view(n, vmax), dev[b:c], cams, inv)
        return self._rows[key]


def dynamic_scene_cameras(cams_stage4: torch.Tensor, fuse_pairs) -> DynamicSceneCameras:
    """Cameras of every view of a scene for the batched dynamic filter.  cams_stage4 (N,2,4,4) on the device (E = [:, 0],
    K = [:, 1, :3, :3], the full-resolution cameras filter_view takes); fuse_pairs[i]: the 1 .. 16 source views of view i.
    The inverse table is built in one launch of effimvs_fusion_invert_cameras_f32, the kernel filter_view(...,
    torch_inverse=False) inverts every view's cameras with, so the batched results are bit-identical to it."""
    if cams_stage4.dim() != 4 or tuple(cams_stage4.shape[1:]) != (2, 4, 4):
        raise ValueError("cams_stage4 must be (N,2,4,4), got {}".format(tuple(cams_stage4.shape)))
    N = cams_stage4.shape[0]
    if len(fuse_pairs) != N:
        raise ValueError("{} source lists for {} views".format(len(fuse_pairs), N))
    pairs = [[int(j) for j in p] for p in fuse_pairs]
    for i, p in enumerate(pairs):
        if not 1 <= len(p) <= MAX_SOURCES:
            raise ValueError("view {} has {} source views; the dynamic filter takes 1 to {}".format(i, len(p), MAX_SOURCES))
        if any(not 0 <= j < N for j in p):
            raise ValueError("view {}: source views {} are outside the scene's {} views".format(i, p, N))
    cams = cams_stage4.detach().float().contiguous()
    inv = ops.fusion_invert_cameras(cams, cams.unsqueeze(1))[:, 0].contiguous()     # (N, 2, 2,4,4): column 0 is camera i's
    return DynamicSceneCameras(cams, inv, pairs)


def filter_views(depth_stack, views, confs, table: DynamicSceneCameras, dist_base, rel_diff_base, thres_view, prob_threshold,
                 relative: bool = False, stack_rows=None):
    """``dynamic_filter_depth`` (test_tank.py:470-515) for the reference views `views` in ONE launch.

    depth_stack (N,h,w) CUDA fp32 holds the depth map of every view of the scene (the scene runner's all-gathered maps);
    each view's reference and source maps are read from it in place.  stack_rows: {view: row of depth_stack} when the
    stack is not in scene order (default: view i is row i, and N is the scene's view count).  confs (n,hc,wc) CUDA fp32,
    nearest-resized to (h,w) in the kernel as filter_view does; table from dynamic_scene_cameras.  Makes no host
    synchronisation once the table's rows for `views` are on the device (table.rows), so it can be captured in a CUDA
    graph.  -> dict(final (n,1,h,w) bool, depth_avg (n,1,h,w), points (n,3,h,w)); view views[b]'s results are
    bit-identical to filter_view(..., torch_inverse=False) on that view alone."""
    views = [int(i) for i in views]
    if not views:
        raise ValueError("no reference view to filter")
    if len(views) > 65535:
        raise ValueError("{} reference views in one launch; at most 65535".format(len(views)))
    thres_view = int(thres_view)
    if thres_view < 1:
        raise ValueError("thres_view must be at least 1, got {}".format(thres_view))
    if not (dist_base > 0 and rel_diff_base > 0):
        raise ValueError("dist_base and rel_diff_base must be positive, got {} and {}".format(dist_base, rel_diff_base))
    table.check(views, thres_view)
    if depth_stack.dim() != 3:
        raise ValueError("depth_stack must be (N,h,w), got {}".format(tuple(depth_stack.shape)))
    N, h, w = depth_stack.shape
    if stack_rows is None and N != table.n_views:
        raise ValueError("the depth stack holds {} maps, the camera table {} views".format(N, table.n_views))
    if stack_rows is not None:
        for i in views:
            need = [i] + table.pairs[i]
            if any(j not in stack_rows or not 0 <= stack_rows[j] < N for j in need):
                raise ValueError("view {}: views {} are not all rows of the {}-map depth stack".format(i, need, N))
        need = sorted({j for i in views for j in [i] + table.pairs[i]})
        if len({stack_rows[j] for j in need}) != len(need):
            raise ValueError("views {} do not have a depth-stack row each".format(need))
    n = len(views)
    if confs.dim() != 3 or confs.shape[0] != n:
        raise ValueError("confs must be (n,hc,wc) for n = {} views, got {}".format(n, tuple(confs.shape)))
    ref, src, count, cams, inv = table.rows(views, depth_stack.device, stack_rows, N)
    final, avg, pts = ops.fusion_filter_views(depth_stack, ref, src, count, cams, inv, confs, float(dist_base), float(rel_diff_base),
                                              thres_view, float(prob_threshold), bool(relative))
    return {"final": final.bool(), "depth_avg": avg, "points": pts}


# ---- SURVEY section 8(f) row 2: the DTU pipeline's filter (test_dtu_dypcd.py:164-350) ---------------------------
DTU_FIRST_RUNG, DTU_END_RUNG = 1, 11          # s, e (test_dtu_dypcd.py:33-34)
DTU_DIST_BASE, DTU_DIFF_BASE = 1 / 2, 0.25    # :36-37


def dtu_camera_pack(K_ref, E_ref, Ks_src, Es_src):
    """The float32 matrices of reproject_with_depth / filter_depth, formed on the host with the same NumPy
    calls upstream uses (np.linalg.inv and np.matmul on float32 arrays, test_dtu_dypcd.py:172-176, 192-196,
    330-333): (34 + 50 v,) float32 in the layout effimvs_dtu_filter_f32 documents."""
    import numpy as np
    f32 = lambda a: np.asarray(a.cpu() if torch.is_tensor(a) else a, dtype=np.float32)   # noqa: E731
    K_ref, E_ref = f32(K_ref), f32(E_ref)
    parts = [np.linalg.inv(K_ref).reshape(-1), K_ref.reshape(-1), np.linalg.inv(E_ref).reshape(-1)]
    for K_src, E_src in zip(Ks_src, Es_src):
        K_src, E_src = f32(K_src), f32(E_src)
        parts += [np.matmul(E_src, np.linalg.inv(E_ref)).reshape(-1), K_src.reshape(-1), np.linalg.inv(K_src).reshape(-1),
                  np.matmul(E_ref, np.linalg.inv(E_src)).reshape(-1)]
    return torch.from_numpy(np.concatenate(parts).astype(np.float32))


def dtu_ladder(first_rung: int, end_rung: int, dist_base: float, diff_base: float):
    """the rung thresholds of check_geometric_consistency (test_dtu_dypcd.py:226-228): i * dist_base as float64 and
    log10(max(i, 1.05)) * diff_base rounded to float32, i = first_rung .. end_rung - 1"""
    import math
    import numpy as np
    rungs = range(first_rung, end_rung)
    return [i * dist_base for i in rungs], [float(np.float32(math.log(max(i, 1.05), 10) * diff_base)) for i in rungs]


def dtu_filter_view(ref_depth, confidence, srcs_depth, K_ref, E_ref, Ks_src, Es_src, conf_thres: float = 0.5,
                    want_masks: bool = False, first_rung: int = DTU_FIRST_RUNG, end_rung: int = DTU_END_RUNG,
                    dist_base: float = DTU_DIST_BASE, diff_base: float = DTU_DIFF_BASE):
    """One reference view of upstream's DTU ``filter_depth`` (test_dtu_dypcd.py:236-337) in a single kernel.

    ref_depth (h,w), srcs_depth (v,h,w) CUDA fp32; confidence (hc,wc) CUDA fp32, resized to (h,w) bilinearly with
    half-pixel centres like cv2.resize (:258) when the sizes differ; cameras as host arrays (3x3 / 4x4).
    -> dict(final, geo (h,w) bool, depth_avg (h,w), points (3,h,w)[, masks (v,K,h,w) bool, reproj_depth (v,h,w)])."""
    h, w = ref_depth.shape[-2:]
    if tuple(confidence.shape[-2:]) != (h, w):
        confidence = torch.nn.functional.interpolate(confidence.reshape(1, 1, *confidence.shape[-2:]), size=(h, w), mode="bilinear",
                                                     align_corners=False).reshape(h, w)
    thr_dist, thr_diff = dtu_ladder(first_rung, end_rung, dist_base, diff_base)
    mats = dtu_camera_pack(K_ref, E_ref, Ks_src, Es_src).to(ref_depth.device)
    final, geo, avg, pts, masks, rep = ops.dtu_filter(ref_depth.reshape(h, w), srcs_depth.reshape(-1, h, w), confidence.reshape(h, w), mats,
                                                      thr_dist, thr_diff, first_rung, end_rung, float(conf_thres), 0.75, bool(want_masks))
    out = {"final": final.bool(), "geo": geo.bool(), "depth_avg": avg, "points": pts}
    if want_masks:
        out["masks"], out["reproj_depth"] = masks.bool(), rep
    return out


# ---- the same filter for a whole scene: all of a rank's reference views in one launch -----------------------------
DTU_MAX_SOURCES = 31          # the kernel's histogram limit


class DtuSceneCameras:
    """The DTU filter's camera packs of every view of a scene, built once on the host (see dtu_scene_cameras).

    mats (N, 34 + 50 vmax) float32: row i is dtu_camera_pack of view i and its sources, zero padded to vmax sources;
    src (N, vmax) int32: the sources of view i, zero padded; count (N,) int32: their number."""

    def __init__(self, mats: torch.Tensor, src: torch.Tensor, count: torch.Tensor):
        self.mats, self.src, self.count = mats, src, count
        self.n_views, self.vmax = src.shape
        self._rows = {}

    def rows(self, views, device, stack_rows=None):
        """the device arrays of effimvs_dtu_filter_views_f32 for reference views `views` (in that order):
        (ref_idx (n,), src_idx (n,vmax), src_count (n,) int32, mats (n, 34 + 50 vmax) float32).  Indices are scene view
        numbers, or stack_rows[view] where the depth stack holds the scene's maps in another order.  Built and uploaded in
        one host -> device copy the first time a list is asked for, then cached: a host -> device copy synchronises the
        host with the stream and cannot be captured in a CUDA graph, so the first call for a list comes before a capture."""
        views = [int(i) for i in views]
        key = (tuple(views), str(device), None if stack_rows is None else tuple(sorted(stack_rows.items())))
        if key not in self._rows:
            for i in views:
                if not 0 <= i < self.n_views:
                    raise ValueError("view {} is outside the scene's {} views".format(i, self.n_views))
            n, R = len(views), self.mats.shape[1]
            sel = torch.as_tensor(views, dtype=torch.long)
            ref, src = sel.to(torch.int32), self.src[sel]
            if stack_rows is not None:
                ref = torch.as_tensor([stack_rows[i] for i in views], dtype=torch.int32)
                for b, i in enumerate(views):
                    c = int(self.count[i])
                    src[b, :c] = torch.as_tensor([stack_rows[int(j)] for j in self.src[i, :c]], dtype=torch.int32)
            host = torch.cat([ref, src.reshape(-1), self.count[sel], self.mats[sel].view(torch.int32).reshape(-1)])
            dev = host.to(device)
            a, b, c = n, n + n * self.vmax, 2 * n + n * self.vmax
            self._rows[key] = (dev[:a], dev[a:b].view(n, self.vmax), dev[b:c], dev[c:].view(torch.float32).view(n, R))
        return self._rows[key]


def dtu_scene_cameras(K, E, fuse_pairs) -> DtuSceneCameras:
    """Camera packs of every view of a scene for the batched DTU filter.  K (N,3,3), E (N,4,4) host arrays (float32, as
    upstream reads them from the cam files); fuse_pairs[i]: the 1 .. 31 source views of view i.  Row i is
    dtu_camera_pack(K[i], E[i], K[fuse_pairs[i]], E[fuse_pairs[i]]) bit for bit: the same NumPy float32 calls."""
    import numpy as np
    K = np.asarray(K.cpu() if torch.is_tensor(K) else K, dtype=np.float32)
    E = np.asarray(E.cpu() if torch.is_tensor(E) else E, dtype=np.float32)
    N = K.shape[0]
    if K.shape != (N, 3, 3) or E.shape != (N, 4, 4):
        raise ValueError("K (N,3,3) and E (N,4,4) of the same N, got {} and {}".format(K.shape, E.shape))
    if len(fuse_pairs) != N:
        raise ValueError("{} source lists for {} views".format(len(fuse_pairs), N))
    pairs = [[int(j) for j in p] for p in fuse_pairs]
    for i, p in enumerate(pairs):
        if not 1 <= len(p) <= DTU_MAX_SOURCES:
            raise ValueError("view {} has {} source views; the DTU filter takes 1 to {}".format(i, len(p), DTU_MAX_SOURCES))
        if any(not 0 <= j < N for j in p):
            raise ValueError("view {}: source views {} are outside the scene's {} views".format(i, p, N))
    vmax = max(len(p) for p in pairs)
    mats = torch.zeros(N, 34 + 50 * vmax, dtype=torch.float32)
    src = torch.zeros(N, vmax, dtype=torch.int32)
    for i, p in enumerate(pairs):
        row = dtu_camera_pack(K[i], E[i], [K[j] for j in p], [E[j] for j in p])
        mats[i, :row.numel()] = row
        src[i, :len(p)] = torch.as_tensor(p, dtype=torch.int32)
    return DtuSceneCameras(mats, src, torch.as_tensor([len(p) for p in pairs], dtype=torch.int32))


def dtu_filter_views(depth_stack, views, confs, table: DtuSceneCameras, conf_thres: float = 0.5, stack_rows=None,
                     first_rung: int = DTU_FIRST_RUNG, end_rung: int = DTU_END_RUNG, dist_base: float = DTU_DIST_BASE,
                     diff_base: float = DTU_DIFF_BASE):
    """Upstream's DTU ``filter_depth`` (test_dtu_dypcd.py:236-337) for the reference views `views` in ONE launch.

    depth_stack (N,h,w) CUDA fp32 holds the depth map of every view of the scene (the scene runner's all-gathered maps);
    each view's reference and source maps are read from it in place.  stack_rows: {view: row of depth_stack} when the
    stack is not in scene order (default: view i is row i, and N is the scene's view count).  confs (n,hc,wc) CUDA fp32,
    resized to (h,w) as dtu_filter_view does; table from dtu_scene_cameras.  Makes no host synchronisation once the
    table's rows for `views` are on the device (table.rows), so it can be captured in a CUDA graph.
    -> dict(final, geo (n,h,w) bool, depth_avg (n,h,w), points (n,3,h,w)); view views[b]'s results are bit-identical to
    dtu_filter_view on that view alone."""
    views = [int(i) for i in views]
    if not views:
        raise ValueError("no reference view to filter")
    if any(not 0 <= i < table.n_views for i in views):
        raise ValueError("views {} are not all inside the scene's {} views".format(views, table.n_views))
    if depth_stack.dim() != 3:
        raise ValueError("depth_stack must be (N,h,w), got {}".format(tuple(depth_stack.shape)))
    N, h, w = depth_stack.shape
    if stack_rows is None and N != table.n_views:
        raise ValueError("the depth stack holds {} maps, the camera table {} views".format(N, table.n_views))
    if stack_rows is not None:
        need = set(views) | {int(j) for i in views for j in table.src[i, :int(table.count[i])]}
        if any(i not in stack_rows or not 0 <= stack_rows[i] < N for i in need):
            raise ValueError("views {} are not all rows of the {}-map depth stack".format(sorted(need), N))
    n = len(views)
    if confs.dim() != 3 or confs.shape[0] != n:
        raise ValueError("confs must be (n,hc,wc) for n = {} views, got {}".format(n, tuple(confs.shape)))
    if tuple(confs.shape[-2:]) != (h, w):
        confs = torch.nn.functional.interpolate(confs.reshape(n, 1, *confs.shape[-2:]), size=(h, w), mode="bilinear",
                                                align_corners=False).reshape(n, h, w)
    thr_dist, thr_diff = dtu_ladder(first_rung, end_rung, dist_base, diff_base)
    ref, src, count, mats = table.rows(views, depth_stack.device, stack_rows)
    final, geo, avg, pts = ops.dtu_filter_views(depth_stack, ref, src, count, mats, confs, thr_dist, thr_diff, first_rung,
                                                end_rung, float(conf_thres), 0.75)
    return {"final": final.bool(), "geo": geo.bool(), "depth_avg": avg, "points": pts}


# ---- the scene's coloured point cloud (test_tank.py:517-570, test_dtu_dypcd.py:339-350) ---------------------------
_IMAGE_ROWS = {}          # (views, device) -> (n,) int32 device copy of the image row of every view


def require_cuda(*tensors):
    """the library's CUDA-only error for any CPU tensor among `tensors` (None entries are skipped)"""
    if any(t is not None and not t.is_cuda for t in tensors):
        raise RuntimeError("effimvs::compact_points got a CPU tensor; the hot path is CUDA-only (no fallback)")


def compact_points(final, points, views, images=None):
    """Upstream's vertex and colour collection for n reference views in three launches: the kept points of every view,
    in the order of `views` and in raster order within a view -- bit for bit ``points[b][:, final[b]].t()`` per view --
    and their colours from the reference images.

    final (n,h,w) or (n,1,h,w) bool and points (n,3,h,w) fp32 CUDA, as filter_views / dtu_filter_views return them;
    views: the scene view number of each of the n rows (the row of `images` its colours come from); images (N,3,h,w) fp32
    CUDA, e.g. run_scene's, or None for points only.  A colour byte is trunc(clamp(image * 255, 0, 255)) (NaN: 0), which
    on [0,1] is NumPy's (image * 255).astype(np.uint8) and gives back the byte of a u8 / 255 image.
    -> (points (total,3) fp32, colors (total,3) uint8 or None, offsets: host list of n+1 ints, view b's points being rows
    offsets[b] .. offsets[b+1] - 1).  The one host synchronisation is the read of the offsets, which sizes the outputs.
    The device copy of the image rows is made once per distinct `views` and cached."""
    views = [int(i) for i in views]
    if not views:
        raise ValueError("no view to take points from")
    if final.dim() == 4 and final.shape[1] == 1:
        final = final.reshape(final.shape[0], *final.shape[2:])
    if final.dim() != 3 or points.dim() != 4 or tuple(points.shape) != (final.shape[0], 3, *final.shape[1:]):
        raise ValueError("final (n,h,w) and points (n,3,h,w) of the same n, h, w, got {} and {}".format(tuple(final.shape),
                                                                                                         tuple(points.shape)))
    n, h, w = final.shape
    if len(views) != n:
        raise ValueError("{} views for {} masks".format(len(views), n))
    if images is not None:
        if images.dim() != 4 or images.shape[1] != 3 or tuple(images.shape[-2:]) != (h, w):
            raise ValueError("images must be (N,3,{},{}) like the depth maps, got {}".format(h, w, tuple(images.shape)))
        if any(not 0 <= i < images.shape[0] for i in views):
            raise ValueError("views {} are not all rows of the {} images".format(views, images.shape[0]))
    require_cuda(final, points, images)
    rows = None
    if images is not None:
        key = (tuple(views), str(images.device))
        if key not in _IMAGE_ROWS:
            _IMAGE_ROWS[key] = torch.as_tensor(views, dtype=torch.int32).to(images.device)
        rows = _IMAGE_ROWS[key]
    view_offsets, ws = ops.point_offsets(final)
    offsets = view_offsets.cpu().tolist()
    pts, colors = ops.gather_points(final, points, images, rows, ws, offsets[-1])
    return pts, (colors if images is not None else None), offsets
