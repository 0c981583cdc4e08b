"""The scene's coloured point cloud on the device (``-m gpu``): fusion.compact_points (csrc/points.cu) against run_scene's
boolean-index extraction ``points[b][:, m].t()`` bit for bit, over mask densities, ragged tile tails, empty views, a total
of zero, views out of scene order and repeated image rows, and the 49-view DTU shape; colours against the NumPy rule of
test_scene_points_host; two runs bit-identical; run_scene(images=) with both filters end to end (points as without images,
colours at the mask, the per-view fuse the same, at most three launches over the filter's one); a PLY round trip."""
import numpy as np
import pytest
import torch

from test_scene_points_host import color_rule

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _assert_same(got, want, what):
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape)
    assert torch.equal(_bits(got), _bits(want)), what


def _reference(final, points, views, images):
    """run_scene's extraction per view, and the colours by the NumPy rule at the same pixels"""
    pts, cols = [], []
    for b, i in enumerate(views):
        m = final[b]
        pts.append(points[b][:, m].t().contiguous())
        if images is not None:
            cols.append(torch.from_numpy(color_rule(images[i][:, m].t().cpu().numpy())))
    return pts, cols


def _inputs(n, h, w, density, n_images, seed, empty=()):
    g = torch.Generator(device=DEV).manual_seed(seed)
    final = torch.rand(n, h, w, generator=g, device=DEV) < density
    for b in empty:
        final[b] = False
    points = torch.randn(n, 3, h, w, generator=g, device=DEV) * 100
    images = torch.rand(n_images, 3, h, w, generator=g, device=DEV)
    return final, points, images


def _check(final, points, views, images, what):
    from effimvs_b200 import fusion
    pts, cols, offs = fusion.compact_points(final, points, views, images)
    want_p, want_c = _reference(final, points, views, images)
    assert offs == [0] + np.cumsum([p.shape[0] for p in want_p]).tolist(), what
    assert pts.shape == (offs[-1], 3) and pts.is_contiguous()
    _assert_same(pts, torch.cat(want_p), (what, "points"))
    for b in range(len(views)):                                  # the per-view slices run_scene hands out
        _assert_same(pts[offs[b]:offs[b + 1]], want_p[b], (what, "points", b))
    if images is None:
        assert cols is None
    else:
        _assert_same(cols.cpu(), torch.cat(want_c), (what, "colors"))
    return pts, cols, offs


# (views, h, w, mask density, images, empty views)
CASES = {"density_0": ([0, 1, 2], 48, 64, 0.0, 3, ()),
         "density_1e-3": ([0, 1, 2], 128, 160, 1e-3, 3, ()),
         "density_half": ([0, 1, 2], 128, 160, 0.5, 3, ()),
         "density_0.999": ([0, 1, 2], 128, 160, 0.999, 3, ()),
         "density_1": ([0, 1, 2], 128, 160, 1.0, 3, ()),
         "one_pixel": ([0, 1, 2, 3, 4], 1, 1, 0.5, 5, ()),
         "37x53": ([0, 1, 2, 3], 37, 53, 0.5, 4, ()),             # h*w not a multiple of 16: the unvectorised path
         "tile_tail": ([0, 1], 16, 257, 0.7, 2, ()),              # one full 4096-pixel tile and a 16-pixel tail
         "one_tile": ([0, 1], 64, 64, 0.7, 2, ()),
         "empty_views": ([0, 1, 2, 3, 4], 48, 64, 0.5, 5, (0, 2, 4)),
         "scene_order": ([4, 1, 1, 3, 0], 40, 72, 0.5, 6, (1,))}   # out of scene order, image row 1 twice


@pytest.mark.parametrize("name", sorted(CASES))
def test_bit_identical_to_boolean_index(name):
    views, h, w, density, n_images, empty = CASES[name]
    final, points, images = _inputs(len(views), h, w, density, n_images, seed=len(name), empty=empty)
    _check(final, points, views, None, (name, "points only"))
    _check(final, points, views, images, name)


def test_total_zero_gives_empty_tensors():
    from effimvs_b200 import fusion
    final, points, images = _inputs(3, 37, 53, 0.0, 3, seed=1)
    pts, cols, offs = fusion.compact_points(final, points, [0, 1, 2], images)
    assert offs == [0, 0, 0, 0]
    assert pts.shape == (0, 3) and pts.dtype == torch.float32 and pts.is_cuda
    assert cols.shape == (0, 3) and cols.dtype == torch.uint8 and cols.is_cuda


def test_dtu_shape_49_views():
    final, points, images = _inputs(49, 1184, 1600, 0.999, 49, seed=3, empty=(20,))
    views = list(range(49))[::-1]
    _, _, offs = _check(final, points, views, images, "dtu49")
    print("49 views at 1600x1184: {} points".format(offs[-1]))


def _special_images(h, w):
    """channel planes of hand-picked values: k/255 and its float32 neighbours, negatives, > 1, NaN and inf"""
    k = np.arange(256, dtype=np.float32) / np.float32(255)
    vals = np.concatenate([k, np.nextafter(k, np.float32(-1)), np.nextafter(k, np.float32(2)),
                           np.float32([-0.0, -1e-30, -0.5, -1e30, 1 + 2 ** -23, 1.5, 255, 1e30, np.inf, -np.inf, np.nan])])
    rng = np.random.default_rng(7)
    img = rng.choice(vals, size=(2, 3, h, w)).astype(np.float32)
    return torch.from_numpy(img).to(DEV)


@pytest.mark.parametrize("kind", ["u8", "uniform", "special"])
def test_colors(kind):
    from effimvs_b200 import fusion
    n, h, w = 3, 96, 128
    g = torch.Generator(device=DEV).manual_seed(5)
    final = torch.rand(n, h, w, generator=g, device=DEV) < 0.6
    points = torch.randn(n, 3, h, w, generator=g, device=DEV)
    views = [1, 0, 1]
    if kind == "u8":
        u8 = torch.randint(0, 256, (2, 3, h, w), generator=g, device=DEV, dtype=torch.uint8)
        images = u8.float() / 255
    elif kind == "uniform":
        images = torch.rand(2, 3, h, w, generator=g, device=DEV)
    else:
        images = _special_images(h, w)
    _, cols, _ = _check(final, points, views, images, kind)
    if kind == "u8":                                               # the byte the image was made from, at every kept pixel
        want = torch.cat([u8[i][:, final[b]].t() for b, i in enumerate(views)])
        _assert_same(cols, want, "u8 round trip")


def test_two_runs_are_bit_identical():
    from effimvs_b200 import fusion
    final, points, images = _inputs(7, 300, 411, 0.6, 7, seed=11, empty=(3,))
    views = [6, 2, 2, 0, 5, 1, 3]
    a = fusion.compact_points(final, points, views, images)
    b = fusion.compact_points(final, points, views, images)
    _assert_same(a[0], b[0], "points")
    _assert_same(a[1], b[1], "colors")
    assert a[2] == b[2]


def _dynamic_scene(n, w, h):
    from effimvs_b200 import scene, synthetic
    E, K = synthetic.camera_arc(n, w, h)
    stack = synthetic.render_plane_scene(E, K, w, h, noise=0.05, seed=2).to(DEV)
    cams = synthetic.stage_cameras(E, K, 1)["stage4"][0].to(DEV)
    imgs = torch.randint(0, 256, (n, 3, h, w), generator=torch.Generator().manual_seed(n), dtype=torch.uint8).to(DEV)
    conf = torch.rand(n, h // 2, w // 2, generator=torch.Generator().manual_seed(4)).to(DEV)
    pairs = [[(i + d) % n for d in (1, -1, 2, -2)] for i in range(n)]
    return stack, cams, imgs, conf, pairs, scene


def _fuses(kind, cams, imgs_f, pairs):
    from effimvs_b200 import scene
    if kind == "dynamic":
        _, fuse = scene.cuda_scene_callables(None, imgs_f, {"stage4": cams}, torch.zeros(4, device=DEV), 2.0, 6.0, 2, 0.3)
    else:
        fuse = scene.cuda_dtu_fuse(cams, pairs)
    return fuse


@pytest.mark.parametrize("n", [9, 49])
@pytest.mark.parametrize("kind", ["dynamic", "dtu"])
def test_run_scene_with_images(kind, n):
    from effimvs_b200 import ops
    w, h = 96, 64
    stack, cams, u8, conf, pairs, scene = _dynamic_scene(n, w, h)
    imgs = u8.float() / 255
    fuse = _fuses(kind, cams, imgs, pairs)

    def infer(i, srcs):
        return stack[i], conf[i]
    plain = scene.run_scene(infer, fuse, n, pairs, 0, 1, DEV)           # builds the camera table, warms the row cache
    scene.run_scene(infer, fuse, n, pairs, 0, 1, DEV, images=imgs)
    before = ops.LAUNCHES
    plain = scene.run_scene(infer, fuse, n, pairs, 0, 1, DEV)
    assert ops.LAUNCHES - before == 1
    before = ops.LAUNCHES
    got = scene.run_scene(infer, fuse, n, pairs, 0, 1, DEV, images=imgs)
    assert ops.LAUNCHES - before <= 1 + 3
    per_view = scene.run_scene(infer, lambda *a: fuse(*a), n, pairs, 0, 1, DEV, images=imgs)
    masks = fuse.batch(list(range(n)), stack, conf, pairs)["final"][:, 0]
    total = 0
    for i in range(n):
        want_cols = u8[i][:, masks[i]].t()
        for run in (got, per_view):
            assert len(run[i]) == 3
            _assert_same(run[i][0], plain[i][0], (kind, "points", i))
            _assert_same(run[i][1], stack[i], (kind, "depth", i))
            _assert_same(run[i][2], want_cols, (kind, "colors", i))
        total += plain[i][0].shape[0]
    assert 0 < total < n * h * w                     # the filter keeps part of the scene: the comparison is not vacuous
    print("{} filter, {} views: {} points".format(kind, n, total))


def test_run_scene_rejects_images_of_another_size():
    w, h, n = 96, 64, 5
    stack, cams, u8, conf, pairs, scene = _dynamic_scene(n, w, h)
    fuse = _fuses("dtu", cams, None, pairs)
    with pytest.raises(ValueError, match="depth maps"):
        scene.run_scene(lambda i, s: (stack[i], conf[i]), fuse, n, pairs, 0, 1, DEV, images=torch.zeros(n, 3, h, w + 1, device=DEV))


def test_ply_round_trip_of_a_49_view_scene(tmp_path):
    from effimvs_b200 import data_io
    w, h, n = 160, 128, 49
    stack, cams, u8, conf, pairs, scene = _dynamic_scene(n, w, h)
    fuse = _fuses("dtu", cams, None, pairs)
    out = scene.run_scene(lambda i, s: (stack[i], conf[i]), fuse, n, pairs, 0, 1, DEV, images=u8.float() / 255)
    points = [out[i][0] for i in range(n)]
    colors = [out[i][2] for i in range(n)]
    path = str(tmp_path / "scene.ply")
    data_io.write_ply(path, torch.cat(points).cpu(), torch.cat(colors).cpu())
    p, c = data_io.read_ply(path)
    total = sum(t.shape[0] for t in points)
    assert total > 0 and p.shape == (total, 3) and c.shape == (total, 3)
    assert np.array_equal(p.view(np.int32), torch.cat(points).cpu().numpy().view(np.int32))
    assert np.array_equal(c, torch.cat(colors).cpu().numpy())
    masks = fuse.batch(list(range(n)), stack, conf, pairs)["final"][:, 0]
    assert np.array_equal(c, torch.cat([u8[i][:, masks[i]].t() for i in range(n)]).cpu().numpy())
