"""The dynamic filter for whole scenes, host side (CPU): the source-list checks of fusion.dynamic_scene_cameras, the
rows handed to the batched kernel (scene order and a stack of its own), the argument checks of fusion.filter_views --
all raised before anything is launched -- and the C-ABI's rejection of bad arguments.  The kernel behind the same
interface is covered by test_gpu_dynamic_scene."""
import ctypes

import pytest
import torch

import effimvs_b200  # noqa: F401
from effimvs_b200 import capi, fusion

H, W = 48, 64
RAGGED = [[1, 2, 3], [0], [4, 6, 0, 1, 5], [2, 4], [3, 5, 6, 0, 1, 2], [6], [5, 4, 3]]     # source lists of a 7-view scene


def _table(pairs=RAGGED):
    """a table built on the host: the cameras and an inverse table of the right shape (the device builds the real one)"""
    n = len(pairs)
    cams = torch.eye(4).repeat(n, 2, 1, 1)
    cams[:, 0, 0, 3] = torch.arange(n, dtype=torch.float32)
    return fusion.DynamicSceneCameras(cams, torch.linalg.inv(cams), pairs)


def test_source_lists_are_checked_before_any_launch():
    cams = torch.zeros(20, 2, 4, 4)
    with pytest.raises(ValueError, match="view 19 has 17 source views"):
        fusion.dynamic_scene_cameras(cams, [[0]] * 19 + [list(range(17))])                     # 16 is the limit
    with pytest.raises(ValueError, match="view 3 has 0"):
        fusion.dynamic_scene_cameras(cams, [[1]] * 3 + [[]] + [[1]] * 16)                      # no source
    with pytest.raises(ValueError, match="view 19: source views"):
        fusion.dynamic_scene_cameras(cams, [[1]] * 19 + [[20]])                                # outside the scene
    with pytest.raises(ValueError, match="view 0: source views"):
        fusion.dynamic_scene_cameras(cams, [[-1]] + [[1]] * 19)
    with pytest.raises(ValueError, match="19 source lists for 20 views"):
        fusion.dynamic_scene_cameras(cams, [[1]] * 19)
    with pytest.raises(ValueError, match=r"\(N,2,4,4\)"):
        fusion.dynamic_scene_cameras(cams[:, 0], [[1]] * 20)
    # valid lists reach the inverse kernel, which takes no host tensor: no silent CPU path
    with pytest.raises(RuntimeError, match="CPU tensor"):
        fusion.dynamic_scene_cameras(cams, [[j for j in range(20) if j != i][:16] for i in range(20)])


def test_rows_in_scene_order_and_in_a_stack_of_its_own():
    table = _table()
    assert table.n_views == 7 and table.vmax == 6
    ref, src, count, cams, inv = table.rows([4, 1, 2], "cpu")
    assert ref.dtype == src.dtype == count.dtype == torch.int32
    assert ref.tolist() == [4, 1, 2] and count.tolist() == [6, 1, 5]
    assert src.tolist() == [RAGGED[4], [0] + [0] * 5, RAGGED[2] + [0]]
    assert cams is table.cams and inv is table.inv                            # scene order: the tables themselves
    assert table.rows([4, 1, 2], "cpu")[0] is ref                             # built once per list
    # view 2 with its own maps stacked as [ref, sources in order] in a 6-map stack
    rows = {2: 0, 4: 1, 6: 2, 0: 3, 1: 4, 5: 5}
    ref, src, count, cams, inv = table.rows([2], "cpu", rows, 6)
    assert ref.tolist() == [0] and src[0, :5].tolist() == [1, 2, 3, 4, 5] and count.tolist() == [5]
    for view, r in rows.items():                                              # the cameras follow the stack's rows
        assert torch.equal(cams[r], table.cams[view]) and torch.equal(inv[r], table.inv[view])


def test_filter_views_rejects_bad_input_naming_the_view():
    table = _table()
    stack, confs = torch.ones(7, H, W), torch.ones(2, H // 2, W // 2)
    args = (2.0, 6.0, 1, 0.3)
    with pytest.raises(ValueError, match="view 7 is outside"):
        fusion.filter_views(stack, [0, 7], confs, table, *args)
    with pytest.raises(ValueError, match="view -1 is outside"):
        fusion.filter_views(stack, [0, -1], confs, table, *args)
    with pytest.raises(ValueError, match="view 1 has 1 source views, fewer than thres_view = 2"):
        fusion.filter_views(stack, [0, 1], confs, table, 2.0, 6.0, 2, 0.3)
    with pytest.raises(ValueError, match="thres_view"):
        fusion.filter_views(stack, [0, 2], confs, table, 2.0, 6.0, 0, 0.3)
    with pytest.raises(ValueError, match="positive"):
        fusion.filter_views(stack, [0, 2], confs, table, 0.0, 6.0, 1, 0.3)
    with pytest.raises(ValueError, match="positive"):
        fusion.filter_views(stack, [0, 2], confs, table, 2.0, -1.0, 1, 0.3)
    with pytest.raises(ValueError, match="6 maps"):
        fusion.filter_views(stack[:6], [0, 1], confs, table, *args)                            # stack != scene
    with pytest.raises(ValueError, match="for n = 3 views"):
        fusion.filter_views(stack, [0, 1, 2], confs, table, *args)                              # 2 maps for 3 views
    with pytest.raises(ValueError, match=r"\(N,h,w\)"):
        fusion.filter_views(stack[0], [0, 1], confs, table, *args)
    with pytest.raises(ValueError, match="view 0: views"):
        fusion.filter_views(stack[:3], [0], confs[:1], table, *args, stack_rows={0: 0, 1: 1, 2: 2})        # source 3 not stacked
    with pytest.raises(ValueError, match="view 0: views"):
        fusion.filter_views(stack[:3], [0], confs[:1], table, *args, stack_rows={0: 0, 1: 1, 2: 2, 3: 3})  # beyond the stack
    with pytest.raises(ValueError, match="a depth-stack row each"):
        fusion.filter_views(stack[:3], [1], confs[:1], table, *args, stack_rows={1: 0, 0: 0})            # two views, one row
    with pytest.raises(ValueError, match="no reference view"):
        fusion.filter_views(stack, [], confs[:0], table, *args)
    assert not table._rows                                                    # nothing was uploaded for a rejected call


def test_c_abi_rejects_bad_arguments():
    """effimvs_fusion_filter_views_f32 checks pointers, sizes, the bases and thres_view on the host, before any launch"""
    lib, one = capi.lib, ctypes.c_void_p(16)

    def call(n_depths=8, vmax=10, n=3, h=8, w=8, hc=4, wc=4, dist_base=2.0, rel_diff_base=6.0, thres_view=2, depths=one,
             inv=one):
        return lib.effimvs_fusion_filter_views_f32(depths, n_depths, one, one, one, vmax, one, inv, one, hc, wc, dist_base,
                                                   rel_diff_base, thres_view, 0.3, 0, n, h, w, one, one, one, None)
    assert call(vmax=17) == capi.EINVAL and "vmax=17" in capi.last_error()        # beyond the shared camera records
    assert call(vmax=0) == capi.EINVAL
    assert call(n=0) == capi.EINVAL
    assert call(n=65536) == capi.EINVAL and "n=65536" in capi.last_error()
    assert call(n_depths=0) == capi.EINVAL
    assert call(h=1) == capi.EINVAL
    assert call(w=0) == capi.EINVAL
    assert call(hc=0) == capi.EINVAL
    assert call(wc=-1) == capi.EINVAL
    assert call(h=65536, w=65536) == capi.EINVAL                                 # h * w beyond int
    assert call(dist_base=0.0) == capi.EINVAL and "positive" in capi.last_error()
    assert call(rel_diff_base=-6.0) == capi.EINVAL
    assert call(thres_view=0) == capi.EINVAL and "thres_view=0" in capi.last_error()
    assert call(thres_view=11) == capi.EINVAL                                    # more than any view can have
    assert call(depths=None) == capi.EINVAL and "null" in capi.last_error()
    assert call(inv=None) == capi.EINVAL and "null" in capi.last_error()
