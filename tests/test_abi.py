"""CPU-side checks of the drop-in boundary: the library loads, exports every symbol include/pn2_abi.h
declares (no compute call is made -- there is no GPU here), and the host layer refuses CPU tensors."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "pn2_abi.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pn2_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_nine_reference_operators():
    syms = declared_symbols()
    for name in ["pn2_furthest_point_sampling", "pn2_gather_points", "pn2_gather_points_grad", "pn2_ball_query",
                 "pn2_group_points", "pn2_group_points_grad", "pn2_three_nn", "pn2_three_interpolate",
                 "pn2_three_interpolate_grad", "pn2_lift_views", "pn2_sa_mlp_max", "pn2_fp_mlp"]:
        assert name in syms


def test_library_exports_every_declared_symbol():
    from pn2_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "run __graft_entry__.build() first"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared_symbols():
        assert hasattr(lib, name), "libpn2_b200.so does not export %s" % name
    # and the ctypes table binds exactly the declared set
    assert sorted(_lib.EXPORTS) == declared_symbols()


def test_abi_version_and_error_string_without_gpu():
    from pn2_b200 import _lib
    lib = _lib.load()
    assert lib.pn2_abi_version() == 1
    # argument validation happens before any CUDA call, so it is testable on a CPU box
    st = lib.pn2_furthest_point_sampling(1, 0, 4, None, None, None, None)
    assert st == 1 and b"n >= 1" in lib.pn2_last_error()
    st = lib.pn2_ball_query(1, 8, 4, 0.1, 4, None, None, None, None)
    assert st == 1 and b"null pointer" in lib.pn2_last_error()
    assert lib.pn2_furthest_point_sampling(0, 8, 4, None, None, None, None) == 0  # empty batch: no-op


def test_argument_validation_of_the_wider_entry_points_without_gpu():
    """Same for the entry points added around the nine operators: bad arguments are refused with a message before any
    CUDA call; empty batches are no-ops."""
    from pn2_b200 import _lib
    lib = _lib.load()
    err = lib.pn2_last_error
    assert lib.pn2_label_counts(2, 8, 0, None, None, None, None, None, None, None) == 1 and b"classes" in err()
    assert lib.pn2_label_counts(2, 8, 21, None, None, None, None, None, None, None) == 1 and b"null pointer" in err()
    assert lib.pn2_label_counts(0, 8, 21, None, None, None, None, None, None, None) == 0
    assert lib.pn2_voxel_first_index(2, 8, None, None, ctypes.c_float(0.0), None, None, None, None, None) == 1 and b"res" in err()
    assert lib.pn2_voxel_first_index(0, 8, None, None, ctypes.c_float(0.02), None, None, None, None, None) == 0
    assert lib.pn2_inverse_index(1, 0, 4, None, None, None, None) == 1 and b"bad dims" in err()
    assert lib.pn2_scatter_rows_det(1, 4, 8, 10, 3, None, None, None, None, None, None) == 1 and b"multiple of div" in err()
    assert lib.pn2_scatter_rows_det(1, 4, 8, 9, 2, None, None, None, None, None, None) == 1 and b"div" in err()
    assert lib.pn2_lift_setup(3, None, None, None, None, None, None, None) == 1 and b"null pointer" in err()
    assert lib.pn2_lift_setup(0, None, None, None, None, None, None, None) == 0
    assert lib.pn2_grid_build(1, (1 << 18) + 1, None, ctypes.c_float(0.1), None, None, None, None, None) == 2 and b"at most" in err()
    assert lib.pn2_grid_max_points() == 1 << 18


def test_fps_policy_switch_returns_previous_value():
    from pn2_b200 import _lib
    lib = _lib.load()
    assert lib.pn2_set_fps_policy(1) == 0
    assert lib.pn2_set_fps_policy(2) == 1
    assert lib.pn2_set_fps_policy(7) == -1          # unknown policy: refused, state unchanged
    assert lib.pn2_set_fps_policy(0) == 2
    lib.pn2_debug_set_fps_mode(2)                   # the developer switch sets the same policy
    assert lib.pn2_set_fps_policy(1) == 2
    lib.pn2_debug_set_fps_mode(6)                   # unknown value: refused, policy unchanged
    assert lib.pn2_set_fps_policy(0) == 1
    from pn2_b200.pointnet_util import fps_policy
    with fps_policy("throughput"):
        assert lib.pn2_set_fps_policy(1) == 1
    assert lib.pn2_set_fps_policy(0) == 0


def test_pointnet2_cuda_dropin_surface():
    import pointnet2_cuda  # top-level shim next to the package, as model/pointnet2_utils.py:7 imports it
    for name in ["ball_query_wrapper", "group_points_wrapper", "group_points_grad_wrapper", "gather_points_wrapper",
                 "gather_points_grad_wrapper", "furthest_point_sampling_wrapper", "three_nn_wrapper",
                 "three_interpolate_wrapper", "three_interpolate_grad_wrapper"]:
        assert callable(getattr(pointnet2_cuda, name))


def test_operators_refuse_cpu_tensors():
    from pn2_b200 import Pn2Error, pointnet2_utils
    xyz = torch.zeros(1, 16, 3)
    with pytest.raises(Pn2Error):
        pointnet2_utils.furthest_point_sample(xyz, 4)
    with pytest.raises(Pn2Error):
        pointnet2_utils.ball_query(0.1, 4, xyz, xyz[:, :2].contiguous())


def test_module_state_dict_keys_match_reference_names():
    from pn2_b200.models import PointNet2SemSeg
    keys = set(PointNet2SemSeg(21).state_dict().keys())
    for k in ["sa1.mlp_convs.0.weight", "sa1.mlp_bns.2.running_var", "fp1.mlp_convs.2.bias", "conv1.weight", "bn1.weight",
              "conv2.bias"]:
        assert k in keys
    from pn2_b200.pointnet_util import PointNetSetAbstractionMsg
    msg = PointNetSetAbstractionMsg(16, [0.1, 0.2], [16, 32], 4, [[8, 16], [8, 16]])
    assert "conv_blocks.1.0.weight" in msg.state_dict() and "bn_blocks.0.1.running_mean" in msg.state_dict()
    assert msg.conv_blocks[0][0].in_channels == 7  # in_channel excludes xyz (model/pointnet_util.py:125)
