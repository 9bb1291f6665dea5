"""CPU: host-side logic of the product package -- URDF loader, model compiler (topology + link
table), API validation and error behaviour, learnable-parameter plumbing, and that the C-ABI
library loads and exports every symbol include/drm_b200.h declares (no compute without a GPU)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from conftest import REPO, assert_close, load_golden, urdf_path
import differentiable_robot_model_b200 as drm
from differentiable_robot_model_b200 import engine, link_table
from differentiable_robot_model_b200.rigid_body_params import PositiveScalar, UnconstrainedScalar, UnconstrainedTensor


def quiet(stem, capsys=None, device="cpu"):
    return drm.DifferentiableRobotModel(urdf_path(stem), stem, device=device)


def test_loader_matches_reference_parse(robot_stem):
    g = load_golden(robot_stem)
    m = quiet(robot_stem)
    N = len(m._bodies)
    assert m.get_link_names() == g["link_names"].tolist()
    assert m._n_dofs == int((g["dof"] >= 0).sum())
    assert m._parent_idx == g["parent"].tolist()
    assert [(-1 if b.joint_idx is None else b.joint_idx) for b in m._bodies] == g["dof"].tolist()
    for i, b in enumerate(m._bodies):
        np.testing.assert_array_equal(b.trans().reshape(3).numpy(), g["trans"][i])
        np.testing.assert_array_equal(b.rot_angles().reshape(3).numpy(), g["rpy"][i])
        np.testing.assert_array_equal(b.joint_axis.reshape(3).numpy(), g["axis"][i])
        np.testing.assert_array_equal(b.inertia.mass().reshape(()).numpy(), g["mass"][i])
        np.testing.assert_array_equal(b.inertia.com().reshape(3).numpy(), g["com"][i])
        np.testing.assert_array_equal(b.inertia.inertia_mat().reshape(3, 3).numpy(), g["inertia"][i])
        d = b.get_joint_damping_const()
        assert (0.0 if d is None else float(d)) == float(g["damping"][i])
    lim = m.get_joint_limits()
    got = np.array([[l["lower"], l["upper"], l["velocity"], l["effort"]] for l in lim])
    np.testing.assert_array_equal(got, g["limits"])
    assert m._controlled_joints == [i for i in range(N) if g["dof"][i] >= 0]


def test_topology_and_table(robot_stem):
    g = load_golden(robot_stem)
    m = quiet(robot_stem)
    t = m._topology
    N = t.n_links
    assert list(t.parent[:N]) == g["parent"].tolist()
    assert list(t.dof[:N]) == g["dof"].tolist()
    for i in range(N):
        ax = g["axis"][i]
        code = t.axis[i]
        if g["dof"][i] < 0:
            assert code == 0
        else:
            k = abs(code) - 1
            assert ax[k] == np.sign(code) and np.count_nonzero(ax) == 1
    table = m._link_table().double().numpy()
    assert table.shape == (N, link_table.TABLE_STRIDE)
    from oracle import drm_oracle as O
    robot = O.load_robot(urdf_path(robot_stem), torch.float64)
    for i in range(N):
        Rj, tj = O.joint_transform(robot, i, torch.zeros(1, max(robot.n_dofs, 1), dtype=torch.float64))
        assert_close(table[i, 0:9].reshape(3, 3), Rj[0].numpy(), what="F")           # Q(0) = I
        assert_close(table[i, 9:12], robot.trans[i].numpy(), what="r")
        c = robot.com[i].numpy()
        S = np.array([[0, -c[2], c[1]], [c[2], 0, -c[0]], [-c[1], c[0], 0]])
        Io = robot.inertia[i].numpy() + float(robot.mass[i]) * S @ S.T
        assert_close(table[i, 12:21].reshape(3, 3), Io, what="I_o")
        assert_close(table[i, 21:24], float(robot.mass[i]) * c, what="mc")
        assert_close(table[i, 24], float(robot.mass[i]), what="m")
        assert_close(table[i, 25], float(robot.damping[i]), what="damping")
    # constant model: the table is cached
    assert m._link_table() is m._link_table()


def test_wrappers_and_exports():
    for cls, n in ((drm.DifferentiableKUKAiiwa, 7), (drm.DifferentiableFrankaPanda, 7),
                   (drm.DifferentiableTwoLinkRobot, 2), (drm.DifferentiableTrifingerEdu, 9)):
        m = cls()
        # the default device is the current CUDA device where there is one, the CPU (a host-side model) elsewhere
        assert m._n_dofs == n and m._device.type == ("cuda" if torch.cuda.is_available() else "cpu")
        assert os.path.exists(m.urdf_path)


def test_argument_validation_matches_reference_exceptions():
    m = drm.DifferentiableKUKAiiwa(device="cpu")
    with pytest.raises(AssertionError):                       # wrong DoF count (robot_model.py:153)
        m.compute_forward_kinematics(torch.zeros(3, 6), "iiwa_link_ee")
    with pytest.raises(AssertionError):                       # ndim 3 (robot_model.py:43)
        m.compute_forward_kinematics(torch.zeros(2, 3, 7), "iiwa_link_ee")
    with pytest.raises(AssertionError):                       # batch mismatch (robot_model.py:45-48)
        m.compute_inverse_dynamics(torch.zeros(3, 7), torch.zeros(4, 7), torch.zeros(3, 7))
    with pytest.raises(KeyError):                             # unknown link (robot_model.py:245)
        m.compute_forward_kinematics(torch.zeros(3, 7), "no_such_link")
    with pytest.raises(AttributeError):                       # bad parameter name (robot_model.py:676)
        m.make_link_param_learnable("iiwa_link_1", "colour", UnconstrainedScalar())
    with pytest.raises(AssertionError):                       # not learnable (robot_model.py:696-698)
        m.freeze_learnable_link_param("iiwa_link_1", "mass")


def test_no_cpu_fallback():
    """The product path must fail loudly instead of computing on the CPU."""
    m = drm.DifferentiableKUKAiiwa(device="cpu")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.compute_forward_kinematics(torch.zeros(3, 7), "iiwa_link_ee")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.compute_inverse_dynamics(torch.zeros(3, 7), torch.zeros(3, 7), torch.zeros(3, 7))


def test_learnable_parameter_plumbing():
    m = drm.DifferentiableKUKAiiwa()
    base = m._link_table().clone()
    m.make_link_param_learnable("iiwa_link_1", "mass", PositiveScalar(init_param=torch.tensor(4.0)))
    m.make_link_param_learnable("iiwa_link_1", "inertia_mat", UnconstrainedTensor(dim1=3, dim2=3))
    m.make_link_param_learnable("iiwa_link_2", "trans", UnconstrainedTensor(dim1=1, dim2=3))
    m.make_link_param_learnable("iiwa_link_2", "rot_angles", UnconstrainedTensor(dim1=1, dim2=3))
    m.make_link_param_learnable("iiwa_link_3", "joint_damping", UnconstrainedScalar())
    m.make_link_param_learnable("iiwa_link_3", "com", UnconstrainedTensor(dim1=1, dim2=3))
    names = [n for n, _ in m.named_parameters()]
    assert sorted(names) == sorted(["_bodies.1.inertia.mass.l", "_bodies.1.inertia.inertia_mat.param",
                                    "_bodies.2.trans.param", "_bodies.2.rot_angles.param",
                                    "_bodies.3.joint_damping.param", "_bodies.3.inertia.com.param"])
    table = m._link_table()
    assert table.requires_grad
    assert float(table[1, 24]) == pytest.approx(4.0)
    assert not torch.equal(table[2, 0:12].detach(), base[2, 0:12])
    table.sum().backward()
    for _, p in m.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all()
    # rows of untouched links are unchanged
    assert torch.equal(table[4:].detach(), base[4:])
    # freeze / unfreeze
    m.freeze_learnable_link_param("iiwa_link_1", "mass")
    assert not m._bodies[1].inertia.mass.l.requires_grad
    m.unfreeze_learnable_link_param("iiwa_link_1", "mass")
    assert m._bodies[1].inertia.mass.l.requires_grad
    # a model with parametrisation modules re-evaluates them on every call (like the reference), so edits that do
    # not bump a Parameter's version counter (p.data.copy_) can never leave a stale table behind
    with torch.no_grad():
        t1 = m._link_table()
        assert torch.equal(m._link_table(), t1)
        m._bodies[2].trans.param.data.add_(1.0)
        t2 = m._link_table()
        assert not torch.equal(t1, t2)
    # a constant model builds its table once; in-place edits of the URDF constants need invalidate_link_table()
    c = drm.DifferentiableKUKAiiwa()
    t1 = c._link_table()
    assert c._link_table() is t1
    c.invalidate_link_table()
    assert c._link_table() is not t1 and torch.equal(c._link_table(), t1)


def test_fixed_joint_origin_is_frozen_like_the_reference():
    """Reference quirk 4: trans / rot_angles of a fixed-joint link are baked in at construction."""
    m = drm.DifferentiableKUKAiiwa()
    base = m._link_table().clone()
    m.make_link_param_learnable("iiwa_link_ee", "trans", UnconstrainedTensor(dim1=1, dim2=3))
    assert torch.equal(m._link_table().detach()[8, 9:12], base[8, 9:12])


def test_non_axis_aligned_joint_is_rejected(tmp_path):
    src = open(urdf_path("2link_robot")).read().replace('<axis xyz="0 0 1"/>', '<axis xyz="0 0.6 0.8"/>', 1)
    p = tmp_path / "skew.urdf"
    p.write_text(src)
    with pytest.raises(ValueError, match="signed coordinate axis"):
        drm.DifferentiableRobotModel(str(p))


def test_c_abi_library_exports_every_declared_symbol():
    lib_path = engine.library_path()
    if not os.path.exists(lib_path):
        subprocess.run(["make", "-C", os.path.dirname(lib_path), "-j8"], check=True, capture_output=True)
    header = open(os.path.join(REPO, "include", "drm_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = sorted(set(re.findall(r"\b(drmb200_\w+)\s*\(", header)))
    assert len(declared) >= 10
    handle = ctypes.CDLL(lib_path)
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in include/drm_b200.h but not exported"
    assert sorted(engine.declared_symbols()) == declared       # the Python binding covers the whole header
    lib = engine.lib()
    assert lib.drmb200_version() >= 100
    launches = lib.drmb200_launch_count()
    if not torch.cuda.is_available():
        assert launches == 0                                   # nothing can have launched without a GPU
    # argument validation happens before any device work, so it can be exercised here
    topo = drm.DifferentiableKUKAiiwa()._topology
    rc = lib.drmb200_fk_jacobian(ctypes.byref(topo), 99, None, None, 4, None, None, None, None, None)
    assert rc == -1 and b"ee_link" in lib.drmb200_last_error()
    rc = lib.drmb200_inverse_dynamics(ctypes.byref(topo), None, None, None, None, -5, 3, None, None)
    assert rc == -1
    assert lib.drmb200_launch_count() == launches              # rejected calls launch nothing


def test_spatial_inertia_value_operations_match_the_oracle():
    """DifferentiableSpatialRigidBodyInertia.multiply_motion_vec / get_spatial_mat (spatial_vector_algebra.py:321-372)
    against the oracle's restatements (pinned to the reference through the dynamics golden vectors)."""
    import differentiable_robot_model_b200 as drm
    from differentiable_robot_model_b200.spatial_vector_algebra import (DifferentiableSpatialRigidBodyInertia,
                                                                         SpatialMotionVec)
    from oracle import drm_oracle as O
    m = drm.DifferentiableKUKAiiwa(device="cpu")
    robot = O.load_robot(m.urdf_path, torch.float32)
    gen = torch.Generator().manual_seed(0)
    ang, lin = torch.randn(5, 3, generator=gen), torch.randn(5, 3, generator=gen)
    for i in (1, 4, 7):
        inertia = m._bodies[i].inertia
        assert isinstance(inertia, DifferentiableSpatialRigidBodyInertia)
        f = inertia.multiply_motion_vec(SpatialMotionVec(lin_motion=lin, ang_motion=ang))
        o_lin, o_ang = O._inertia_times(robot, i, ang, lin)
        assert torch.allclose(f.lin, o_lin, atol=1e-6) and torch.allclose(f.ang, o_ang, atol=1e-6)
        assert torch.allclose(inertia.get_spatial_mat(), O._spatial_inertia(robot, i), atol=1e-7)


def test_per_joint_value_helpers_match_the_oracle():
    """DifferentiableRigidBody.update_joint_state / update_joint_acc (rigid_body.py:130-165) against the oracle's
    joint_transform for every movable Kuka joint."""
    import differentiable_robot_model_b200 as drm
    from oracle import drm_oracle as O
    m = drm.DifferentiableKUKAiiwa()
    robot = O.load_robot(m.urdf_path, torch.float32)
    q, qd, qdd = O.sample_inputs(robot, 6, seed=2)
    for i, body in enumerate(m._bodies):
        if body.joint_idx is None:
            continue
        k = body.joint_idx
        body.update_joint_state(q[:, k:k + 1], qd[:, k:k + 1])
        body.update_joint_acc(qdd[:, k:k + 1])
        Rj, tj = O.joint_transform(robot, i, q)
        assert torch.allclose(body.joint_pose.rotation(), Rj, atol=1e-6)
        assert torch.allclose(body.joint_pose.translation(), tj.expand(6, 3), atol=1e-7)
        assert torch.allclose(body.joint_vel.ang, qd[:, k:k + 1] @ robot.axis[i:i + 1]) and float(body.joint_vel.lin.abs().max()) == 0
        assert torch.allclose(body.joint_acc.ang, qdd[:, k:k + 1] @ robot.axis[i:i + 1])


def test_table_staging_permutation_matches_its_definition(tmp_path):
    """The select-based row permutation the kernels stage the link table with (canonical_row, csrc/drm_common.cuh)
    against the element-wise definition canon_map(), all 49 (parent axis, link axis) code pairs -- compiled for the
    host with nvcc and run on the CPU."""
    import shutil
    import subprocess
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "canon_check")
    subprocess.run([nvcc, "-std=c++17", "-arch=sm_100a", "-I", os.path.join(repo, "differentiable_robot_model_b200", "csrc"),
                    "-o", exe, os.path.join(repo, "tests", "host_checks", "canon_check.cu")], check=True, capture_output=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert "all 49" in out.stdout


def test_fused_parameter_map_reproduces_the_per_module_raw_rows():
    """link_table.FusedLinkParameters (one flat Parameter for all learnable link parameters): applying its
    (src, kind, off) map to the flat vector on the CPU gives exactly the raw rows the per-module path gathers, for
    identity (UnconstrainedScalar / UnconstrainedTensor) and squared (PositiveScalar) parametrisations; modules on
    fixed-joint origins feed nothing; the modules' own Parameters become views of the flat storage."""
    from differentiable_robot_model_b200.link_table import FusedLinkParameters, gather_raw_parameters
    from differentiable_robot_model_b200.rigid_body_params import PositiveScalar, UnconstrainedScalar
    torch.manual_seed(0)
    m = drm.DifferentiableKUKAiiwa(device="cpu")
    m.make_link_param_learnable("iiwa_link_1", "mass", PositiveScalar(min_val=0.5))
    m.make_link_param_learnable("iiwa_link_3", "com", UnconstrainedTensor(dim1=1, dim2=3))
    m.make_link_param_learnable("iiwa_link_3", "inertia_mat", UnconstrainedTensor(dim1=3, dim2=3))
    m.make_link_param_learnable("iiwa_link_5", "joint_damping", UnconstrainedScalar())
    m.make_link_param_learnable("iiwa_link_2", "trans", UnconstrainedTensor(dim1=1, dim2=3))
    m.make_link_param_learnable("iiwa_link_ee", "trans", UnconstrainedTensor(dim1=1, dim2=3))      # fixed joint: frozen
    want = gather_raw_parameters(m._bodies, torch.device("cpu")).detach().clone()
    fused = FusedLinkParameters(m._bodies, torch.device("cpu"))
    flat = fused.flat.detach()
    assert flat.numel() == 1 + 3 + 9 + 1 + 3 + 3
    src, kind, off = fused.src.long(), fused.kind, fused.off
    vals = torch.where(kind == 1, flat[src.clamp_min(0)] ** 2 + off, flat[src.clamp_min(0)])
    raw = torch.where(src >= 0, vals, fused.const_raw.reshape(-1)).reshape(want.shape)
    assert torch.equal(raw, want)
    assert int((src >= 0).sum()) == flat.numel() - 3                    # the fixed link's trans feeds nothing
    # the modules' Parameters alias the flat vector: an optimiser step on `flat` is visible through the modules
    with torch.no_grad():
        fused.flat.add_(1.0)
    com = m._bodies[3].inertia.com.param
    start = (com.data_ptr() - fused.flat.data_ptr()) // 4
    assert 0 <= start <= flat.numel() - 3 and torch.equal(com.detach().reshape(-1), fused.flat.detach()[start:start + 3])
    assert all(not p.requires_grad for n, p in m.named_parameters())


def test_tuning_options_round_trip_without_a_gpu():
    """drmb200_set_option / drmb200_get_option are host-side state: defaults, round trip, unknown names."""
    from differentiable_robot_model_b200 import engine

    assert engine.get_option("rnea_bwd_chain") in (0, 1)
    before = engine.get_option("rnea_tile")
    try:
        engine.set_option("rnea_tile", 64)
        assert engine.get_option("rnea_tile") == 64
    finally:
        engine.set_option("rnea_tile", before)
    with pytest.raises(RuntimeError):
        engine.get_option("no_such_option")
    with pytest.raises(RuntimeError):
        engine.set_option("no_such_option", 1)
