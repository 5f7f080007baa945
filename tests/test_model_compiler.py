"""URDF -> model-constants compiler: pinned against forward kinematics computed straight from the reference URDFs by
an independent homogeneous-transform walk (tests/golden/fk_reference_urdf.json, made by make_golden.py), the
known answers of SURVEY.md Appendix B, and the reference's own example configs and compiled URDFs
(tests/golden/reference_examples.json, made by make_reference_examples.py)."""
import json
import os

import numpy as np
import pytest

from mppi_isaac_b200.model.blob import compiled_path, build_scene
from mppi_isaac_b200.model.urdf import (compile_urdf, forward_kinematics, load_compiled, mesh_inertia, quat_xyzw_to_R)
from mppi_isaac_b200.utils.config_store import load_actor_cfgs, load_config, load_isaacgym_config

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_fk_of_compiled_models_matches_reference_urdf_fk():
    with open(os.path.join(GOLD, "fk_reference_urdf.json")) as f:
        gold = json.load(f)
    for case in gold["cases"]:
        model = load_compiled(compiled_path(case["urdf"]))
        pos, quat = forward_kinematics(model, case["q"], base_pos=case["base_pos"])
        assert set(model.link_names) <= set(case["links"])
        for i, name in enumerate(model.link_names):
            g = case["links"][name]
            np.testing.assert_allclose(pos[i], g["p"], atol=1e-9)
            np.testing.assert_allclose(quat_xyzw_to_R(quat[i]), np.asarray(g["R"]), atol=1e-9)


def test_appendix_b_known_answers():
    m = load_compiled(compiled_path("panda_isaac/robots/franka_panda_stick.urdf"))
    q = [0, -0.94, 0, -2.8, 0, 1.8675, 0]                        # conf/actors/panda_stick.yaml:8 de-interleaved
    pos, quat = forward_kinematics(m, q)
    n = m.link_names
    np.testing.assert_allclose(pos[n.index("panda_link7")], (0.273048, 0, 0.556218), atol=1e-6)
    np.testing.assert_allclose(pos[n.index("panda_ee_finger")], (0.273850, 0, 0.449221), atol=1e-6)
    np.testing.assert_allclose(pos[n.index("panda_ee_tip")], (0.276025, 0, 0.159229), atol=1e-6)
    np.testing.assert_allclose(np.abs(quat[n.index("panda_ee_tip")]), (0.999993, 0, 0.003750, 0), atol=1e-6)
    pos0, quat0 = forward_kinematics(m, [0] * 7)
    np.testing.assert_allclose(pos0[n.index("panda_ee_tip")], (0.088, 0, 0.636), atol=1e-9)
    g = load_compiled(compiled_path("panda_isaac/robots/franka_panda_gripper.urdf"))
    pos, quat = forward_kinematics(g, q + [0.02, 0.02])
    gn = g.link_names
    assert "panda_link8" not in gn                               # orphan second root is ignored
    np.testing.assert_allclose(pos[gn.index("panda_ee")], (0.274623, 0, 0.346224), atol=1e-6)
    np.testing.assert_allclose(pos[gn.index("panda_leftfinger")], (0.288430, -0.014142, 0.390929), atol=1e-6)
    h = load_compiled(compiled_path("heijn/heijn.urdf"))
    pos, quat = forward_kinematics(h, [0.3, -0.2, 0.5], base_pos=(0, 1.5, 0.05))
    np.testing.assert_allclose(pos[h.link_names.index("front_link")], (0.572051, 1.448622, 0.15), atol=1e-6)
    np.testing.assert_allclose(quat[h.link_names.index("front_link")], (0, 0, 0.247404, 0.968912), atol=1e-6)


def test_collision_derived_mass_properties():
    """Masses at 1000 kg/m^3 of SURVEY Appendix B (all panda URDFs have zero <inertial> tags)."""
    m = load_compiled(compiled_path("panda_isaac/robots/franka_panda_stick.urdf"))
    expect = [2.975, 3.004, 2.328, 2.374, 3.419, 1.435]           # link1..link6 (link7 carries the stick as well)
    np.testing.assert_allclose(m.mass[:6], expect, atol=1.5e-3)
    assert abs(m.mass[6] - (0.446 + 0.0911)) < 1e-3               # link7 + cylinder r=0.01 l=0.29
    np.testing.assert_allclose(m.mcom[0] / m.mass[0], (0, -0.0313, -0.0694), atol=2e-4)
    # integrator self-check: unit cube
    v = np.array([[x, y, z] for x in (0, 1) for y in (0, 1) for z in (0, 1)], float)
    t = np.array([[0, 2, 1], [1, 2, 3], [4, 5, 6], [5, 7, 6], [0, 1, 4], [1, 5, 4], [2, 6, 3], [3, 6, 7], [0, 4, 2], [2, 4, 6], [1, 3, 5], [3, 7, 5]])
    mass, com, Ic = mesh_inertia(v, t, 1000.0)
    assert abs(mass - 1000) < 1e-9 and np.allclose(com, 0.5) and np.allclose(np.diag(Ic), 1000 / 6)


def test_scene_blob_and_command_map():
    sc = build_scene(load_actor_cfgs(["panda_stick", "goal"]))
    m = sc.model
    assert (m.nb, m.nlinks, m.nu, sc.ndof) == (7, 10, 7, 7)
    assert m.gravity_on == 0 and m.drive_mode == 0 and abs(m.kd[0] - 600.0) < 1e-6      # isaacgym_wrapper.py:497-500
    assert list(m.parent[:7]) == [-1, 0, 1, 2, 3, 4, 5]
    assert [m.cmd_i0[i] for i in range(7)] == list(range(7)) and all(m.cmd_c0[i] == 1.0 for i in range(7))
    assert sc.body_names[0][-1] == "panda_ee_tip" and sc.body_names[1] == ["sphere"]
    assert sc.num_bodies == 11                                                              # SURVEY section 8 table, C2
    np.testing.assert_allclose(sc.root_state0[1, :7], [1, 1, 0.5, 0, 0, 0, 1])
    p = build_scene(load_actor_cfgs(["point_robot", "goal"]))
    assert (p.model.nb, p.model.nlinks, p.num_bodies) == (3, 7, 8)                          # C1: 7 links / 8 env bodies
    assert list(p.model.jtype[:3]) == [1, 1, 0]


def test_config_loader_builtin_and_errors(tmp_path):
    cfg = load_isaacgym_config("config_panda_b200")
    assert (cfg.mppi.num_samples, cfg.mppi.horizon, cfg.nx, cfg.isaacgym.dt, cfg.isaacgym.substeps) == (10000, 30, 14, 0.05, 2)
    assert cfg.actors == ["panda_stick", "goal"] and cfg.mppi.u_min == [-0.2]
    f = tmp_path / "t.yaml"
    f.write_text("defaults:\n  - mppi: panda_b200\n  - isaacgym: push\nnx: 14\nactors: ['panda_stick']\nmppi:\n  horizon: 12\n")
    c2 = load_config(str(f), overrides=["mppi.lambda_=0.3"])
    assert c2.mppi.horizon == 12 and c2.mppi.lambda_ == 0.3 and c2.isaacgym.dt == 0.1 and c2.mppi.num_samples == 10000
    f.write_text("defaults:\n  - mppi: panda_b200\nbogus_key: 1\n")
    with pytest.raises(KeyError):
        load_config(str(f))


def test_reference_configs_and_urdfs_load_unchanged(tmp_path):
    import glob
    with open(os.path.join(GOLD, "reference_examples.json")) as f:
        gold = json.load(f)
    for rel, text in gold["files"].items():                       # the reference's conf/ and examples/ YAMLs, verbatim
        (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
        (tmp_path / rel).write_text(text)
    conf = [str(tmp_path / "conf")]
    tasks = sorted(glob.glob(str(tmp_path / "examples" / "*" / "*.yaml")))
    assert len(tasks) >= 10
    for t in tasks:
        cfg = load_config(t, conf)
        assert cfg.mppi.num_samples > 0 and len(cfg.actors) > 0
    for rel, fresh in gold["urdf"].items():                        # compiled from the reference's assets/
        shipped = load_compiled(compiled_path(rel))
        np.testing.assert_allclose(fresh["mass"], shipped.mass, rtol=1e-12)
        np.testing.assert_allclose(fresh["inertia_o"], shipped.inertia_o, rtol=1e-9, atol=1e-12)
        assert fresh["link_names"] == shipped.link_names and fresh["dof_names"] == shipped.dof_names
    # every example scene of the reference builds from ITS conf/ on the shipped models_compiled/ into the scene its own assets/ gave
    # (anymal: legged floating base, out of scope)
    built = {}
    for t in tasks:
        cfg = load_config(t, conf)
        name = os.path.basename(os.path.dirname(t))
        try:
            sc = build_scene(load_actor_cfgs(cfg.actors, conf), substep=cfg.isaacgym.dt / cfg.isaacgym.substeps)
            built[name] = [sc.model.nb, sc.nu, sc.model.nlinks, sc.num_bodies]
        except NotImplementedError:
            built[name] = "NotImplementedError"
    assert built == gold["scenes"]
    assert built.pop("anymal") == "NotImplementedError"
    assert all(isinstance(v, list) for v in built.values()), built
    assert built["albert"][:2] == [12, 9] and built["omni_panda_pick"][:2] == [12, 12] and built["panda_effort"][:2] == [7, 7] and built["panda_stick_push"][0] == 7
    a = load_actor_cfgs(["panda_stick", "goal"], conf)
    b = load_actor_cfgs(["panda_stick", "goal"])
    assert a[0].urdf_file == b[0].urdf_file and a[0].init_joint_pose == b[0].init_joint_pose and a[1].init_pos == b[1].init_pos
