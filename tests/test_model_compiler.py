"""MJCF -> constant tables: sizes, MuJoCo compile rules, blob round trip, committed blobs in sync with the sources.

The reference's MJCF assets are not redistributed: what the tests below need from them (digests of a fresh compile, masses and an
inertial frame read from fetch/robot.xml, the unfused mass matrix) is recorded in golden/fetch_model_facts.json by
golden/make_fetch_model_facts.py."""
import hashlib
import json
import os

import numpy as np
import pytest

from gymnasium_robotics_b200.mjcf import Model, compile_mjcf
from gymnasium_robotics_b200.models import MODEL_DIR, MODEL_SOURCES, load_model

FACTS = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fetch_model_facts.json")))


def test_committed_blobs_load_and_have_expected_sizes():
    m = load_model("fetch_pick_and_place")
    assert (m.nq, m.nv, m.nu, m.nmocap, m.neq) == (22, 21, 2, 1, 1)  # SURVEY.md section 8 sizes table
    r = load_model("fetch_reach")
    assert (r.nq, r.nv, r.nu) == (15, 15, 0)
    robot = [n for n in m.names["joint"] if n.startswith("robot")]
    assert len(robot) == 15 and robot[-2:] == ["robot0:r_gripper_finger_joint", "robot0:l_gripper_finger_joint"]


def test_blob_round_trip_is_lossless():
    m = load_model("fetch_pick_and_place")
    m2 = Model.from_blob(m.to_blob())
    for f in Model.INT_FIELDS + Model.FLT_FIELDS:
        assert np.array_equal(np.asarray(getattr(m, f)), np.asarray(getattr(m2, f))), f
    assert m.names == m2.names


def test_committed_blobs_match_a_fresh_compile():
    assert sorted(FACTS["blob_sha256"]) == sorted(MODEL_SOURCES)
    for name, digest in FACTS["blob_sha256"].items():
        assert hashlib.sha256(open(os.path.join(MODEL_DIR, name + ".b200m"), "rb").read()).hexdigest() == digest, name


def test_fused_runtime_model_keeps_the_dynamics():
    """Fusing jointless bodies (MuJoCo `fusestatic`) must not change the mass matrix; collision filters follow MuJoCo."""
    from oracle.oracle_sim import OracleSim

    m = load_model("fetch_pick_and_place")
    full = FACTS["fetch_pick_and_place_mjcf"]
    s = OracleSim(m)
    s.forward()
    assert np.abs(s.M - np.array(full["M0"])).max() < 1e-10  # oracle CRB on the fused tree vs dense sum on the MJCF tree
    assert m.nbody == 16 and full["bodies"] == 33  # 33 MJCF bodies (world included) fuse into 16
    geoms = m.names["geom"]
    pairs = {(geoms[a], geoms[b]) for a, b in zip(m.pair_geom1, m.pair_geom2)}
    assert ("robot0:r_gripper_finger_link", "robot0:l_gripper_finger_link") not in pairs  # <exclude>
    assert not any("robot0:gripper_link" in p and "finger" in p[0] + p[1] for p in pairs)  # parent-child filter
    assert ("object0", "robot0:r_gripper_finger_link") in pairs or ("robot0:r_gripper_finger_link", "object0") in pairs


def test_defaults_childclass_euler_fromto(mjcf_file):
    xml = """
    <mujoco><compiler angle="degree"/>
      <default><joint damping="3"/><default class="a"><geom friction="0.7 0.1 0.1" condim="4"/><joint armature="2"/></default></default>
      <worldbody>
        <body name="b1" pos="0 0 1" euler="0 0 90" childclass="a">
          <joint name="j1" type="hinge" axis="0 1 0" range="-90 90" limited="true"/>
          <geom type="capsule" fromto="0 0 0 0 0 0.4" size="0.05"/>
          <body name="b2" pos="0 0 0.4"><joint name="j2" type="slide" axis="1 0 0" class="main"/><geom type="sphere" size="0.1" class="main"/></body>
        </body>
      </worldbody>
    </mujoco>"""
    m = compile_mjcf(mjcf_file(xml))
    assert m.nv == 2 and list(m.dof_damping) == [3, 3] and list(m.dof_armature) == [2, 0]
    assert np.allclose(m.jnt_range[0], [-np.pi / 2, np.pi / 2])
    assert np.allclose(m.body_quat[1], [np.cos(np.pi / 4), 0, 0, np.sin(np.pi / 4)])
    assert np.allclose(m.geom_size[0][:2], [0.05, 0.2]) and np.allclose(m.geom_pos[0], [0, 0, 0.2])
    assert m.pair_condim.size == 0  # both geoms hang off a parent-child pair: filtered


# ----------------------------------------------------------------------------------------------------------------------------
# Closed-form / independently recomputed checks of the compiled constants.  The oracle and the kernels consume the SAME blob, so an
# error in the compiler (inertia from geoms / <inertial>, fusing, invweight0) is common-mode and invisible to the parity tests;
# these tests anchor the constants to numbers taken straight from the XML text and to a second computation path (the C oracle's
# kinematics + mass matrix, finite-difference Jacobians, numpy), not to the compiler's own arithmetic.
def test_fetch_closed_form_totals():
    """Total robot mass, the composite inertia seen by the three base slides, and the gravity load on the torso lift joint of the
    Fetch model: XML numbers against the compiled blob, the oracle (C, fp64) and the kernel emulation (fp32)."""
    from oracle.oracle_sim import OracleSim
    from tests.hostsim import HostSim
    from gymnasium_robotics_b200.fetch import REF_POINT, welded_eq_data

    sub = FACTS["fetch_robot_xml"]["subtree_mass"]
    robot_mass = sub["robot0:base_link"]
    assert robot_mass == pytest.approx(70.1294 + 10.7796 + 2.2556 + 0.9087 + 2.5587 + 2.6615 + 2.3311 + 2.1299 + 1.6563 + 1.725 + 0.1354 + 1.5175 +
                                       4 + 4 + 0.002 + 0.0083 + 13.2775, abs=1e-9)
    m = load_model("fetch_pick_and_place")
    bm = m.names["body_map"]
    robot_rt = sorted({rt for name, rt in bm.items() if name.startswith("robot0:") and name != "robot0:mocap"})
    assert float(np.sum(m.body_mass[robot_rt])) == pytest.approx(robot_mass, rel=1e-12)          # fusing loses no mass
    assert float(m.body_mass[bm["object0"]]) == pytest.approx(2.0, rel=1e-12)                    # pick_and_place.xml:24 mass="2"
    # composite inertia: the three base slides translate the whole robot
    s = OracleSim(m)
    s.forward()
    hs = HostSim(m, eq_data=welded_eq_data(m), ref=REF_POINT)
    hs.qpos[:] = m.qpos0
    hs.forward()
    Mh = hs.dense_M()
    for name in ("robot0:slide0", "robot0:slide1", "robot0:slide2"):
        d = int(m.jnt_dofadr[m.joint_id(name)])
        arm = float(m.dof_armature[d])
        assert s.M[d, d] - arm == pytest.approx(robot_mass, rel=1e-10), name
        assert Mh[d, d] - arm == pytest.approx(robot_mass, rel=2e-6), name
    # gravity load at rest on the vertical torso lift slide = g x (mass of everything it carries)
    d = int(m.jnt_dofadr[m.joint_id("robot0:torso_lift_joint")])
    load = 9.81 * sub["robot0:torso_lift_link"]
    assert abs(float(m.jnt_axis[m.joint_id("robot0:torso_lift_joint")][2])) == 1.0
    assert s.qfrc_bias[d] == pytest.approx(load, rel=1e-9)
    passive_and_act = float(s.qfrc_passive[d] + s.qfrc_actuator[d])
    assert hs.fsmooth[d] == pytest.approx(passive_and_act - load, rel=5e-6)


def test_invweight0_recomputed_along_a_second_path():
    """dof_invweight0 = diag(M^-1) and the weld's body_invweight0 = block averages of J M^-1 J^T at qpos0 -- recomputed from the C
    oracle's mass matrix and finite-difference Jacobians of its kinematics (the compiler uses analytic Jacobians on the unfused
    tree in numpy), plus the free box whose values are closed-form (1/m and the mean of 1/I)."""
    from oracle.oracle_sim import OracleSim

    m = load_model("fetch_pick_and_place")
    s = OracleSim(m)
    s.qpos[:] = m.qpos0
    s.forward()
    Minv = np.linalg.inv(s.M.copy())
    assert np.allclose(np.diag(Minv), m.dof_invweight0, rtol=1e-9)
    # weld robot0:mocap <-> robot0:gripper_link: invweight = that of the gripper link (the mocap body has no dofs)
    site = m.frame_site("robot0:gripper_link")
    ipos = np.array(FACTS["fetch_robot_xml"]["gripper_link_inertial_pos"])

    def com():
        return s.site_xpos[site] + s.site_xmat[site].reshape(3, 3) @ ipos

    nv, eps = m.nv, 1e-6
    Jp = np.zeros((3, nv))
    q0 = np.array(m.qpos0, dtype=np.float64)
    for j in range(m.njnt):
        if int(m.jnt_type[j]) == 0:
            continue        # the object's free joint does not move the gripper
        a, d = int(m.jnt_qposadr[j]), int(m.jnt_dofadr[j])
        s.qpos[:] = q0; s.qpos[a] += eps; s.forward(); hi = com().copy()
        s.qpos[:] = q0; s.qpos[a] -= eps; s.forward(); lo = com().copy()
        Jp[:, d] = (hi - lo) / (2 * eps)
    s.qpos[:] = q0
    s.forward()
    _, Jr = s.jac_site(site)
    A_t, A_r = Jp @ Minv @ Jp.T, Jr @ Minv @ Jr.T
    want = [np.trace(A_t) / 3, np.trace(A_r) / 3]
    assert np.allclose(m.eq_invweight[0], want, rtol=1e-5), (m.eq_invweight[0], want)
    # the free 5 cm box of 2 kg: translational 1/m, rotational mean(1/I) with I = m (a^2 + b^2) / 3 = 2 * 2 * 0.025^2 / 3
    gn = m.names["geom"]
    p = next(k for k, (a, b) in enumerate(zip(m.pair_geom1, m.pair_geom2)) if {gn[a], gn[b]} == {"object0", "table0"} or
             ("object0" in (gn[a], gn[b]) and int(m.geom_body[a]) * int(m.geom_body[b]) == 0))
    I = 2.0 * 2 * 0.025 ** 2 / 3
    assert np.allclose(m.pair_invweight[p], [0.5, 1.0 / I], rtol=1e-9), m.pair_invweight[p]
