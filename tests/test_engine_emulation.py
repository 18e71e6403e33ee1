"""The engine kernel source (csrc/mj_*.cuh) compiled for the host with one lane, checked against the fp64 checker
(oracle/mjengine.c) -- the CPU-side guard for the code the GPU runs.  North-star bar: from identical states and
actions, one-step qpos / qvel within 1e-4 absolute (fp32 engine vs fp64)."""
import os

import numpy as np
import pytest

from earl_benchmark_b200.envs.sawyer_door import MODEL_PATH
from earl_benchmark_b200.mjcf.compile import Model
from host_emulation.emu import Emu, door_task
from oracle.engine import SawyerDoorOracle

TOL = 1e-4


@pytest.fixture(scope="module")
def door():
    m = Model.load(MODEL_PATH)
    return m, SawyerDoorOracle(m), Emu(m, door_task(m))


def test_mass_matrix_bias_and_kinematics_match(door):
    m, o, em = door
    rs = np.random.RandomState(0)
    for _ in range(8):
        q = m.qpos0 + rs.uniform(-1, 1, int(m.nq)) * np.array([1.0] * 7 + [0.02, 0.02, 0.7])
        q[1] -= 1.5
        v = rs.uniform(-2, 2, int(m.nv))
        o.e.reset()
        o.e.qpos[:], o.e.qvel[:] = q, v
        M_ref, b_ref = o.e.mass_matrix(), o.e.bias()
        x_ref = o.e.arr("xpos", (24, 3))[:int(m.nbody)].copy()
        em.set_state(q, v, np.zeros(int(m.nv)), [0, 0.4, 0.2])
        M, b, x = em.forward_parts()
        assert np.abs(M - M_ref).max() <= 1e-6 * np.abs(M_ref).max()
        assert np.abs(b - b_ref).max() <= 2e-6 * max(1.0, np.abs(b_ref).max())
        assert np.abs(x - x_ref).max() <= 1e-6


def test_one_env_step_parity_along_the_reset_transient(door):
    """sim.reset() + _reset_hand(): 50 x 5 substeps with joint limits active and the weld pulling the arm 1 m;
    before every env step the emulated engine is re-synchronised to the checker's state (one-step test)."""
    m, o, em = door
    e = o.e
    e.reset()
    nv = int(m.nv)
    worst_q = worst_v = 0.0
    for it in range(50):
        e.mocap_pos[:], e.mocap_quat[:], e.ctrl[:] = o.HAND_INIT, [1, 0, 1, 0], [-1, 1]
        em.set_state(e.qpos, e.qvel, e.arr("qacc_warmstart", (32,))[:nv], o.HAND_INIT, ctrl=(-1, 1))
        e.step(5)
        em.substeps(5)
        q, v, _, _ = em.get_state()
        worst_q, worst_v = max(worst_q, np.abs(q - e.qpos).max()), max(worst_v, np.abs(v - e.qvel).max())
        assert em.info("bad") == 0
        assert em.info("iter") <= 6          # Newton converges in a handful of iterations in fp32 too
    assert worst_q < TOL and worst_v < TOL, (worst_q, worst_v)


def test_open_loop_rollout_tracks_the_checker(door):
    """250 settle substeps + 60 random-action env steps without any re-synchronisation."""
    m, o, em = door
    e = o.e
    e.reset()
    em.set_state(e.qpos, e.qvel, np.zeros(int(m.nv)), o.HAND_INIT, ctrl=(-1, 1))
    for _ in range(50):
        e.mocap_pos[:], e.mocap_quat[:], e.ctrl[:] = o.HAND_INIT, [1, 0, 1, 0], [-1, 1]
        e.step(5)
        em.substeps(5)
    q, v, w, _ = em.get_state()
    assert np.abs(q - e.qpos).max() < TOL and np.abs(v - e.qvel).max() < TOL
    e.qpos[o.door_qadr], e.qvel[o.door_qadr] = -1.0, 0.0
    q[o.door_qadr], v[o.door_qadr] = -1.0, 0.0
    em.set_state(q, v, w, o.HAND_INIT)
    rs = np.random.RandomState(1)
    for _ in range(60):
        a = rs.uniform(-1, 1, 4).astype(np.float32)
        ob_ref, _ = o.step(a)
        ob = em.env_step(a)
        assert np.abs(ob_ref[:7] - ob).max() < 5e-5
    q, v, _, mp = em.get_state()
    assert np.abs(q - e.qpos).max() < TOL and np.abs(v - e.qvel).max() < TOL
    assert np.abs(mp - e.mocap_pos).max() < 1e-7


def _door_angle(handle_xy):
    """Inverse of the handle forward kinematics (SURVEY.md Appendix E.2)."""
    p0, hinge = np.array([0.375721629, -0.107139896]), np.array([-0.085, 0.85])
    return np.arctan2(handle_xy[1] - hinge[1], handle_xy[0] - hinge[0]) - np.arctan2(p0[1], p0[0])


def test_contact_rich_demo_replay_one_step_parity(door):
    """First shipped forward demonstration (the hand pushes the door shut against 1.7 kN of door-on-table friction,
    up to 10 contacts / 43 constraint rows): before every env step the emulated fp32 engine is re-synchronised to the
    checker, then both step.  Same contact and row counts on (nearly) every step; one-step qpos within 1e-5
    everywhere; one-step qvel within 1e-4 while the contacts are light and within 5e-3 under kN contact forces,
    where fp32 positions times kN forces on gram-scale wrist inertias set the floor."""
    from earl_benchmark_b200 import demos
    m, o, em = door
    e, nv = o.e, int(m.nv)
    demo = demos.load("sawyer_door", "forward")
    obs, act = demo["observations"], demo["actions"]
    o.reset(door_angle=_door_angle(obs[0][4:6]))
    same = light_ok = 0
    worst_q = worst_v = 0.0
    steps = 78
    for t in range(steps):
        em.set_state(e.qpos, e.qvel, e.arr("qacc_warmstart", (32,))[:nv], e.mocap_pos)
        ob_ref, _ = o.step(act[t])
        ob = em.env_step(act[t])
        q, v, _, _ = em.get_state()
        dq, dv = np.abs(q - e.qpos).max(), np.abs(v - e.qvel).max()
        worst_q, worst_v = max(worst_q, dq), max(worst_v, dv)
        same += int(e.ncon == em.info("ncon") and e.nefc == em.info("nefc"))
        if e.ncon <= 4:
            light_ok += int(dv < 1e-4)
        assert np.abs(ob_ref[:7] - ob).max() < 1e-4
        assert em.info("bad") == 0
    assert same >= steps - 2
    assert worst_q < 3e-5 and worst_v < 5e-3, (worst_q, worst_v)  # north-star bar: 1e-4
    assert light_ok >= 15


# ------------------------------------------------------------------------------------------------ sawyer_peg scene
@pytest.fixture(scope="module")
def peg():
    from earl_benchmark_b200.envs.sawyer_peg import MODEL_PATH as PEG_MODEL
    from host_emulation.emu import peg_task
    from oracle.engine import SawyerPegOracle
    m = Model.load(PEG_MODEL)
    return m, SawyerPegOracle(m), Emu(m, peg_task(m))


def test_peg_scene_one_step_parity(peg):
    """Free-joint peg (nq 16, nv 15): sim.reset() + _reset_hand() (the peg drops 1.5 cm onto the table: 4 box-box
    contacts) and 80 env steps of the hand pressing down on the peg (up to 12 contacts, condim-4 pads), re-synchronised
    before every env step.  Only box-box contacts occur, so fp32 stays within 1e-4 everywhere."""
    m, o, em = peg
    e, nv = o.e, int(m.nv)
    e.reset()
    worst_q = worst_v = 0.0
    for _ in range(50):
        e.mocap_pos[:], e.mocap_quat[:], e.ctrl[:] = o.HAND_INIT, [1, 0, 1, 0], [-1, 1]
        em.set_state(e.qpos, e.qvel, e.arr("qacc_warmstart", (32,))[:nv], o.HAND_INIT, ctrl=(-1, 1))
        e.step(5)
        em.substeps(5)
        q, v, _, _ = em.get_state()
        worst_q, worst_v = max(worst_q, np.abs(q - e.qpos).max()), max(worst_v, np.abs(v - e.qvel).max())
    assert e.ncon == 4 and em.info("ncon") == 4
    o.reset(peg_pos=[0.05, 0.6, 0.02])
    rs = np.random.RandomState(0)
    max_con = 0
    for _ in range(80):
        a = np.clip(rs.uniform(-1, 1, 4) + [0, 0, -0.6, 0], -1, 1).astype(np.float32)
        em.set_state(e.qpos, e.qvel, e.arr("qacc_warmstart", (32,))[:nv], e.mocap_pos)
        ob_ref, _ = o.step(a)
        ob = em.env_step(a)
        q, v, _, _ = em.get_state()
        worst_q, worst_v = max(worst_q, np.abs(q - e.qpos).max()), max(worst_v, np.abs(v - e.qvel).max())
        assert e.ncon == em.info("ncon") and e.nefc == em.info("nefc")
        assert np.abs(ob_ref[:7] - ob).max() < 1e-5 and em.info("bad") == 0
        max_con = max(max_con, e.ncon)
    assert max_con >= 10
    assert worst_q < TOL and worst_v < TOL, (worst_q, worst_v)


def test_device_harness_compiles_for_every_capacity_set(tmp_path):
    """The 32-lane twin of this file's one-lane build (tests/host_emulation/devemul.cu, run on the GPU by
    test_engine_device_phases_gpu.py) cross-compiles for sm_100a with the product's engine flags in all four capacity
    sets: door / peg primary and extra-large, kitchen primary and extra-large.  No GPU needed."""
    from host_emulation.emu import CAPSETS, build_device
    for so in build_device(tuple(CAPSETS), out_dir=str(tmp_path)):
        assert os.path.getsize(so) > 0
