"""Each lane-parallel phase of the warp-per-env engine (csrc/mj_engine.cuh, mj_collide.cuh, mj_step.cuh) ON THE B200,
stopped after the phase and read back (tests/host_emulation/devemul.cu: the engine source with NL = 32 and the product's
engine flags), against the fp64 checker (oracle/engine.py) or the one-lane host build of the same source on identical
inputs.  The end-to-end step tests compare whole steps with bars loose enough to hide a lane-indexing or reduction error
that moves a minority of states by 1e-3 or drops a row now and then; these checks pin the pieces that exist only in the
32-lane build: the ballot-compacted joint-limit rows, the ballot / popc hit and candidate lists, the lane-parallel hull
argmax, the shuffle Cholesky (`spd_solve_reg`), the warp reductions of the line search, and the lane-strided loops over
more than 32 rows / Hessian pairs.

State sets (inputs rounded to fp32, so that every build starts from the same numbers): door -- random-action checker
rollouts and the shipped forward / reverse demonstrations (gripper on the handle: portal-refinement contacts); peg -- the
press-down states of test_engine_emulation.test_peg_scene_one_step_parity; kitchen -- the scripted reach into the cabinets
of test_kitchen_engine_gpu.py and states with every limited joint pushed outside its range."""
import numpy as np
import pytest

from earl_benchmark_b200.mjcf.compile import Model
from host_emulation import emu as E
from oracle.engine import Engine

pytestmark = pytest.mark.gpu

LIMIT_BAD = 8   # Work::bad bit 3: constraint rows beyond the capacity set were dropped
HIT_BAD = 2     # Work::bad bit 1: candidate pairs beyond MAXHIT were dropped
CON_BAD = 4     # Work::bad bit 2: contacts beyond MAXCON were dropped


@pytest.fixture(scope="module", autouse=True)
def _harness():
    E.build_device()   # the four capacity sets in parallel


# ------------------------------------------------------------------------------------------------ state sets
def _f32(a):
    return np.asarray(a, np.float64).astype(np.float32).astype(np.float64)


def _snap(e, nv, out):
    out.append(dict(qpos=_f32(e.qpos), qvel=_f32(e.qvel), warm=_f32(e.arr("qacc_warmstart", (32,))[:nv]), mocap_pos=e.mocap_pos.copy(),
                    mocap_quat=_f32(e.mocap_quat), ctrl=_f32(e.ctrl)))


def _door_states():
    from earl_benchmark_b200 import demos
    from earl_benchmark_b200.envs import sawyer_door
    from oracle.engine import SawyerDoorOracle
    from test_engine_oracle import door_angle
    m = Model.load(sawyer_door.MODEL_PATH)
    o = SawyerDoorOracle(m)
    e, nv, out = o.e, int(m.nv), []
    rs = np.random.RandomState(3)
    for _ in range(4):                                   # random-action rollouts from the reset pose
        o.reset(door_angle=-np.pi / 3 + rs.uniform(0, np.pi / 20))
        bias = rs.uniform(-0.5, 0.5, 4)
        for t in range(40):
            o.step(np.clip(bias + rs.uniform(-1, 1, 4), -1, 1))
            if t % 2 == 1:
                _snap(e, nv, out)
    for which in ("forward", "reverse"):                 # the shipped demonstrations: the gripper pushes / pulls the handle
        d = demos.load("sawyer_door", which)
        ends = list(np.nonzero(d["terminals"].ravel())[0] + 1)
        for s, en in zip([0] + ends[:-1], ends):
            o.goal = d["observations"][s][7:14].astype(np.float64)
            o.reset(door_angle=door_angle(d["observations"][s][4:6]))
            for t, a in enumerate(d["actions"][s:en]):
                o.step(a)
                if t % 5 == 2:
                    _snap(e, nv, out)
    return m, out


def _peg_states():
    from earl_benchmark_b200.envs.sawyer_peg import MODEL_PATH
    from oracle.engine import SawyerPegOracle
    m = Model.load(MODEL_PATH)
    o = SawyerPegOracle(m)
    e, nv, out = o.e, int(m.nv), []
    e.reset()
    for _ in range(50):                                  # _reset_hand: the peg drops onto the table
        e.mocap_pos[:], e.mocap_quat[:], e.ctrl[:] = o.HAND_INIT, [1, 0, 1, 0], [-1, 1]
        e.step(5)
    o.reset(peg_pos=[0.05, 0.6, 0.02])
    rs = np.random.RandomState(0)
    for _ in range(80):                                  # the hand presses down on the peg: up to 12 contacts
        a = np.clip(rs.uniform(-1, 1, 4) + [0, 0, -0.6, 0], -1, 1)
        e.mocap_pos[:] = np.clip(e.mocap_pos + a[:3] * o.ACTION_SCALE, o.MOCAP_LOW, o.MOCAP_HIGH)
        e.mocap_quat[:], e.ctrl[:] = [1, 0, 1, 0], [a[3], -a[3]]
        for s in range(5):
            if s % 2 == 0:
                _snap(e, nv, out)
            e.step(1)
    return m, out


def _kitchen_states():
    from earl_benchmark_b200.kitchen_engine import MODEL_PATH
    from oracle import kitchen_logic as KL
    from oracle.engine import KitchenOracle
    m = Model.load(MODEL_PATH)
    k = KitchenOracle(m)
    k.seed(3)
    np.random.seed(2)
    k.reset()
    e, nv, out = k.e, int(m.nv), []
    target = e.site_xpos("slide_site").copy()
    for t in range(100):
        d = target - e.site_xpos("end_effector") if t < 70 else np.array([0.5, 0.0, 0.0])
        a = np.zeros(9)
        a[:3] = np.clip(d * 10, -1, 1) * 0.5
        mocap, ctrl = k.logic.control(a, e.mocap_pos.copy())
        e.mocap_pos[:], e.ctrl[:] = mocap, ctrl
        for s in range(KL.FRAME_SKIP):
            if s % 20 == 0:
                _snap(e, nv, out)
            e.step(1)
        k.logic.observe(e.qpos)
    return m, out


def _limit_states(m, base, count, seed):
    """`count` states of `base` with EVERY limited hinge / slide joint pushed 1 mrad .. 0.1 rad (or mm) outside one end
    of its range: one active limit row per joint, candidates in both ballot passes of make_constraints."""
    rs = np.random.RandomState(seed)
    out = []
    for i in range(count):
        s = dict(base[rs.randint(len(base))])
        q = s["qpos"].copy()
        for j in range(len(m.jnt_type)):
            if m.jnt_limited[j] and m.jnt_type[j] >= 2:
                lo, hi = m.jnt_range[j]
                over = rs.uniform(1e-3, 0.1)
                q[m.jnt_qposadr[j]] = lo - over if rs.rand() < 0.5 else hi + over
        s["qpos"] = _f32(q)
        out.append(s)
    return out


_CACHE = {}


def states(name):
    if name not in _CACHE:
        _CACHE[name] = {"door": _door_states, "peg": _peg_states, "kitchen": _kitchen_states}[name]()
    return _CACHE[name]


def task(name, m):
    return {"door": E.door_task, "peg": E.peg_task, "kitchen": E.kitchen_task}[name](m)


def stack(S, key):
    return np.stack([s[key] for s in S])


def device(name, m, S, capset):
    d = E.DevEmu(m, task(name, m), capset=capset, batch=len(S))
    d.set_states(stack(S, "qpos"), stack(S, "qvel"), stack(S, "warm"), stack(S, "mocap_pos"), stack(S, "mocap_quat"), stack(S, "ctrl"))
    return d


def host_run(em, s, stage, nsub=1):
    em.set_state(s["qpos"], s["qvel"], s["warm"], s["mocap_pos"], mocap_quat=s["mocap_quat"], ctrl=s["ctrl"])
    em.run(stage, nsub)
    return em


def checker(e, s, qpos=None):
    e.reset()
    e.qpos[:] = s["qpos"] if qpos is None else qpos
    e.qvel[:], e.mocap_pos[:], e.mocap_quat[:], e.ctrl[:] = s["qvel"], s["mocap_pos"], s["mocap_quat"], s["ctrl"]
    e.arr("qacc_warmstart", (32,))[:e.nv] = s["warm"]
    e.forward()
    return e


def checker_geoms(e):
    from oracle.engine import lib
    return [divmod(lib().mje_con_geoms(e.d, k), 1000) for k in range(e.ncon)]


def checker_flips(e, s, rs, trials=12):
    """True when the checker's own contact set changes under a 1e-7 perturbation of qpos (a contact at its activation
    margin, a portal-refinement branch): such a state has no single right answer at fp32 resolution."""
    g0 = checker_geoms(checker(e, s))
    for _ in range(trials):
        if checker_geoms(checker(e, s, s["qpos"] + rs.choice([-1e-7, 1e-7], len(s["qpos"])))) != g0:
            return True
    return False


def host_hits_flip(em, s, rs, trials=12):
    h0 = host_run(em, s, "collide").hits().tolist()
    for _ in range(trials):
        p = dict(s, qpos=s["qpos"] + rs.choice([-1e-7, 1e-7], len(s["qpos"])))
        if host_run(em, p, "collide").hits().tolist() != h0:
            return True
    return False


MODELS = ["door", "peg", "kitchen"]
PRIMARY = {"door": "small", "peg": "small", "kitchen": "kitchen"}
XL = {"door": "xl", "peg": "xl", "kitchen": "kitchen_xl"}


# ------------------------------------------------------------------------------------------------ forward parts
@pytest.mark.parametrize("name", MODELS)
def test_forward_parts_match_checker(name):
    """Kinematics, mass matrix (composite rigid body, lane per dof) and bias forces (RNE, lane per body / dof) against
    the checker: the one-lane bars of test_engine_emulation (xpos 1e-6, M 1e-6 of its largest entry, bias 2e-6)."""
    m, S = states(name)
    d = device(name, m, S, PRIMARY[name])
    d.run("forward_parts")
    e, nb = Engine(m), int(m.nbody)
    worst = dict(x=0.0, R=0.0, M=0.0, b=0.0)
    for i, s in enumerate(S):
        x, R, M, b = d.forward(i)
        checker(e, s)
        M_ref, b_ref = e.mass_matrix(), e.bias()
        worst["x"] = max(worst["x"], np.abs(x - e.arr("xpos", (24, 3))[:nb]).max())
        worst["R"] = max(worst["R"], np.abs(R - e.arr("xmat", (24, 9))[:nb]).max())
        worst["M"] = max(worst["M"], np.abs(M - M_ref).max() / np.abs(M_ref).max())
        worst["b"] = max(worst["b"], np.abs(b - b_ref).max() / max(1.0, np.abs(b_ref).max()))
    print(f"{name} forward parts, {len(S)} states, device vs checker:", {k: f"{v:.2e}" for k, v in worst.items()})
    assert worst["x"] <= 1e-6 and worst["R"] <= 1e-6 and worst["M"] <= 1e-6 and worst["b"] <= 2e-6, worst


# ------------------------------------------------------------------------------------------------ collision
@pytest.mark.parametrize("name", MODELS)
def test_collision_matches_host_build_and_checker(name):
    """Broad-phase hit list (ballot / popc compaction; kitchen: through the cached candidate list) equal to the one-lane
    build's, contact count and geom pairs equal to both the one-lane build's and the checker's, contact distance /
    position / normal close to the checker's.  A state is excused only if the reference it disagrees with flips by
    itself under a 1e-7 perturbation of qpos."""
    m, S = states(name)
    d = device(name, m, S, PRIMARY[name])
    d.run("collide")
    em, e = E.Emu(m, task(name, m), capset=PRIMARY[name]), Engine(m)
    rs = np.random.RandomState(1)
    excused_hits, excused_con, nconv, maxcon = [], [], 0, 0
    worst = dict(dist=0.0, pos=0.0, normal=0.0)
    for i, s in enumerate(S):
        assert d.info(i)["bad"] == 0
        hits = d.hits(i).tolist()
        dist, pos, frame, geoms = d.contacts(i)
        host_run(em, s, "collide")
        if hits != em.hits().tolist():
            assert host_hits_flip(em, s, rs), (i, hits, em.hits().tolist())
            excused_hits.append(i)
        hd, hp, hf, hg = em.contacts()
        ref_geoms = checker_geoms(checker(e, s))
        same_host = np.array_equal(geoms, hg)
        same_ref = [tuple(sorted(g)) for g in geoms.tolist()] == [tuple(sorted(g)) for g in ref_geoms]
        if not (same_host and same_ref):
            assert checker_flips(e, s, rs), (i, geoms.tolist(), hg.tolist(), ref_geoms)
            excused_con.append(i)
            continue
        checker(e, s)
        nc = len(dist)
        maxcon = max(maxcon, nc)
        nconv += int(any(m.geom_hullnum[g] > 0 for g in geoms.ravel()))
        if nc:
            worst["dist"] = max(worst["dist"], np.abs(dist - e.arr("con_dist", (64,))[:nc]).max())
            worst["pos"] = max(worst["pos"], np.abs(pos - e.arr("con_pos", (64, 3))[:nc]).max())
            worst["normal"] = max(worst["normal"], np.abs(frame[:, :3] - e.arr("con_frame", (64, 9))[:nc, :3]).max())
    print(f"{name} collision, {len(S)} states ({nconv} with mesh contacts, up to {maxcon} contacts): device vs checker",
          {k: f"{v:.2e}" for k, v in worst.items()}, "excused (hits, contacts):", excused_hits, excused_con)
    assert len(excused_con) <= len(S) // 10
    assert maxcon >= {"door": 6, "peg": 10, "kitchen": 8}[name]
    if name == "door":
        assert nconv >= 20          # the gripper on the handle: portal refinement over the mesh hulls
    # normals: the door's pad-on-handle contacts come out of portal refinement, whose result moves with the last bits of
    # the fp32 poses near a degenerate portal (the one-lane build: 3.3e-4 from the checker on the same states)
    assert worst["dist"] < 2e-6 and worst["pos"] < 5e-6 and worst["normal"] < 1e-3, worst


# ------------------------------------------------------------------------------------------------ constraint rows
def _row_errors(a, b, n):
    """Differences of the first n rows: J and aref against the largest entry of the state, R and D relative per row, pos
    against max(0.1, largest |pos|) -- fp32 rounding of the inputs (positions, contact frames from portal refinement) is
    what separates the two builds, and a misplaced or dropped row differs by O(1) on these scales."""
    if n == 0:
        return dict(J=0.0, aref=0.0, RD=0.0, pos=0.0)
    x = {k: a[k][:n] for k in ("J", "aref", "R", "D", "pos")}
    y = {k: b[k][:n] for k in ("J", "aref", "R", "D", "pos")}
    rel = lambda k: (np.abs(x[k] - y[k]) / np.abs(y[k])).max()  # noqa: E731
    return dict(J=np.abs(x["J"] - y["J"]).max() / max(1e-30, np.abs(y["J"]).max()),
                aref=np.abs(x["aref"] - y["aref"]).max() / max(1e-30, np.abs(y["aref"]).max()),
                RD=max(rel("R"), rel("D")), pos=np.abs(x["pos"] - y["pos"]).max() / max(0.1, np.abs(y["pos"]).max()))


# measured on the B200 against the one-lane build (max over the state set, scales of _row_errors): J 3.5e-4 / 4.8e-7 /
# 4.2e-7, aref 4.7e-4 / 5.5e-5 / 1.3e-5, R and D 5.3e-5 / 5.4e-6 / 5.2e-5, pos 2.6e-6 / 3.0e-6 / 2.4e-7 (door / peg /
# kitchen).  The door's largest ones are contact rows of the pads on the handle, whose frames come out of portal
# refinement (normals 3e-4 apart between the builds, as between the one-lane build and the checker); aref carries the
# weld / contact stiffness times the fp32 rounding of a position.
ROW_TOL = dict(J=1e-3, aref=1e-3, RD=5e-4, pos=1e-5)
# rows that do not come from a contact (weld, equality, friction loss, joint limits), all-joints-at-limit states, B200: J
# 1.8e-9, aref 1.9e-7, R and D bit-equal, pos 1.2e-7
NONCONTACT_TOL = dict(J=1e-6, aref=1e-5, RD=1e-6, pos=1e-5)


def _compare_rows(name, m, S, capset, host_capset, noncontact_only=False):
    """Device rows of capacity set `capset` against the one-lane build of `host_capset` on the same states: row count,
    row types and contact-to-row map equal; values within the returned worst differences (_row_errors)."""
    d = device(name, m, S, capset)
    d.run("constraints")
    em = E.Emu(m, task(name, m), capset=host_capset)
    cap_dev = d.L.caps["MAXEFC"]
    worst, nrows, overflow, skipped = dict(J=0.0, aref=0.0, RD=0.0, pos=0.0), [], 0, 0
    for i, s in enumerate(S):
        host_run(em, s, "constraints")
        gd, gh = d.contacts(i)[3], em.contacts()[3]
        # contact_rows keeps the contacts whose rows fit: a device set with fewer rows keeps a prefix of the host's contacts
        if not np.array_equal(gd, gh[:len(gd)]):
            skipped += 1        # a contact at its margin (test_collision_matches_host_build_and_checker)
            continue
        a, b = d.rows(i), em.rows()
        hb, db = em.info()["bad"], d.info(i)["bad"]
        # contacts beyond MAXCON (same in both builds of a set) are dropped alike; nothing else may be flagged
        assert hb & ~(LIMIT_BAD | CON_BAD) == 0 and db & ~(LIMIT_BAD | CON_BAD) == 0 and hb & CON_BAD == db & CON_BAD, (i, hb, db)
        n = len(a["type"])
        if len(b["type"]) > cap_dev or hb & LIMIT_BAD:
            # more rows than the device set holds: dropped there and flagged, the rows kept are the host's first ones
            assert db & LIMIT_BAD and n <= cap_dev, (i, n, len(b["type"]))
            overflow += 1
        else:
            assert db == hb and n == len(b["type"]), (i, n, len(b["type"]))
            assert np.array_equal(a["con_row"], b["con_row"]) and np.array_equal(a["con_dim"], b["con_dim"])
        assert np.array_equal(a["type"], b["type"][:n]), i
        if noncontact_only and len(a["con_row"]):
            n = int(a["con_row"][0])
        for k, v in _row_errors(a, b, n).items():
            worst[k] = max(worst[k], v)
        nrows.append(len(b["type"]))
    return worst, np.array(nrows), overflow, skipped, cap_dev


@pytest.mark.parametrize("name", MODELS)
def test_constraint_rows_match_host_build(name):
    """make_constraints (weld, joint equality, friction loss, ballot-compacted joint limits) + contact_rows against the
    one-lane build on identical inputs: same row count and row types, J / aref / R / D to fp32 rounding."""
    m, S = states(name)
    worst, nrows, overflow, skipped, _ = _compare_rows(name, m, S, PRIMARY[name], PRIMARY[name])
    print(f"{name} constraint rows, {len(S)} states (rows {nrows.min()}..{nrows.max()}, {skipped} skipped, {overflow} beyond "
          f"the primary set): max differences", {k: f"{v:.2e}" for k, v in worst.items()})
    assert all(worst[k] <= ROW_TOL[k] for k in ROW_TOL), worst
    assert skipped <= len(S) // 20 and nrows.max() > 32


def test_kitchen_rows_with_every_joint_beyond_its_limit():
    """Every one of the kitchen's 23 limited joints outside its range: 46 limit candidates, so the ballot of
    make_constraints takes a second pass (base 32) with active lanes; rows beyond 32 and 64, and (with the contacts the
    folded arm makes) beyond the 112 of the primary set, where the primary set drops rows and sets bit 3 and the
    extra-large set (544 rows) keeps them all.  Row structure is compared everywhere; values on the rows before the
    contacts (the contacts of these folded poses are deep portal-refinement penetrations)."""
    m, S = states("kitchen")
    L = _limit_states(m, S, 96, seed=5)
    w1, n1, over1, sk1, cap1 = _compare_rows("kitchen", m, L, "kitchen", "kitchen", noncontact_only=True)
    w2, n2, over2, sk2, _ = _compare_rows("kitchen", m, L, "kitchen_xl", "kitchen_xl", noncontact_only=True)
    print(f"kitchen, every joint beyond its limit ({len(L)} states): rows {n2.min()}..{n2.max()}; primary set {over1} "
          f"overflowing; skipped {sk1} / {sk2}; max differences of the rows before the contacts",
          {k: f"{max(w1[k], w2[k]):.2e}" for k in w1})
    assert all(w1[k] <= NONCONTACT_TOL[k] and w2[k] <= NONCONTACT_TOL[k] for k in NONCONTACT_TOL), (w1, w2)
    assert over2 == 0 and n2.min() > 32 + 6 + 5 and (n2 > 64).sum() >= 5
    assert sk1 <= len(L) // 10 and sk2 <= len(L) // 10
    assert over1 == int((n2 > cap1).sum()) and over1 >= 1, (over1, n2.max())


# ------------------------------------------------------------------------------------------------ solve
def _row_forces(r, jar):
    """Force of every row at jar = J a - aref (fp64): the gradient of the row costs of the primal problem."""
    f = np.zeros_like(jar)
    t, D, R, pos = r["type"], r["D"], r["R"], r["pos"]
    for k in range(len(jar)):
        if t[k] == 0:
            f[k] = -D[k] * jar[k]
        elif t[k] == 1:
            f[k] = -D[k] * jar[k] if jar[k] < 0 else 0.0
        elif t[k] == 4:
            f[k] = np.clip(-D[k] * jar[k], -pos[k], pos[k])
    for c, (r0, dim) in enumerate(zip(r["con_row"], r["con_dim"])):
        if dim <= 0:
            continue
        mu, fri = r["mu"][c], r["fri"][c]
        U = np.concatenate([[jar[r0] * mu], jar[r0 + 1:r0 + dim] * fri[:dim - 1]])
        N, T = U[0], np.sqrt((U[1:] ** 2).sum())
        if N >= mu * T or (T <= 0 and N >= 0):
            f[r0:r0 + dim] = 0
        elif mu * N + T <= 0 or (T <= 0 and N < 0):
            f[r0:r0 + dim] = -D[r0:r0 + dim] * jar[r0:r0 + dim]
        else:
            Dm = D[r0] / (mu * mu * (1 + mu * mu))
            f0 = -Dm * (N - mu * T) * mu
            f[r0] = f0
            f[r0 + 1:r0 + dim] = -f0 / T * U[1:] * fri[:dim - 1]
    return f


@pytest.mark.parametrize("name", MODELS)
def test_solve_satisfies_the_optimality_conditions(name):
    """The Newton solve (Hessian over nv(nv+1)/2 lane-strided pairs, shuffle Cholesky, line search on warp sums) checked
    without trusting any other solver: from the device's own M, J, aref, R, D and qfrc_smooth, recomputed in fp64, the
    returned acceleration a and row forces f satisfy the optimality conditions of the primal problem --
      stationarity  M a - qfrc_smooth = J' f(a)   relative residual (per dof, against |M||a| + |qfrc_smooth| + |J'||f|),
      each row's force = the force of its type and zone at jar = J a - aref (relative to the largest force).
    Against the checker's qacc / qfrc_constraint where the two have the same contacts and rows."""
    m, S = states(name)
    capset = XL[name]       # every state solved with all its rows (the primary kitchen set flags a few)
    d = device(name, m, S, capset)
    d.run("solve")
    e = Engine(m)
    stat, force_err, acc_err, fc_err, iters, compared = [], [], [], [], [], 0
    for i, s in enumerate(S):
        inf = d.info(i)
        assert inf["bad"] == 0, (i, inf)
        _, _, M, _ = d.forward(i)
        r, out = d.rows(i), d.solved(i)
        a, f = out["acc"], out["force"]
        jar = r["J"] @ a - r["aref"]
        f_ref = _row_forces(r, jar)
        res = M @ a - out["smooth"] - r["J"].T @ f_ref
        scale = np.abs(M) @ np.abs(a) + np.abs(out["smooth"]) + np.abs(r["J"].T) @ np.abs(f_ref)
        scale += 1e-6 * scale.max()     # a free body at rest has dofs with nothing acting on them
        stat.append((np.abs(res) / scale).max())
        force_err.append(np.abs(f - f_ref).max() / max(1e-6, np.abs(f_ref).max()) if len(f) else 0.0)
        assert np.abs(out["fcon"] - r["J"].T @ f).max() <= 1e-5 * max(1.0, (np.abs(r["J"].T) @ np.abs(f)).max())
        iters.append(inf["iter"])
        checker(e, s)
        if e.ncon == inf["ncon"] and e.nefc == inf["nefc"]:
            compared += 1
            acc_err.append(np.abs(a - e.qacc).max() / (1.0 + np.abs(e.qacc).max()))
            qfc = e.arr("qfrc_constraint", (32,))[:e.nv]
            fc_err.append(np.abs(out["fcon"] - qfc).max() / (1.0 + np.abs(qfc).max()))
    stat, force_err, acc_err, fc_err = map(np.array, (stat, force_err, acc_err, fc_err))
    print(f"{name} solve, {len(S)} states (Newton iterations {min(iters)}..{max(iters)}): stationarity residual max "
          f"{stat.max():.2e} p99 {np.percentile(stat, 99):.2e}, row force max {force_err.max():.2e}; vs checker on {compared}: "
          f"qacc max {acc_err.max():.2e} median {np.median(acc_err):.2e}, qfrc_constraint max {fc_err.max():.2e}")
    assert stat.max() < SOLVE_TOL[name]["stat"] and force_err.max() < SOLVE_TOL[name]["force"]
    assert compared >= len(S) * 0.8
    assert np.median(acc_err) < SOLVE_TOL[name]["acc_median"] and acc_err.max() < SOLVE_TOL[name]["acc_max"]
    assert fc_err.max() < SOLVE_TOL[name]["acc_max"]


# measured on the B200 (max over the set): stationarity 2.1e-5 / 2.5e-5 / 2.4e-5, row force 2.2e-7 / 4.5e-6 / 2.0e-7,
# qacc vs checker max 3.8e-4 / 9.2e-5 / 1.2e-3, median 1.1e-5 / 7.1e-6 / 4.6e-5 (door / peg / kitchen); the one-lane build
# on the same states: stationarity 6.0e-5 / 1.3e-4 / 4.3e-5 -- the Newton iteration stops at its fp32 step floor
SOLVE_TOL = {
    "door": dict(stat=1e-3, force=1e-4, acc_median=2e-4, acc_max=5e-3),
    "peg": dict(stat=1e-3, force=1e-4, acc_median=2e-4, acc_max=5e-3),
    "kitchen": dict(stat=1e-3, force=1e-4, acc_median=2e-4, acc_max=5e-3),
}


# ------------------------------------------------------------------------------------------------ spd_solve
def _spd(n, cond, rs):
    Q, _ = np.linalg.qr(rs.standard_normal((n, n)))
    ev = np.logspace(0, -np.log10(cond), n) if n > 1 else np.ones(1)
    return (Q * rs.permutation(ev)) @ Q.T * rs.uniform(0.1, 100)


@pytest.mark.parametrize("capset", ["small", "kitchen"])
def test_spd_solve_backward_error_pivots_and_untouched_entries(capset):
    """spd_solve<32> (register / shuffle Cholesky with rsqrtf) for n = 1 .. MAXV and condition numbers 1 .. 1e6 against
    numpy in fp64: backward error |A x - b| <= 4 n eps |A| |x| (2-norms, eps = 2^-24; measured on the B200: 2.25 n eps);
    forward error within 4 n eps cond(A); a zero or negative pivot returns 0
    exactly where the one-lane build's chol_factor does; nothing outside the n x n block and the first n entries of x
    is written."""
    L = E.dev_lib(capset)
    maxv, ldm = L.caps["MAXV"], L.caps["LDM"]
    rs = np.random.RandomState(7)
    ns, As, xs = [], [], []
    for n in range(1, maxv + 1):
        for cond in (1.0, 1e2, 1e4, 1e6):
            A = np.full((maxv, ldm), 7.0, np.float32)
            A[:n, :n] = _spd(n, cond, rs)
            x = np.full(maxv, -3.0, np.float32)
            x[:n] = rs.standard_normal(n)
            ns.append(n), As.append(A), xs.append(x)
    n_good = len(ns)
    for n in range(2, maxv + 1):                 # a zero pivot at k, a negative one at k
        for kind in ("zero", "negative"):
            k = rs.randint(n)
            A = np.full((maxv, ldm), 7.0, np.float32)
            A[:n, :n] = _spd(n, 10.0, rs)
            A[k, :n] = A[:n, k] = 0
            A[k, k] = 0.0 if kind == "zero" else -1.0
            x = np.full(maxv, -3.0, np.float32)
            x[:n] = rs.standard_normal(n)
            ns.append(n), As.append(A), xs.append(x)
    A0, x0 = np.stack(As), np.stack(xs)
    A1, x1 = A0.copy(), x0.copy()
    ok = E.spd_solve_device(ns, A1, x1, capset=capset)
    eps = 2.0 ** -24
    worst = 0.0
    for c, n in enumerate(ns):
        outside = np.ones((maxv, ldm), bool)
        outside[:n, :n] = False
        assert np.array_equal(A1[c][outside], A0[c][outside]) and np.array_equal(x1[c][n:], x0[c][n:]), c
        host_A, host_x = A0[c].copy(), x0[c].copy()
        host_ok = E.lib(capset).emu_spd_solve(n, host_A, host_x)
        assert ok[c] == host_ok, (c, n, ok[c], host_ok)
        if c < n_good:
            A = np.tril(A0[c][:n, :n].astype(np.float64))
            A = A + np.tril(A, -1).T
            x, b = x1[c][:n].astype(np.float64), x0[c][:n].astype(np.float64)
            be = np.linalg.norm(A @ x - b) / (n * eps * np.linalg.norm(A, 2) * np.linalg.norm(x))
            worst = max(worst, be)
            assert ok[c] == 1
            fe = np.abs(x - np.linalg.solve(A, b)).max() / np.abs(np.linalg.solve(A, b)).max()
            assert fe < 4 * n * eps * np.linalg.cond(A) + 1e-6, (c, n, fe)
        else:
            assert ok[c] == 0
    print(f"spd_solve<32> ({capset}, n 1..{maxv}): backward error max {worst:.2f} n eps |A| |x|")
    assert worst <= 4.0


# ------------------------------------------------------------------------------------------------ hit / candidate lists
def _flag_patterns(cap, rs):
    """Flag arrays over several 32-item passes whose total count is cap - 1, cap, cap + 1 (crossing cap in the middle of
    a pass), and far beyond cap."""
    out = []
    for total in (0, 1, cap - 1, cap, cap + 1, cap + 17, 3 * cap + 5):
        for _ in range(4):
            nitems = max(total, 1) + rs.randint(0, 4 * 32)
            f = np.zeros(nitems, np.int32)
            f[rs.choice(nitems, total, replace=False)] = 1
            out.append(f)
    # the cap-th flagged item in the middle of a pass, dense runs around it
    f = np.zeros(cap + 64, np.int32)
    f[:cap + 10] = 1
    out.append(f)
    f = np.zeros(cap + 64, np.int32)
    f[1:cap] = 1
    f[cap + 20] = 1
    f[cap + 21] = 1
    out.append(f)
    return out


@pytest.mark.parametrize("capset", ["small", "kitchen"])
@pytest.mark.parametrize("which", ["hit", "cand"])
def test_ballot_compaction_keeps_item_order_and_flags_overflow(capset, which):
    """compact_append<32> / cand_append<32> against the serial loop: the flagged items in item order, the count clamped
    to the capacity, the overflow flag (hit: bad bit 1; cand: broad_valid cleared) set exactly when an item was dropped,
    and nothing written past the list (the neighbouring list in the workspace keeps its contents)."""
    if which == "cand" and capset == "small":
        pytest.skip("the door / peg capacity set has no cached broad phase")
    L = E.dev_lib(capset)
    cap = L.caps["MAXHIT" if which == "hit" else "MAXCAND"]
    rs = np.random.RandomState(11)
    pats = _flag_patterns(cap, rs)
    width = max(len(p) for p in pats)
    flags = np.zeros((len(pats), width), np.int32)
    for c, p in enumerate(pats):
        flags[c, :len(p)] = p
    hit, cand, info = E.append_device(which, flags, capset=capset)
    lst, other = (hit, cand) if which == "hit" else (cand, hit)
    for c, p in enumerate(pats):
        items = np.nonzero(p)[0]
        n = min(len(items), cap)
        assert info[c, 0] == n, (c, info[c], len(items))
        assert np.array_equal(lst[c, :n], items[:n]) and np.all(lst[c, n:] == 0xFFFF), c
        assert np.all(other[c] == 0xFFFF), c
        if which == "hit":
            assert info[c, 1] == (HIT_BAD if len(items) > cap else 0), (c, info[c])
        else:
            assert info[c, 1] == (0 if len(items) > cap else 1), (c, info[c])


# ------------------------------------------------------------------------------------------------ mesh support point
def test_mesh_support_is_the_first_maximum():
    """support_geom<32>'s lane-parallel argmax over a hull (883-vertex gripper base of the Sawyer models) against numpy's
    argmax (first maximum wins): axis-aligned directions (many exact ties) and random ones; then a hull with exact
    duplicates of the extreme vertices and distinct vertices tied along an axis, placed so that the later index sits in
    an earlier lane."""
    from earl_benchmark_b200.envs import sawyer_door
    m = Model.load(sawyer_door.MODEL_PATH)
    g = int(np.argmax(m.geom_hullnum))
    hv = np.asarray(m.hull_vert, np.float64).reshape(-1, 3)
    hull = hv[int(m.geom_hulladr[g]):int(m.geom_hulladr[g]) + int(m.geom_hullnum[g])].astype(np.float32)
    assert len(hull) == 883
    rs = np.random.RandomState(13)
    axes = np.concatenate([np.eye(3), -np.eye(3)])
    diag = np.array([[a, b, c] for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1) if (a, b, c) != (0, 0, 0)], np.float64)
    rnd = rs.standard_normal((400, 3))

    def check(H, dirs, exact):
        got = E.support_device(H, dirs)
        dd = H.astype(np.float64) @ dirs.T            # [nvert, ndir]
        for k in range(len(dirs)):
            best = int(np.argmax(dd[:, k]))
            if exact[k]:
                assert np.array_equal(got[k], H[best].astype(np.float64)), (k, dirs[k], got[k], best)
            else:
                # rounding of the fp64 dot products (FMA) can only decide between vertices within 1e-12 of the maximum
                near = np.nonzero(dd[:, k] >= dd[best, k] - 1e-12 * np.abs(dd[:, k]).max())[0]
                assert any(np.array_equal(got[k], H[j].astype(np.float64)) for j in near), (k, dirs[k])
    check(hull, np.concatenate([axes, diag, rnd]), [True] * (len(axes) + len(diag)) + [False] * len(rnd))
    # ties placed against the lane order: index 40 (lane 8) and index 70 (lane 6) both reach the maximum along +z
    H = (rs.standard_normal((100, 3)) * 0.3).astype(np.float32)
    H[40], H[70] = (0.2, -0.1, 2.0), (-0.3, 0.1, 2.0)
    H[45], H[90] = (3.0, 0.5, 0.1), (3.0, 0.5, 0.1)     # exact duplicates, lanes 13 and 26, along +x
    H[33], H[2] = (0.0, -4.0, 0.25), (0.5, -4.0, -0.25)  # tie along -y: index 2 (lane 2) before index 33 (lane 1)
    dirs = np.array([[0, 0, 1.0], [1.0, 0, 0], [0, -1.0, 0]])
    got = E.support_device(H, dirs)
    assert np.array_equal(got[0], H[40].astype(np.float64)) and np.array_equal(got[1], H[45].astype(np.float64))
    assert np.array_equal(got[2], H[2].astype(np.float64))
    check(H, np.concatenate([dirs, rnd[:50]]), [True] * 3 + [False] * 50)


# ------------------------------------------------------------------------------------------------ one substep
@pytest.mark.parametrize("name", MODELS)
@pytest.mark.parametrize("which", ["primary", "xl"])
def test_one_substep_every_capacity_set(name, which):
    """One whole substep per state in each capacity set against the one-lane build of the same set and the checker,
    with bars far tighter than the end-to-end tests (the measured maxima are printed).  Primary kitchen set: a state whose
    rows outgrow the 112 is flagged (bit 3) and left to the extra-large set, as the product does."""
    m, S = states(name)
    capset = PRIMARY[name] if which == "primary" else XL[name]
    d = device(name, m, S, capset)
    d.run("substeps", 1)
    em, e = E.Emu(m, task(name, m), capset=capset), Engine(m)
    rs = np.random.RandomState(2)
    dh, dc, flagged, excused = [], [], 0, []
    for i, s in enumerate(S):
        q, v, w = d.state(i)
        bad = d.info(i)["bad"]
        if bad:
            # the primary kitchen set drops rows beyond its 112 and flags the state for the extra-large set
            assert capset == "kitchen" and bad == LIMIT_BAD, (i, bad)
            flagged += 1
            continue
        host_run(em, s, "substeps", 1)
        hq, hv, hw = em.state()
        gd, gh = d.contacts(i)[3], em.contacts()[3]
        ref_geoms = checker_geoms(checker(e, s))
        if not (np.array_equal(gd, gh) and [tuple(sorted(g)) for g in gd.tolist()] == [tuple(sorted(g)) for g in ref_geoms]):
            assert checker_flips(e, s, rs), i      # a contact at its activation margin (see the collision test)
            excused.append(i)
            continue
        checker(e, s)
        e.step(1)
        dh.append(max(np.abs(q - hq).max(), np.abs(v - hv).max()))
        dc.append((np.abs(q - e.qpos).max(), np.abs(v - e.qvel).max()))
    dh, dc = np.array(dh), np.array(dc)
    print(f"{name} one substep ({capset}, {len(S)} states, {flagged} flagged, excused {excused}): device vs one-lane max "
          f"{dh.max():.2e} median {np.median(dh):.2e}; vs checker dq max {dc[:, 0].max():.2e}, dv max {dc[:, 1].max():.2e} "
          f"p99 {np.percentile(dc[:, 1], 99):.2e}")
    assert len(dh) >= 100 and len(excused) <= len(S) // 20
    tol = SUBSTEP_TOL[name]
    assert dh.max() < tol["host"] and dc[:, 0].max() < tol["dq"] and dc[:, 1].max() < tol["dv"], (dh.max(), dc.max(axis=0))


# measured on the B200 (max over the set, one substep): device vs one-lane 1.0e-4 / 9.1e-6 / 3.7e-5, device vs checker dq
# 2.2e-7 / 1.2e-7 / 1.4e-7, dv 8.5e-5 / 5.3e-6 / 6.0e-5 (door / peg / kitchen); kN contact forces on gram-scale wrist inertias
# make qvel the sensitive output (fp32 positions: the one-lane build is 9.8e-5 from the checker on the door)
SUBSTEP_TOL = {
    "door": dict(host=5e-4, dq=1e-6, dv=5e-4),
    "peg": dict(host=5e-5, dq=1e-6, dv=5e-5),
    "kitchen": dict(host=2e-4, dq=1e-6, dv=2e-4),
}
