"""Pins the CPU oracle's Unitree G1 whole-body terms.

The reference has NO known-answer test for the G1 rigid-body / cost / constraint blocks (SURVEY.md §8c: "G1 parity unpinned by
the reference's tests"), and Pinocchio is not in this image.  The oracle is therefore pinned by
  (a) physical identities (recipes x-xi of §8c: zero momentum rate under weight-compensating wrenches, total mass, M = M' > 0,
      RNEA(q,v,a) = M a + nle computed by two different algorithms, frame velocity/acceleration = time derivatives of position),
  (b) central finite differences of every Jacobian the oracle produces with dual numbers,
  (c) the model loader's facts: 23 joints, total mass 35.115 kg (sum of URDF <mass>), joint order of task.info.
"""
import numpy as np
import pytest

import oracle_lib as orc
from wb_humanoid_mpc_b200 import model_loader, references


@pytest.fixture(scope="module")
def model():
    return model_loader.load_packaged_model()


@pytest.fixture(scope="module")
def wb(model):
    return orc.WbOracle(model)


def rand_state(model, rng, scale=1.0):
    x = np.array(model["x_init"], float)
    nj = model["nj"]
    x[0:3] += rng.uniform(-0.05, 0.05, 3) * scale
    x[3:6] += rng.uniform(-0.2, 0.2, 3) * scale
    x[6:6 + nj] += rng.uniform(-0.3, 0.3, nj) * scale
    x[6 + nj:] += rng.uniform(-0.5, 0.5, 6 + nj) * scale
    return x


def rand_input(model, rng):
    u = references.weight_compensating_input(model, (1, 1))
    u[:12] += rng.uniform(-20, 20, 12)
    u[3:6] *= 0.1
    u[9:12] *= 0.1
    u[12:] += rng.uniform(-2, 2, model["nj"])
    return u


def fd_jac(f, z, eps=1e-6):
    f0 = f(z)
    J = np.zeros((len(f0), len(z)))
    for i in range(len(z)):
        zp, zm = z.copy(), z.copy()
        zp[i] += eps
        zm[i] -= eps
        J[:, i] = (f(zp) - f(zm)) / (2 * eps)
    return J


def test_model_facts(model, wb):
    assert model["nj"] == 23 and model["nx"] == 58 and model["nu"] == 35
    assert abs(wb.total_mass() - 35.11514202) < 1e-9
    assert model["joint_names"][0] == "left_hip_pitch_joint" and model["joint_names"][-1] == "right_elbow_joint"
    assert model["joint_names"][12] == "waist_yaw_joint"
    # task.info initialState ordering: knees at index 3 / 9 start at 0.1 rad
    assert model["x_init"][6 + 3] == 0.1 and model["x_init"][6 + 9] == 0.1
    # the weight-loading quirk (EndEffectorDynamicsCostHelpers.cpp:103-108): velocity weights carry the acceleration entries
    assert model["foot_cost_weights"][6:9] == [5.0, 5.0, 0.0] and model["foot_cost_weights"][12:] == [0.01] * 6


def test_packaged_model_matches_reference_files(model):
    """the committed JSON is what the loader derives from the reference's URDF/task.info (copies under tests/golden/g1_config)"""
    from pathlib import Path

    fresh = model_loader.build_g1_wb_from_reference(Path(__file__).resolve().parent / "golden" / "g1_config")
    import json

    assert json.loads(json.dumps(fresh)) == model


def test_mass_matrix_properties(model, wb):
    rng = np.random.default_rng(0)
    for _ in range(3):
        x = rand_state(model, rng)
        M, _ = wb.crba_nle(x)
        assert np.allclose(M, M.T, atol=1e-12)
        assert np.min(np.linalg.eigvalsh(M)) > 0
        assert np.allclose(M[:3, :3], wb.total_mass() * np.eye(3), atol=1e-10)


def test_rnea_equals_crba_plus_nle(model, wb):
    """two independent algorithms: RNEA(q,v,a) == CRBA(q) a + RNEA(q,v,0)"""
    rng = np.random.default_rng(1)
    nv = 6 + model["nj"]
    for _ in range(4):
        x = rand_state(model, rng)
        a = rng.uniform(-3, 3, nv)
        M, nle = wb.crba_nle(x)
        tau = wb.rnea(x[:nv], x[nv:], a)
        assert np.allclose(tau, M @ a + nle, atol=1e-9)


def test_gravity_and_static_equilibrium(model, wb):
    """recipe (x): at rest, weight-compensating wrenches give zero base linear acceleration; nle_lin = m g e_z"""
    x = np.array(model["x_init"], float)
    M, nle = wb.crba_nle(x)
    assert np.allclose(nle[:3], [0, 0, wb.total_mass() * 9.81], atol=1e-9)
    u = references.weight_compensating_input(model, (1, 1))
    xd = wb.flow_map(x, u)
    nv = 6 + model["nj"]
    assert np.allclose(xd[nv:nv + 3], 0.0, atol=1e-10)
    # single support carries the full weight on one foot
    u1 = references.weight_compensating_input(model, (1, 0))
    assert abs(u1[2] - wb.total_mass() * 9.81) < 1e-12 and u1[8] == 0
    assert np.allclose(wb.flow_map(x, u1)[nv:nv + 3], 0.0, atol=1e-10)


def test_base_acceleration_matches_literal_restatement(model, wb):
    """fused RNEA form == literal crba/nle/Jacobian products with the block-diagonal M_bb inverse
    (humanoid_common_mpc/src/pinocchio_model/DynamicsHelperFunctions.cpp:196-218)"""
    rng = np.random.default_rng(2)
    nv = 6 + model["nj"]
    for _ in range(4):
        x, u = rand_state(model, rng), rand_input(model, rng)
        lit = wb.base_accel_literal(x, u)
        xd = wb.flow_map(x, u)
        assert np.allclose(xd[nv:nv + 6], lit, rtol=1e-10, atol=1e-9)
        assert np.allclose(xd[:nv], x[nv:])
        assert np.allclose(xd[nv + 6:], u[12:])


def test_block_diagonal_inverse_differs_from_exact(model, wb):
    """the dropped lin/ang coupling is part of the spec: the reference's base acceleration is NOT the exact forward dynamics"""
    rng = np.random.default_rng(3)
    nv = 6 + model["nj"]
    x, u = rand_state(model, rng), rand_input(model, rng)
    M, nle = wb.crba_nle(x)
    xd = wb.flow_map(x, u)
    qdd = xd[nv:]
    # exact base rows residual would vanish for the exact solve; here only the block-diagonal part is satisfied
    feet, _ = wb.foot_state(x, u)
    lin_res = M[:3, :3] @ qdd[:3] + M[:3, 6:] @ qdd[6:] + nle[:3] - (u[0:3] + u[6:9])
    assert np.allclose(lin_res, 0.0, atol=1e-8)
    full_res = M[:3] @ qdd + nle[:3] - (u[0:3] + u[6:9])
    assert np.max(np.abs(full_res)) > 1e-4


def test_frame_kinematics_are_time_derivatives(model, wb):
    """getFrameVelocity / getFrameClassicalAcceleration(LOCAL_WORLD_ALIGNED) = d/dt of frame position / velocity along the flow"""
    rng = np.random.default_rng(4)
    nv = 6 + model["nj"]
    x, u = rand_state(model, rng), rand_input(model, rng)
    xd = wb.flow_map(x, u)
    h = 1e-6

    def feet_at(s):
        # second-order Taylor step of (q, v) along (v, a)
        xs = x.copy()
        xs[:nv] = x[:nv] + s * x[nv:] + 0.5 * s * s * xd[nv:]
        xs[nv:] = x[nv:] + s * xd[nv:]
        return wb.foot_state(xs, u)[0]

    f0, fp, fm = wb.foot_state(x, u)[0], feet_at(h), feet_at(-h)
    for c in range(2):
        v_fd = (fp[c]["pos"] - fm[c]["pos"]) / (2 * h)
        a_fd = (fp[c]["vlin"] - fm[c]["vlin"]) / (2 * h)
        assert np.allclose(f0[c]["vlin"], v_fd, atol=1e-7)
        assert np.allclose(f0[c]["alin"], a_fd, atol=1e-5)
        w_fd = (fp[c]["vang"] - fm[c]["vang"]) / (2 * h)
        assert np.allclose(f0[c]["aang"], w_fd, atol=1e-5)
        # R' = [w]x R
        Rd = (fp[c]["R"] - fm[c]["R"]) / (2 * h)
        W = Rd @ f0[c]["R"].T
        assert np.allclose([W[2, 1], W[0, 2], W[1, 0]], f0[c]["vang"], atol=1e-6)


def test_contact_frames_geometry(model, wb):
    """foot contact frames sit 3.5 cm below / ahead of the ankle-roll joints; in the nominal pose both feet are near z = 0"""
    x = np.array(model["x_init"], float)
    x[2] = model["reference"]["defaultBaseHeight"]
    feet, frames = wb.foot_state(x, np.zeros(model["nu"]))
    assert abs(feet[0]["pos"][2]) < 0.02 and abs(feet[1]["pos"][2]) < 0.02
    assert feet[0]["pos"][1] > 0.05 and feet[1]["pos"][1] < -0.05  # left is +y
    assert np.allclose(frames[1] - frames[0], feet[0]["R"] @ [0.054, 0, 0], atol=1e-12)
    assert np.allclose(frames[2] - frames[0], feet[0]["R"] @ [-0.054, 0, 0], atol=1e-12)


def test_flow_map_jacobian_vs_finite_differences(model, wb):
    rng = np.random.default_rng(5)
    nx, nu = model["nx"], model["nu"]
    x, u = rand_state(model, rng), rand_input(model, rng)
    f, A, B = wb.flow_map_lin(x, u)
    assert np.allclose(f, wb.flow_map(x, u), atol=1e-12)
    J = fd_jac(lambda z: wb.flow_map(z[:nx], z[nx:]), np.concatenate([x, u]), 1e-6)
    assert np.max(np.abs(A - J[:, :nx])) < 2e-6
    assert np.max(np.abs(B - J[:, nx:])) < 2e-6
    # structure: only the six base-acceleration rows are dense
    nv = nx // 2
    assert np.allclose(A[:nv, :nv], 0) and np.allclose(A[:nv, nv:], np.eye(nv))
    assert np.allclose(A[nv + 6:], 0) and np.allclose(B[:nv], 0)
    assert np.allclose(B[nv + 6:, 12:], np.eye(model["nj"])) and np.allclose(B[nv + 6:, :12], 0)
    assert np.allclose(A[nv:nv + 6, :3], 0)  # base acceleration does not depend on the base position


def _nodes(model, contact, swing=None, impact=None, arm=0.3):
    n = 1
    xref = np.array(model["x_init"], float)[None].copy()
    xref[0, 29:31] = [0.4, 0.1]
    sw = np.zeros((n, 2, 3)) if swing is None else np.asarray(swing, float).reshape(n, 2, 3)
    ip = np.ones((n, 2)) if impact is None else np.asarray(impact, float).reshape(n, 2)
    return dict(contact=np.array([contact], dtype=np.uint8), swing=sw, impact=ip, arm_phase=np.array([arm]), xref=xref)


@pytest.mark.parametrize("contact,nc", [((1, 1), 12), ((1, 0), 13), ((0, 1), 13), ((0, 0), 14)])
def test_constraints_jacobian_and_counts(model, wb, contact, nc):
    rng = np.random.default_rng(6)
    nx = model["nx"]
    nd = _nodes(model, contact, swing=[[0.03, 0.2, -1.0], [0.05, -0.1, 0.5]])
    wb.set_nodes(nd["contact"], nd["swing"], nd["impact"], nd["arm_phase"], nd["xref"])
    x, u = rand_state(model, rng), rand_input(model, rng)
    g, Cm, Dm = wb.eq_constraint_lin(0, x, u)
    assert len(g) == nc
    assert np.allclose(g, wb.eq_constraint(0, x, u), atol=1e-12)
    J = fd_jac(lambda z: wb.eq_constraint(0, z[:nx], z[nx:]), np.concatenate([x, u]), 1e-6)
    assert np.max(np.abs(Cm - J[:, :nx])) < 5e-5 * max(1.0, np.max(np.abs(Cm)))
    assert np.max(np.abs(Dm - J[:, nx:])) < 5e-6 * max(1.0, np.max(np.abs(Dm)))
    assert np.linalg.matrix_rank(Dm) == nc
    # zero-wrench rows are identity blocks on the swing foot's wrench
    row = 0
    for c in range(2):
        if not contact[c]:
            assert np.allclose(Dm[row:row + 6, 6 * c:6 * c + 6], np.eye(6)) and np.allclose(Cm[row:row + 6], 0)
            assert np.allclose(g[row:row + 6], u[6 * c:6 * c + 6])
            row += 7
        else:
            row += 6


@pytest.mark.parametrize("contact", [(1, 1), (1, 0), (0, 0)])
def test_cost_gradient_vs_finite_differences(model, wb, contact):
    rng = np.random.default_rng(7)
    nx = model["nx"]
    nd = _nodes(model, contact, impact=[0.7, 0.4])
    wb.set_nodes(nd["contact"], nd["swing"], nd["impact"], nd["arm_phase"], nd["xref"])
    x, u = rand_state(model, rng, 0.5), rand_input(model, rng)
    u[2] += 100
    u[8] += 100  # keep the friction cone in its log-barrier branch
    x[6 + 3] = model["q_upper"][3] - 0.03  # activate a joint-limit barrier
    q = wb.cost_quad(0, x, u)
    assert abs(q["f"] - wb.cost(0, x, u)) < 1e-9 * max(1.0, abs(q["f"]))
    assert np.allclose(q["Q"], q["Q"].T, atol=1e-10) and np.allclose(q["R"], q["R"].T, atol=1e-10)
    assert np.min(np.linalg.eigvalsh(q["R"])) > 0

    # the reference's quadratic tracking cost treats xNominal(x) as constant: compare against FD with frozen yaw dependence by
    # differentiating a cost whose arm-swing reference is evaluated at the expansion point -> set arm phase to 0 for the FD check
    nd0 = _nodes(model, contact, impact=[0.7, 0.4], arm=0.0)
    wb.set_nodes(nd0["contact"], nd0["swing"], nd0["impact"], nd0["arm_phase"], nd0["xref"])
    q0 = wb.cost_quad(0, x, u)
    g_fd = fd_jac(lambda z: np.array([wb.cost(0, z[:nx], z[nx:])]), np.concatenate([x, u]), 1e-6)[0]
    scale = max(1.0, np.max(np.abs(g_fd)))
    assert np.max(np.abs(q0["q"] - g_fd[:nx])) < 1e-5 * scale
    assert np.max(np.abs(q0["r"] - g_fd[nx:])) < 1e-5 * scale


def test_instance_builder_grid_matches_oracle_grid(model):
    """the product's host-side time grid (references.py) equals the oracle's restatement of timeDiscretizationWithEvents"""
    for gait, horizon in [("stance", 1.1), ("walk", 1.1), ("slow_walk", 3.5)]:
        inst = references.build_instance(model, model["x_init"], t0=0.13, horizon=horizon, gait=gait)
        t, e = orc.time_discretization(0.13, 0.13 + horizon, model["sqp"]["dt"], inst["mode_schedule"].event_times)
        assert np.array_equal(e, inst["node_event"]) and np.allclose(t, inst["t_nodes"], atol=0, rtol=0)


def test_walk_instance_schedule(model):
    inst = references.build_instance(model, model["x_init"], t0=0.0, horizon=3.5, gait="walk", cmd=[0.5, 0.0, 0.7925, 0.0])
    cf = inst["contact_flags"]
    assert cf.min() == 0 and cf.max() == 1
    assert (cf.sum(axis=1) >= 1).all()  # walking: never both feet in the air
    sw = inst["swing_ref"]
    # swing height reference peaks near swingHeight for a full-length swing and is zero for stance feet
    assert 0.07 < sw[:, :, 0].max() <= 0.0801
    assert np.all(sw[cf == 1][:, 0] == 0.0)
    assert inst["impact_factor"].min() < 0.1 and inst["impact_factor"].max() <= 1.0 + 1e-12
    assert len(inst["t_nodes"]) > 100


def test_warm_start_initialization(model):
    """initializeStateInputTrajectories: cold start = (x0, weight compensation); warm start interpolates the previous solution inside
    the overlap and falls back to the initializer for the tail (Initialization.cpp:35-79)."""
    x0 = np.array(model["x_init"], float)
    cold = references.build_instance(model, x0, t0=0.0, horizon=1.1, gait="walk")
    n = len(cold["t_nodes"])
    assert np.allclose(cold["x_init"], np.tile(x0, (n, 1)))
    for i in range(n - 1):
        if cold["node_event"][i] == 1:
            assert not cold["u_init"][i].any()
        else:
            assert np.allclose(cold["u_init"][i], references.weight_compensating_input(model, cold["contact_flags"][i]))
    # a synthetic previous solution: linear-in-time states/inputs so that interpolation can be checked exactly
    rng = np.random.default_rng(0)
    a, b = rng.uniform(-1, 1, model["nx"]), rng.uniform(-1, 1, model["nu"])
    prev_x = np.array([x0 + t * a for t in cold["t_nodes"]])
    prev_u = np.array([t * b for t in cold["t_nodes"][:-1]])
    prev = references.to_primal_solution(cold["t_nodes"], cold["node_event"], prev_x, prev_u)
    assert len(prev["t"]) == len(prev["x"]) == len(prev["u"])
    shift = 0.02
    warm = references.build_instance(model, x0 + shift * a, t0=shift, horizon=1.1, gait="walk", previous=prev)
    t_state_till, t_input_till = prev["t"][-1], prev["t"][-2]
    assert np.allclose(warm["x_init"][0], x0 + shift * a)
    checked_tail = checked_overlap = 0
    for i in range(len(warm["t_nodes"]) - 1):
        if warm["node_event"][i] == 1:
            continue
        t = references.interval_start(warm["t_nodes"][i], warm["node_event"][i])
        t_next = warm["t_nodes"][i + 1]
        if t > t_input_till or t_next > t_state_till:
            assert np.allclose(warm["u_init"][i], references.weight_compensating_input(model, warm["contact_flags"][i]))
            assert np.allclose(warm["x_init"][i + 1], warm["x_init"][i])
            checked_tail += 1
        elif warm["node_event"][i + 1] == 0 and warm["node_event"][i] == 0:
            assert np.allclose(warm["x_init"][i + 1], x0 + t_next * a, atol=1e-6)
            checked_overlap += 1
    assert checked_tail >= 1 and checked_overlap > 20
