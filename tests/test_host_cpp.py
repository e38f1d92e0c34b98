"""The C++ host layer (wb_humanoid_mpc_b200/host/*.hpp) against the independent Python restatement (references.py): every per-node array of
b200sqp_upload_instances must agree for cold and warm starts, all gaits, shifted gait phases.  CPU only (no compute calls)."""
import numpy as np
import pytest

from wb_humanoid_mpc_b200 import host_lib, model_loader, references


@pytest.fixture(scope="module")
def model():
    return model_loader.load_packaged_model()


@pytest.fixture(scope="module")
def hmodel():
    m = host_lib.HostModel()
    yield m
    m.close()


def test_flat_model_file_matches_json(model, hmodel):
    from wb_humanoid_mpc_b200 import abi

    d_py = abi.model_desc(model)
    d_cc, st = hmodel.desc_and_settings()
    assert bytes(d_py) == bytes(d_cc), "b200sqp_model_desc read by the C++ host differs from the Python mirror"
    sp = abi.default_settings(model)
    assert bytes(sp) == bytes(st)
    assert (hmodel.nx, hmodel.nu, hmodel.dt, hmodel.horizon) == (model["nx"], model["nu"], model["sqp"]["dt"], model["sqp"]["timeHorizon"])


KEYS = ["t_nodes", "node_event", "contact_flags", "swing_ref", "impact_factor", "arm_phase", "x_ref", "x_init", "u_init"]


def x0_of(model, rng):
    x0 = np.array(model["x_init"], float)
    x0[:6] += rng.uniform(-0.05, 0.05, 6)
    x0[29:35] += rng.uniform(-0.3, 0.3, 6)
    return x0


@pytest.mark.parametrize("gait,t0,horizon,start", [("stance", 0.0, 1.1, None), ("walk", 0.0, 3.5, None), ("walk", 0.37, 2.0, 0.1),
                                                   ("slow_walk", 1.25, 3.5, 0.5), ("trot", 0.0, 1.1, None), ("left_leg", 0.2, 1.5, 0.2)])
def test_cold_start_instance_matches_python(model, hmodel, gait, t0, horizon, start):
    rng = np.random.default_rng(7)
    x0 = x0_of(model, rng)
    cmd = [0.6, -0.1, model["reference"]["defaultBaseHeight"], 0.3]
    py = references.build_instance(model, x0, t0=t0, horizon=horizon, gait=gait, gait_start=start, cmd=cmd)
    cc = hmodel.build_instance(x0, t0=t0, horizon=horizon, gait=gait, gait_start=start, cmd=cmd)
    for k in KEYS:
        a, b = np.asarray(py[k]), np.asarray(cc[k])
        assert a.shape == b.shape, (k, a.shape, b.shape)
        assert np.allclose(a, b, rtol=0, atol=1e-13), (k, np.abs(a.astype(float) - b.astype(float)).max())


def test_warm_start_instance_matches_python(model, hmodel):
    rng = np.random.default_rng(9)
    x0 = x0_of(model, rng)
    first = references.build_instance(model, x0, t0=0.0, horizon=1.1, gait="walk")
    n = len(first["t_nodes"])
    # a made-up previous solution on the first grid (values are irrelevant to the interpolation logic)
    xs, us = rng.normal(size=(n, 58)), rng.normal(size=(n - 1, 35))
    prev = references.to_primal_solution(first["t_nodes"], first["node_event"], xs, us)
    x1 = x0 + 0.01
    py = references.build_instance(model, x1, t0=0.105, horizon=1.1, gait="walk", gait_start=0.0, previous=prev)
    cc = hmodel.build_instance(x1, t0=0.105, horizon=1.1, gait="walk", gait_start=0.0, previous=prev)
    for k in KEYS:
        assert np.allclose(np.asarray(py[k], float), np.asarray(cc[k], float), rtol=0, atol=1e-13), k
    # the overlap really is interpolated, the tail really is the weight-compensating initializer
    assert not np.allclose(cc["u_init"][0], cc["u_init"][-1])


def test_errors_are_reported(hmodel):
    with pytest.raises(RuntimeError, match="unknown gait"):
        hmodel.build_instance(np.zeros(58), gait="moonwalk")
    with pytest.raises(RuntimeError, match="not found"):
        host_lib.HostModel("/nonexistent/model.txt")


# ---- trajectorySpread (SqpSolver.cpp:211-213; ocs2_oc TrajectorySpreading) ----------------------------------------------------------------
def _rollout_like(ms, t0, tf, dt, eps=1e-9):
    """time trajectory in the OCS2 rollout convention (pre-event sample at t_e, post-event sample at t_e + eps) tagged with the active mode"""
    t, tags = [], []
    events = [e for e in ms.event_times if t0 < e < tf]
    grid = sorted(set(np.round(np.arange(t0, tf + 1e-12, dt), 12).tolist() + [tf]))
    for a in grid:
        t.append(a)
    for e in events:
        t += [e, e + eps]
    t = sorted(set(t))
    for a in t:
        tags.append(ms.mode_sequence[np.searchsorted(ms.event_times, a, side="left")])
    return np.array(t), np.array(tags, float)[:, None]


@pytest.mark.parametrize("seed", range(8))
def test_trajectory_spread_matches_python_and_reproduces_the_new_mode_sequence(seed):
    """the reference's own test idea (ocs2_oc/test/trajectory_adjustment/TrajectorySpreadingTest.cpp): tag every sample with its mode, spread
    to a perturbed schedule, and the tags must follow the new schedule wherever the matched window covers; C++ and Python must agree exactly"""
    rng = np.random.default_rng(seed)
    n_ev = int(rng.integers(2, 6))
    ev = np.sort(rng.uniform(0.3, 2.7, n_ev))
    modes = [int(m) for m in rng.permutation(8)[: n_ev + 1]]
    old = references.ModeSchedule(list(ev), modes)
    shifted = np.sort(np.clip(ev + rng.uniform(-0.12, 0.12, n_ev), 0.05, 2.95))
    new_modes = list(modes)
    if seed % 3 == 2:
        new_modes[-1] = 9                        # the tail mode changes: truncation
    new = references.ModeSchedule(list(shifted), new_modes)
    t, tags = _rollout_like(old, 0.0, 3.0, 0.1)
    prim = dict(t=t, x=tags, u=tags.copy())
    py = references.trajectory_spread(old, new, prim)
    ct, cx, cu, trunc, spread = host_lib.trajectory_spread(old.event_times, old.mode_sequence, new.event_times, new.mode_sequence, t, tags, tags)
    assert np.array_equal(py["t"], ct) and np.array_equal(py["x"], cx) and np.array_equal(py["u"], cu)
    assert (py["will_truncate"], py["will_spread"]) == (trunc, spread)
    # property: after spreading, every kept sample carries the mode the NEW schedule prescribes at its (adjusted) time
    for a, tag in zip(ct, cx[:, 0]):
        want = new.mode_sequence[np.searchsorted(new.event_times, a, side="left")]
        assert int(tag) == want, (a, tag, want)


def test_trajectory_spread_identical_schedules_sqp_time_convention(model):
    """the SQP's primal solution keeps pre- and post-event samples at the same time, so the reference's spreading moves the time of the
    sample after every event to event + eps even when nothing changed (documented quirk, reproduced by both restatements)"""
    inst = references.build_instance(model, np.array(model["x_init"], float), t0=0.0, horizon=1.1, gait="walk")
    n = len(inst["t_nodes"])
    prim = references.to_primal_solution(inst["t_nodes"], inst["node_event"], np.zeros((n, 58)), np.zeros((n - 1, 35)), inst["mode_schedule"])
    py = references.trajectory_spread(inst["mode_schedule"], inst["mode_schedule"], prim)
    ms = inst["mode_schedule"]
    ct, cx, cu, trunc, spread = host_lib.trajectory_spread(ms.event_times, ms.mode_sequence, ms.event_times, ms.mode_sequence, prim["t"], prim["x"], prim["u"])
    assert np.array_equal(py["t"], ct) and not trunc and not spread and len(ct) == n
    post = [i for i in range(1, n) if inst["node_event"][i] == 2]   # (an event at the initial time is outside the matched window)
    assert post, "the walk gait puts events inside the horizon"
    for i in post:
        if i + 1 < n - 1:
            assert abs(ct[i + 1] - (inst["t_nodes"][i] + 1e-9)) < 1e-15


# ---- centroidal model file and instance builder ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cmodel():
    return model_loader.load_packaged_model("g1_centroidal")


@pytest.fixture(scope="module")
def chmodel():
    m = host_lib.HostModel(host_lib.CEN_MODEL_TXT)
    yield m
    m.close()


def test_centroidal_flat_model_file_matches_json(cmodel, chmodel, hmodel):
    from wb_humanoid_mpc_b200 import abi

    d_cc, st = chmodel.desc_and_settings()
    assert bytes(abi.model_desc(cmodel)) == bytes(d_cc)
    assert bytes(abi.cen_desc(cmodel)) == bytes(chmodel.cen_desc())
    assert bytes(abi.default_settings(cmodel)) == bytes(st)
    assert (chmodel.nx, chmodel.nu, chmodel.dt, chmodel.horizon) == (35, 35, 0.02, 1.2)
    assert hmodel.cen_desc() is None


@pytest.mark.parametrize("gait,t0,horizon,start", [("stance", 0.0, 0.4, None), ("walk", 0.0, 2.0, None), ("walk", 0.37, 1.2, 0.1), ("trot", 0.0, 0.6, None)])
def test_centroidal_instance_matches_python(cmodel, chmodel, gait, t0, horizon, start):
    rng = np.random.default_rng(11)
    x0 = np.array(cmodel["x_init"], float)
    x0[:6] = rng.uniform(-0.1, 0.1, 6)
    x0[6:12] += rng.uniform(-0.05, 0.05, 6)
    bv = rng.uniform(-0.2, 0.2, 6)   # stands for Ab^-1 x0[:6] (a device quantity; any vector exercises the rule)
    cmd = [0.6, -0.1, cmodel["reference"]["defaultBaseHeight"], 0.3]
    py = references.build_instance(cmodel, x0, t0=t0, horizon=horizon, gait=gait, gait_start=start, cmd=cmd, base_vel=bv)
    cc = chmodel.build_instance(x0, t0=t0, horizon=horizon, gait=gait, gait_start=start, cmd=cmd, base_vel=bv)
    for k in KEYS:
        a, b = np.asarray(py[k]), np.asarray(cc[k])
        assert a.shape == b.shape, (k, a.shape, b.shape)
        assert np.allclose(a, b, rtol=0, atol=1e-13), (k, np.abs(a.astype(float) - b.astype(float)).max())
    # the target momentum rides in the first six reference states, the pose in the next six
    assert np.allclose(py["x_ref"][0, 2:5], 0) and py["x_ref"].shape[1] == 35
    # a non-zero momentum without base_vel is refused by the Python restatement
    with pytest.raises(ValueError):
        references.build_instance(cmodel, x0, t0=t0, horizon=horizon, gait=gait, cmd=cmd)


def test_srbd_model_file_and_base_velocity(cmodel, tmp_path):
    """centroidalModelType 1: the flat file carries the nominal inertia / com offset; the host's closed-form Ab^-1 hbar equals the Python one"""
    from wb_humanoid_mpc_b200 import abi, centroidal

    m1 = dict(cmodel)
    m1["centroidalModelType"] = 1
    path = tmp_path / "g1_srbd.txt"
    model_loader.write_flat(m1, path)
    hm = host_lib.HostModel(path)
    assert bytes(abi.cen_desc(m1)) == bytes(hm.cen_desc()) and hm.cen_desc().model_type == 1
    rng = np.random.default_rng(12)
    x0 = np.array(cmodel["x_init"], float)
    x0[:6] = rng.uniform(-0.2, 0.2, 6)
    x0[9:12] = rng.uniform(-0.4, 0.4, 3)
    assert np.allclose(hm.base_velocity(x0), centroidal.base_velocity(m1, x0), rtol=0, atol=1e-14)
    hm.close()


def test_example_application_compiles_links_and_fails_loudly_without_a_gpu(tmp_path):
    """examples/host_batch.cpp: the header-only host layer + SqpLogging build warning-free against the C ABI alone; without a CUDA device
    the application must stop with the library's error (no CPU fallback)"""
    import subprocess
    from pathlib import Path

    from wb_humanoid_mpc_b200 import lib

    root = Path(__file__).resolve().parents[1]
    lib.lib()   # make sure libb200sqp.so exists
    exe = tmp_path / "host_batch"
    pkg = root / "wb_humanoid_mpc_b200"
    res = subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", f"-I{root}", str(root / "examples" / "host_batch.cpp"), f"-L{pkg}", "-lb200sqp",
                          "-pthread", f"-Wl,-rpath,{pkg}", "-o", str(exe)], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    import torch

    if not torch.cuda.is_available():
        run = subprocess.run([str(exe), str(pkg / "data" / "g1_wb_model.txt"), "2"], capture_output=True, text=True, cwd=tmp_path)
        assert run.returncode == 1 and "no CPU fallback" in run.stderr


# ---- mpc_flattened_controller packing (MPC_ROS_Interface.cpp:98-178; SURVEY 8(f)-4) -----------------------------------------------------------------
@pytest.mark.parametrize("linear", [False, True])
def test_policy_message_packing_round_trip(model, linear):
    """createMpcPolicyMsg restated on plain structs: the feed-forward policy packs the inputs, the linear one [uff_i, K_i,:] per input with
    uff = u - K x; unflattening a sample and evaluating it at its own state gives the planned input back (float32 wire precision)"""
    import ctypes as C

    rng = np.random.default_rng(8)
    inst = references.build_instance(model, np.array(model["x_init"], float), t0=0.0, horizon=1.1, gait="walk")
    n, nx, nu = len(inst["t_nodes"]), 58, 35
    x, u = rng.normal(size=(n, nx)), rng.normal(size=(n - 1, nu))
    K = rng.normal(size=(n - 1, nx, nu)) * 0.1 if linear else None     # column-major (nu x nx) per stage = [n-1][nx][nu] in C order
    L = host_lib.lib()
    stride = nu * (1 + nx) if linear else nu
    data = np.zeros((n, stride), dtype=np.float32)
    post = np.zeros(n, dtype=np.uint16)
    n_post = C.c_int(0)
    probe = 7
    u_probe = np.zeros(nu)
    dp, u8p = C.POINTER(C.c_double), C.POINTER(C.c_uint8)
    ev = np.ascontiguousarray(inst["node_event"], dtype=np.uint8)
    tt = np.ascontiguousarray(inst["t_nodes"], dtype=np.float64)
    L.b200host_policy_msg.restype = C.c_int
    rc = L.b200host_policy_msg(n, nx, nu, tt.ctypes.data_as(dp), ev.ctypes.data_as(u8p), x.ctypes.data_as(dp), u.ctypes.data_as(dp),
                               None if K is None else K.ctypes.data_as(dp), data.ctypes.data_as(C.POINTER(C.c_float)), data.size,
                               post.ctypes.data_as(C.POINTER(C.c_uint16)), C.byref(n_post), probe, x[probe].ctypes.data_as(dp), u_probe.ctypes.data_as(dp))
    assert rc == stride, host_lib.lib().b200host_last_error()
    prim = references.to_primal_solution(inst["t_nodes"], inst["node_event"], x, u)
    assert list(post[: n_post.value]) == [i for i in range(n) if inst["node_event"][i] == 2]
    if not linear:
        assert np.allclose(data, np.asarray(prim["u"], dtype=np.float32))
    else:
        Kk = K[probe].T                                  # nu x nx
        assert np.allclose(data[probe].reshape(nu, 1 + nx)[:, 1:], Kk.astype(np.float32))
        assert np.allclose(data[probe].reshape(nu, 1 + nx)[:, 0], (prim["u"][probe] - Kk @ x[probe]).astype(np.float32), atol=1e-5)
    assert np.allclose(u_probe, prim["u"][probe], atol=2e-4)   # u = uff + K x at the sample's own state


def test_cpp_config_loader_equals_the_flat_model_file():
    """host/model_from_config.hpp reads the reference's OWN files (URDF + task.info + reference.info + gait.info: boost INFO subset, URDF subset,
    welded fixed joints, Pinocchio joint order, frames, weights) -- what a node passes to WBMpcInterface -- and must produce the HostModel the flat
    model file gives (that file is derived from the same config files by the Python loader, model_loader.py): every field of b200sqp_model_desc,
    the settings, the reference-manager parameters and the gait table.  The config files are copies under tests/golden/g1_config."""
    import ctypes as C
    from pathlib import Path

    from wb_humanoid_mpc_b200 import host_lib, model_loader

    root = Path(__file__).resolve().parent / "golden" / "g1_config"
    rel = model_loader.G1_REL
    files = [root / rel["urdf"], root / rel["task"], root / rel["reference"], root / rel["gait"]]
    a = host_lib.HostModel()                 # flat file
    b = host_lib.HostModel(config=files)     # C++ loader of the config files
    assert (a.nx, a.nu, a.dt, a.horizon) == (b.nx, b.nu, b.dt, b.horizon)
    (da, sa), (db, sb) = a.desc_and_settings(), b.desc_and_settings()
    for name, ctype in da._fields_:
        va, vb = np.ctypeslib.as_array(getattr(da, name)) if hasattr(getattr(da, name), "_length_") else getattr(da, name), \
            np.ctypeslib.as_array(getattr(db, name)) if hasattr(getattr(db, name), "_length_") else getattr(db, name)
        assert np.allclose(va, vb, rtol=1e-14, atol=1e-15, equal_nan=True), name
    assert bytes(sa) == bytes(sb)
    xa, xb = a.dump(), b.dump()
    assert xa.shape == xb.shape and np.allclose(xa, xb, rtol=1e-14, atol=1e-15)
    # missing files raise like the reference interfaces do (std::invalid_argument -> RuntimeError through the C layer)
    with pytest.raises(RuntimeError, match="not found"):
        host_lib.HostModel(config=[root / "nope.urdf", files[1], files[2], files[3]])
    # the centroidal MPC: other state layout and weights, task-space link frame, ICP / leg-torque costs, nominal inertia of the SRBD model type
    cfiles = [files[0], root / rel["centroidal_task"], root / rel["centroidal_reference"], files[3]]
    ca, cb = host_lib.HostModel(host_lib.CEN_MODEL_TXT), host_lib.HostModel(config=cfiles, centroidal=True)
    assert (ca.nx, ca.nu, ca.dt, ca.horizon) == (cb.nx, cb.nu, cb.dt, cb.horizon) and ca.nx == 35
    (da, sa), (db, sb) = ca.desc_and_settings(), cb.desc_and_settings()
    for name, _ in da._fields_:
        va, vb = getattr(da, name), getattr(db, name)
        if hasattr(va, "_length_"):
            va, vb = np.ctypeslib.as_array(va), np.ctypeslib.as_array(vb)
        assert np.allclose(va, vb, rtol=1e-13, atol=1e-15, equal_nan=True), name
    assert bytes(sa) == bytes(sb)
    xa, xb = ca.cen_desc(), cb.cen_desc()
    assert xa is not None and xb is not None
    for name, _ in xa._fields_:
        va, vb = getattr(xa, name), getattr(xb, name)
        if hasattr(va, "_length_"):
            va, vb = np.ctypeslib.as_array(va), np.ctypeslib.as_array(vb)
        assert np.allclose(va, vb, rtol=1e-12, atol=1e-14), name
    assert np.allclose(ca.dump(), cb.dump(), rtol=1e-14, atol=1e-15)
