"""The reference's ROS nodes, compiled unmodified (oracle/Makefile `nodes`, tests/ros_lite) and replayed on scripted
message sequences:

* nurtlesim/src/tube_world.cpp with every noise source switched off pins the arithmetic of the trace generator
  (ekf-slam-ml_b200/tracegen.py) - truth kinematics, wheel increments, collision snap-back, fake sensor transform and
  visibility, 360-beam ray cast - to the reference itself (SURVEY.md section 8 f-1);
* nuslam/src/{slam,unknown_data_assoc,landmarks}.cpp built against this repository's facade headers + C ABI publish
  the same paths, landmark maps and transforms as the same sources built against the reference's own rigid2d classes
  (section 8 f-2; GPU).

The binaries are built by oracle/Makefile where EKF_SLAM_REFERENCE names a reference checkout; tests skip without them."""
import numpy as np
import pytest

import _ros_lite as rl


def _noise_free_world(tg, tubes=None):
    w = tg.default_world()
    if tubes is not None:
        w.tubes_x, w.tubes_y = np.array(tubes[0], float), np.array(tubes[1], float)
    w.vx_std = w.the_std = w.sensor_std = w.range_std = 0.0
    w.slip_min = w.slip_max = 1.0
    return w


def _tube_world_params(w):
    p = dict(rl.ROBOT_PARAMS)
    p.update(vx_mu=0.0, vx_std=w.vx_std, the_mu=0.0, the_std=w.the_std, slip_min=w.slip_min, slip_max=w.slip_max,
             tube_coor_x=list(w.tubes_x), tube_coor_y=list(w.tubes_y), tube_radius=w.tube_radius,
             covar_sensor_x=w.sensor_std, covar_sensor_y=w.sensor_std, max_visible_dis=w.max_visible,
             world_border_width=w.border, range_std=w.range_std)
    return p


@pytest.mark.parametrize("case", ["circle", "collision"])
def test_tube_world_pins_the_trace_generator(pkg, case):
    binary = rl.node_path("node_tube_world")
    if binary is None:
        pytest.skip("oracle/_ref/node_tube_world not built (set EKF_SLAM_REFERENCE to a reference checkout and build)")
    tg = pkg.tracegen
    if case == "circle":
        w = _noise_free_world(tg)
    else:  # a tube on the path: the robot runs into it and is snapped back every tick (tube_world.cpp:338-366)
        w = _noise_free_world(tg, tubes=([0.25, -0.5], [0.02, 0.6]))
        w.cmd_radius = 5.0
    ticks = 480
    sc = rl.Scenario(_tube_world_params(w))
    for k in range(0, ticks, 10):  # a command every 100 ms, ahead of the tick that consumes it
        sc.cmd_vel(k / 100.0 + 0.005, w.cmd_v, w.cmd_v / w.cmd_radius)
    out, _ = rl.run_node(binary, sc, ticks / 100.0, topics=["joint_states", "fake_sensor", "scan", "real_path"])
    sim = tg.TubeWorldSim(w, 1, seed=0)
    joints = {round(t, 3): f for t, f in out["joint_states"]}
    fake = {round(t, 3): f for t, f in out["fake_sensor"]}
    scans = {round(t, 3): f for t, f in out.get("scan", [])}
    lw = rw = 0.0
    worst = dict(joint=0.0, fake=0.0, scan=0.0)
    n_fake = n_scan = 0
    for k in range(1, ticks + 1):
        sim.step_tick()
        t = round(k / 100.0, 3)
        lw += float(sim.dl[0])
        rw += float(sim.dr[0])
        j = joints[t]
        worst["joint"] = max(worst["joint"], abs(j[0] - lw), abs(j[1] - rw), abs(j[2] - float(sim.dl[0])), abs(j[3] - float(sim.dr[0])))
        if t in fake:
            rx, ry, vis = sim.fake_sensor()
            f = fake[t]
            assert int(f[0]) == w.n_tubes
            for i in range(w.n_tubes):
                assert (f[2 + 4 * i] == 0.0) == bool(vis[0, i]), f"visibility of tube {i} at t={t}"
                worst["fake"] = max(worst["fake"], abs(f[3 + 4 * i] - rx[0, i]), abs(f[4 + 4 * i] - ry[0, i]))
            n_fake += 1
        if t in scans:
            r = sim.laser_scan(360)[0]
            got = np.array(scans[t][1:], dtype=np.float32)
            assert got.size == 360
            worst["scan"] = max(worst["scan"], float(np.max(np.abs(got - r))))
            n_scan += 1
    assert n_fake >= 40 and n_scan >= 20
    assert worst["joint"] < 1e-12 and worst["fake"] < 1e-9 and worst["scan"] < 2e-6, worst


def _known_scenario(tg, steps, seed):
    """Joint states at 100 Hz and the fake-sensor message every 11th tick, as nurtlesim publishes them."""
    w = tg.default_world()
    sim = tg.TubeWorldSim(w, 1, seed=seed)
    sc = rl.Scenario(rl.ROBOT_PARAMS)
    lw = rw = 0.0
    k = 0
    for _ in range(steps):
        for _ in range(11):
            sim.step_tick()
            k += 1
            lw += float(sim.dl[0])
            rw += float(sim.dr[0])
            sc.joint(k / 100.0 - 0.005, lw, rw, float(sim.dl[0]), float(sim.dr[0]))
        rx, ry, vis = sim.fake_sensor()
        sc.fake_sensor(k / 100.0 - 0.004, rx[0], ry[0], vis[0])
    return sc, k / 100.0 + 0.3


@pytest.mark.gpu
def test_slam_node_source_runs_on_the_facade(gpu_pkg):
    ref, ours = rl.node_path("node_slam_ref"), rl.node_path("node_slam_b200")
    if ref is None or ours is None:
        pytest.skip("oracle/_ref/node_slam_* not built (set EKF_SLAM_REFERENCE to a reference checkout and build)")
    sc, t_end = _known_scenario(gpu_pkg.tracegen, steps=110, seed=3)
    topics = ["slam_path", "slam_tube", "/tf"]
    a, _ = rl.run_node(ours, sc, t_end, topics)
    b, _ = rl.run_node(ref, sc, t_end, topics)
    assert len(b["slam_path"]) > 100
    for topic in topics:
        rl.compare_streams(a, b, topic, 1e-9)


def _scan_scenario(tg, n_scans, seed):
    w = tg.default_world()
    sim = tg.TubeWorldSim(w, 1, seed=seed)
    sc = rl.Scenario(rl.ROBOT_PARAMS)
    k = 0
    for _ in range(n_scans):
        for _ in range(21):
            sim.step_tick()
            k += 1
        sc.scan(k / 100.0 - 0.004, sim.laser_scan(360)[0])
    return sc, k / 100.0 + 0.05


@pytest.mark.gpu
def test_landmarks_node_source_runs_on_the_facade(gpu_pkg):
    ref, ours = rl.node_path("node_landmarks_ref"), rl.node_path("node_landmarks_b200")
    if ref is None or ours is None:
        pytest.skip("oracle/_ref/node_landmarks_* not built (set EKF_SLAM_REFERENCE to a reference checkout and build)")
    sc, t_end = _scan_scenario(gpu_pkg.tracegen, n_scans=12, seed=5)
    a, _ = rl.run_node(ours, sc, t_end, ["scan_sensor"])
    b, _ = rl.run_node(ref, sc, t_end, ["scan_sensor"])
    assert sum(int(f[0]) for _, f in b["scan_sensor"]) > 0, "the reference found no circle in any scan"
    rl.compare_streams(a, b, "scan_sensor", 1e-9)


@pytest.mark.gpu
def test_unknown_data_assoc_node_source_runs_on_the_facade(gpu_pkg):
    ref, ours = rl.node_path("node_unknown_data_assoc_ref"), rl.node_path("node_unknown_data_assoc_b200")
    lm = rl.node_path("node_landmarks_ref")
    if ref is None or ours is None or lm is None:
        pytest.skip("oracle/_ref/node_unknown_data_assoc_* not built (set EKF_SLAM_REFERENCE to a reference checkout and build)")
    tg = gpu_pkg.tracegen
    w = tg.default_world()
    sim = tg.TubeWorldSim(w, 1, seed=9)
    sc = rl.Scenario(rl.ROBOT_PARAMS)
    scans = rl.Scenario(rl.ROBOT_PARAMS)
    lw = rw = 0.0
    k = 0
    scan_ticks = []
    for _ in range(40):
        for _ in range(21):
            sim.step_tick()
            k += 1
            lw += float(sim.dl[0])
            rw += float(sim.dr[0])
            sc.joint(k / 100.0 - 0.005, lw, rw, float(sim.dl[0]), float(sim.dr[0]))
        scans.scan(k / 100.0 - 0.004, sim.laser_scan(360)[0])
        scan_ticks.append(k)
    t_end = k / 100.0 + 0.3
    # the landmark detector (the reference's own build) turns the scans into circle centres: one message per 10 ms tick
    # while a scan is current; the association node takes the first one after each scan
    circ, _ = rl.run_node(lm, scans, t_end, ["scan_sensor"])
    by_t = {round(t, 3): f for t, f in circ["scan_sensor"]}
    fed = 0
    for kt in scan_ticks:
        f = by_t.get(round(kt / 100.0, 3))
        if f is None:
            continue
        m = int(f[0])
        sc.circles(kt / 100.0 + 0.001, [(f[3 + 4 * i], f[4 + 4 * i]) for i in range(m)])
        fed += m
    assert fed > 20, "too few circle detections to exercise the association"
    topics = ["slam_path", "slam_tube", "/tf"]
    a, _ = rl.run_node(ours, sc, t_end, topics)
    b, _ = rl.run_node(ref, sc, t_end, topics)
    for topic in topics:
        rl.compare_streams(a, b, topic, 1e-9)
