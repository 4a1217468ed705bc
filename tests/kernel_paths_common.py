"""Kernel paths against the oracle over the whole joint range: a state sampler that reaches every quadrant of the joint
angles, every contact situation and the saturation branches of the motors, and a probe that compares ONE hot-path
evaluation of the device with the oracle.  Shared by tests/test_kernel_paths.py (warp emulator) and
tests/test_gpu_kernel_paths.py (`-m gpu`); `api=None` is the CUDA library."""
import contextlib
import os

import numpy as np

from jiminy_b200 import model as M
from jiminy_b200 import robots as R
from jiminy_b200.core import BatchedEngine
from oracle.oracle import OracleBatch

# development switches of the evaluation path (INTEGRATION.md); every one is read when a batch is created
SWITCHES = ("JB_LANES", "JB_QUADRUPED_ABA", "JB_NO_STATIC_PLAN", "JB_FORCE_PER_LANE", "JB_NO_FAST_KERNEL",
            "JB_NO_UNIFORM_SOLVER", "JB_NO_STRUCTURED_CONS", "JB_NO_BODY_CONS", "JB_NO_BLOCK_CONS", "JB_NO_FAST_BOUNDS")

# ANYmal's evaluation paths: (name, switches, what `describe()` must then say)
PATHS = (
    ("crba", {}, "hot path: quadruped signature, composite-rigid-body evaluation"),
    ("quadruped_aba", {"JB_QUADRUPED_ABA": "1"}, "hot path: quadruped signature, ABA sweeps"),
    ("no_static_plan", {"JB_NO_STATIC_PLAN": "1"}, "hot path: ABA sweeps (dynamic plan, lane-uniform descriptors)"),
    ("force_per_lane", {"JB_FORCE_PER_LANE": "1"}, "hot path: ABA sweeps (dynamic plan, per-lane descriptors)"),
    ("no_fast_kernel", {"JB_NO_FAST_KERNEL": "1"}, "hot path: none, every step runs the full kernel"),
    ("lanes1", {"JB_LANES": "1"}, "lanes=1 "),
    ("lanes2", {"JB_LANES": "2"}, "lanes=2 "),
)
PATH_NAMES = tuple(p[0] for p in PATHS)

# one evaluation of the right-hand side, relative to max(1, |reference|) (the RHS tolerance of the GPU suite)
RHS_TOL = 1e-12
# two paths from the same states after one 2 ms step: (q, v), relative.  Each path's evaluation agrees with the oracle to
# ~1e-13 (RHS_TOL above), but 20 steps through the 4e6 N/m ground amplify those rounding differences -- the paths differ
# in summation order and in their sin / cos (the default path's inline `jb_sincos` against the library's).  Measured on v:
# 1.4e-13 at 9 envs (emulator), 1.9e-12 at 1024 envs (emulator with nvcc's multiply-add contraction), 7.7e-12 at 4096
# envs (B200, explicit Euler; profiles/r03_kernel_paths_deviations.json); q within 3.6e-13 everywhere.  `a` at the final
# state is not compared across paths: it is the dynamics at slightly different states, where the stiff ground turns
# 1e-12 of state into 1e-11 of acceleration.
PATH_TOL = 2e-11


@contextlib.contextmanager
def switches(env):
    """Exactly the switches of `env` set while the block runs (any other one unset), the previous environment restored
    afterwards whatever happens."""
    saved = {k: os.environ.get(k) for k in SWITCHES}
    try:
        for k in SWITCHES:
            os.environ.pop(k, None)
        os.environ.update(env)
        yield
    finally:
        for k, x in saved.items():
            if x is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = x


def _quat_mul(a, b):
    ax, ay, az, aw = a
    bx, by, bz, bw = b
    return np.array([aw * bx + ax * bw + ay * bz - az * by, aw * by - ax * bz + ay * bw + az * bx,
                     aw * bz + ax * by - ay * bx + az * bw, aw * bw - ax * bx - ay * by - az * bz])


CONTACT_MODES = ("none", "some", "all")


def full_range_states(robot, n, rng, v_max=20.0, snap_fraction=0.25, tilt_max=np.pi / 3):
    """States over each joint's whole range, inside its bounds.

    * bounded revolute joints: uniform over their own bounds, less a margin (min(0.25 rad, 10 % of the range)) so that one
      env-step does not reach them; `snap_fraction` of them within 1e-9 rad of a multiple of pi/4 (the quadrant and octant
      boundaries of a sin / cos argument reduction);
    * continuous (unbounded) revolute joints at any angle; prismatic joints uniform inside their bounds;
    * free-flyer: any heading, tilted by up to `tilt_max` (60 degrees), at a height that puts none, some or all of the
      contact frames into the ground (env i gets CONTACT_MODES[i % 3]; "some" = the lowest frame 0.1-2 mm deep);
    * joint velocities uniform in +-v_max (20 rad/s, beyond the motors' velocity limits), base velocities up to 1 m/s
      and 2 rad/s.
    Returns (q, v, contact mode of every env)."""
    q = np.tile(robot.neutral(), (n, 1))
    v = np.zeros((n, robot.nv))
    for j in range(1, robot.njoints):
        t, iq, iv = int(robot.joint_type[j]), int(robot.idx_q[j]), int(robot.idx_v[j])
        if t == M.JB_JOINT_FREEFLYER:
            v[:, iv:iv + 3] = rng.uniform(-1.0, 1.0, size=(n, 3))
            v[:, iv + 3:iv + 6] = rng.uniform(-2.0, 2.0, size=(n, 3))
            continue
        if t == M.JB_JOINT_SPHERICAL:          # flexibility joint: a moderate rotation (its bounds are not angles)
            w = rng.normal(size=(n, 3)) * 0.2
            ang = np.linalg.norm(w, axis=1, keepdims=True)
            q[:, iq:iq + 3] = np.sin(ang / 2) * w / ang
            q[:, iq + 3] = np.cos(ang[:, 0] / 2)
            v[:, iv:iv + 3] = rng.uniform(-2.0, 2.0, size=(n, 3))
            continue
        v[:, iv] = rng.uniform(-v_max, v_max, size=n)
        if t in (M.JB_JOINT_RUBX, M.JB_JOINT_RUBY, M.JB_JOINT_RUBZ, M.JB_JOINT_RUBU):
            a = rng.uniform(-np.pi, np.pi, size=n)
            q[:, iq], q[:, iq + 1] = np.cos(a), np.sin(a)
            continue
        lo, hi = float(robot.q_lower[iq]), float(robot.q_upper[iq])
        m = min(0.25, 0.1 * (hi - lo))
        lo, hi = lo + m, hi - m
        x = rng.uniform(lo, hi, size=n)
        if t in (M.JB_JOINT_RX, M.JB_JOINT_RY, M.JB_JOINT_RZ, M.JB_JOINT_RU):
            ks = np.arange(np.ceil(lo / (np.pi / 4)), np.floor(hi / (np.pi / 4)) + 1)
            snap = rng.uniform(size=n) < snap_fraction
            if ks.size and snap.any():
                k = rng.choice(ks, size=int(snap.sum()))
                x[snap] = np.clip(k * (np.pi / 4) + rng.uniform(-1e-9, 1e-9, size=k.size), lo, hi)
        q[:, iq] = x
    modes = [CONTACT_MODES[i % 3] for i in range(n)]
    if robot.has_freeflyer:
        names = list(robot.contact_frame_names)
        legs = _leg_joints(robot, names)
        for i in range(n):
            for _ in range(100):
                yaw, tilt, phi = rng.uniform(-np.pi, np.pi), rng.uniform(0.0, tilt_max), rng.uniform(-np.pi, np.pi)
                qy = np.array([0.0, 0.0, np.sin(yaw / 2), np.cos(yaw / 2)])
                qt = np.array([np.cos(phi) * np.sin(tilt / 2), np.sin(phi) * np.sin(tilt / 2), 0.0, np.cos(tilt / 2)])
                q[i, 3:7] = _quat_mul(qy, qt)
                q[i, :3] = [rng.normal() * 0.1, rng.normal() * 0.1, 0.0]
                if not names:
                    q[i, 2] = 0.5
                    break
                if modes[i] == "all" and legs is not None and not _feet_level(robot, q[i], names, legs, rng):
                    for j in legs:                      # no common foot height: draw another leg posture and tilt
                        iq = int(robot.idx_q[j])
                        q[i, iq] = rng.uniform(robot.q_lower[iq] + 0.25, robot.q_upper[iq] - 0.25)
                    continue
                z = np.array([p.p[2] for p in R.frame_placements(robot, q[i], names).values()])
                if modes[i] == "none":
                    q[i, 2] = -z.min() + rng.uniform(0.01, 0.1)
                elif modes[i] == "some":
                    q[i, 2] = -z.min() - rng.uniform(1e-4, 2e-3)
                else:
                    q[i, 2] = -z.max() - rng.uniform(1e-4, 2e-3)
                break
    return q, v, modes


def _leg_joints(robot, names):
    """For each contact frame, a joint of its chain that no other contact frame depends on and that turns a full turn
    inside its bounds (ANYmal: the HFE of the leg), or None when some frame has none."""
    chains = []
    for nm in names:
        j, chain = robot.frames[nm].joint, []
        while j > 0:
            chain.append(j)
            j = int(robot.parent[j])
        chains.append(chain)
    legs = []
    for k, chain in enumerate(chains):
        others = {j for m, c in enumerate(chains) if m != k for j in c}
        cand = [j for j in chain if j not in others and int(robot.joint_type[j]) in (M.JB_JOINT_RX, M.JB_JOINT_RY, M.JB_JOINT_RZ, M.JB_JOINT_RU)
                and robot.q_upper[robot.idx_q[j]] - robot.q_lower[robot.idx_q[j]] > 2 * np.pi + 1.0]
        if not cand:
            return None
        legs.append(cand[-1])                   # the one nearest the root
    return legs


def _feet_level(robot, qi, names, legs, rng):
    """Turns the leg joint of every contact frame so that all the frames are at one height (with the base at z = 0), the
    angle kept anywhere in the joint's bounds (a random number of full turns).  False if no common height exists."""
    coef = []
    for nm, j in zip(names, legs):
        iq = int(robot.idx_q[j])
        z = []
        for th in (0.0, np.pi / 2, np.pi):      # a frame's height is A + B cos(th) + C sin(th) in the angle of one joint
            x = qi.copy()
            x[iq] = th
            z.append(R.frame_placements(robot, x, [nm])[nm].p[2])
        a = 0.5 * (z[0] + z[2])
        coef.append((a, 0.5 * (z[0] - z[2]), z[1] - a))
    lo = max(a - np.hypot(b, c) for a, b, c in coef)
    hi = min(a + np.hypot(b, c) for a, b, c in coef)
    if lo > hi - 1e-3:
        return False
    target = rng.uniform(lo + 2e-4, hi - 2e-4)
    for (a, b, c), j in zip(coef, legs):
        iq = int(robot.idx_q[j])
        th = np.arctan2(c, b) + rng.choice([-1.0, 1.0]) * np.arccos(np.clip((target - a) / np.hypot(b, c), -1.0, 1.0))
        lo_j, hi_j = robot.q_lower[iq] + 0.25, robot.q_upper[iq] - 0.25
        turns = np.arange(np.ceil((lo_j - th) / (2 * np.pi)), np.floor((hi_j - th) / (2 * np.pi)) + 1)
        qi[iq] = th + 2 * np.pi * rng.choice(turns)
    return True


def clean_velocities(robot, opt, q, v, cmd, step_dt):
    """The envs the oracle cannot run cleanly from (q, v) under `cmd` for one step -- `Engine::start` refuses a contact
    force above 1e5 N (a foot moving fast into the ground: the damping term), or the stiff ground throws a leg into its
    bounds or past what explicit steps resolve -- get their velocities halved until every env starts and steps cleanly.
    A handful of envs in a thousand are affected."""
    v = v.copy()
    for _ in range(20):
        orc = OracleBatch(robot, opt, len(q))
        orc.set_command(cmd)
        bad = orc.start(q, v) != 0
        if not bad.any():
            bad = (orc.step(step_dt, parallel=True) != 0) | (orc.get_status() != 0)
        if not bad.any():
            return v
        v[bad] *= 0.5
    raise AssertionError("no velocities the oracle steps cleanly from")


def over_limit_commands(robot, n, rng, factor=1.5):
    """Motor commands uniform in +-factor x the effort limit: the effort saturation of the motors is exercised."""
    lim = np.array([m.effort_limit if np.isfinite(m.effort_limit) else 50.0 for m in robot.motors])
    return rng.uniform(-factor, factor, size=(n, max(robot.nmotors, 1))) * np.r_[lim, np.ones(max(robot.nmotors, 1) - lim.size)]


def rel_dev(x1, x0):
    """max |x1 - x0| / max(1, max |x0|) over the batch: how the parity suite measures an evaluation (a contact force
    is k = 4e6 N/m times a penetration that is the difference of two lengths, so the force of a grazing contact carries
    the rounding of its position amplified -- only the scale of the batch makes it a rounding-level quantity)."""
    x1, x0 = np.asarray(x1), np.asarray(x0)
    if x0.size == 0:
        return 0.0
    return float(np.abs(x1 - x0).max() / max(1.0, np.abs(x0).max()))


def _outputs(x):
    """Everything a batch holds about the state it ended on, by name."""
    e, ja, jf = x.get_extra_terms()
    u, um, _, fext = x.get_efforts()
    out = {"a": x.get_state()[3], "u": u, "motor_efforts": um, "f_external": fext, "energy": e,
           "joint_accelerations": ja, "joint_wrenches": jf, "sensors": x.get_sensors()}
    for k, c in zip(("ycrb", "com", "vcom", "hg", "dhg"), x.get_centroidal()):
        out[k] = np.asarray(c)
    return out


def probe_options(solver):
    robot, opt = R.load_robot("anymal")
    opt = R.baseline_options("anymal", opt)
    # sensors and controller refreshed every 1 ms: the 2 ms step ends on a refresh, so the sensors are those of the final state
    opt["stepper"].update(odeSolver=solver, dtMax=1e-4,
                          sensorsUpdatePeriod=1e-3, controllerUpdatePeriod=1e-3)
    return robot, opt


def hot_path_probe(api, path, solver, n_env, seed=0, step_dt=2e-3, tol=RHS_TOL):
    """One hot-path evaluation of ANYmal (torque mode, spring-damper contacts) against the oracle, over the full range.

    A step leaves in `a` (and in the efforts, extra terms, centroidal terms and sensors) what the dynamics give at the
    state the step ended on.  So the device steps from full-range states, and the oracle is started at the DEVICE's final
    (q, v) with the same held command: the difference is that of the last evaluation of the step, made by the path under
    test (the fast kernel's evaluation, unless the path is the full kernel).  The premise is first checked on the oracle
    itself, bit for bit: started at the state its own step ended on, it reproduces everything the step left.
    Returns (per-quantity max relative deviation, device (q, v, a))."""
    name, env, want = next(p for p in PATHS if p[0] == path)
    robot, opt = probe_options(solver)
    rng = np.random.default_rng(seed)
    q, v, _ = full_range_states(robot, n_env, rng)
    cmd = over_limit_commands(robot, n_env, rng)
    v = clean_velocities(robot, opt, q, v, cmd, step_dt)
    with switches(env):
        eng = BatchedEngine(robot, opt, n_env, api_=api)
    desc = eng.describe()
    assert want in desc, (path, desc)
    orc = OracleBatch(robot, opt, n_env)
    for x in (eng, orc):
        x.set_command(cmd)
    eng.start(q, v)
    assert not orc.start(q, v).any()
    eng.step(step_dt)
    assert not orc.step(step_dt, parallel=True).any()
    # nothing left the hot path: no bound reached (the constraint path would take over), nothing diverged
    np.testing.assert_array_equal(eng.get_status(), 0)
    np.testing.assert_array_equal(orc.get_status(), 0)

    # premise, on the oracle: what a step leaves in `a`, the efforts and the contact forces is the evaluation at its
    # final state, bit for bit
    _, q0, v0, a0 = orc.get_state()
    stepped = _outputs(orc)
    for k, x in zip(("a", "f_external", "u"), OracleBatch(robot, opt, n_env).compute_dynamics(q0, v0, cmd)):
        np.testing.assert_array_equal(x, stepped[k], err_msg=f"premise: {k}")
    # ... and a restart there reproduces everything else the step left, in the envs where the restart reproduces `a`.
    # `start` renormalises the free-flyer quaternion, an ulp that a foot deep in the 4e6 N/m ground can amplify to
    # 1e-12 of the accelerations; and it refuses a state with a contact force above 1e5 N.  Those envs are compared on
    # the outputs of `compute_dynamics` (a, u, contact forces) only.
    usable = _restart_reference(robot, opt, cmd, q0, v0, a0, min_share=0.75)[1]
    for k, x in _restart_reference(robot, opt, cmd, q0, v0, a0)[0].items():
        e = rel_dev(x[usable], stepped[k][usable])
        assert e <= 1e-13, f"premise: {k} of a restart at the final state deviates by {e:.3e}"

    # the device's last evaluation against the oracle's at the device's final state
    _, q1, v1, a1 = eng.get_state()
    a_ref, f_ref, u_ref = OracleBatch(robot, opt, n_env).compute_dynamics(q1, v1, cmd)
    want_out, usable = _restart_reference(robot, opt, cmd, q1, v1, a_ref, min_share=0.75)
    got = _outputs(eng)
    dev = {}
    for k, x0 in want_out.items():
        e = rel_dev(got[k], {"a": a_ref, "f_external": f_ref, "u": u_ref}[k]) if k in ("a", "f_external", "u") else \
            rel_dev(got[k][usable], x0[usable])
        dev[k] = e
        assert e <= tol, f"{path} / {solver}: {k} deviates by {e:.3e} relative"
    return dev, (q1, v1, a1)


def _restart_reference(robot, opt, cmd, q, v, a, min_share=0.75):
    """The oracle started at (q, v): its outputs, and the envs where it reproduces the evaluation `a` at (q, v) to 1e-14."""
    ref = OracleBatch(robot, opt, len(q))
    ref.set_command(cmd)
    ok = ref.start(q, v) == 0
    out = _outputs(ref)
    usable = ok & (np.abs(out["a"] - a).max(axis=1) <= 1e-14 * np.maximum(1.0, np.abs(a).max(axis=1)))
    assert usable.mean() >= min_share, f"only {usable.sum()} of {len(q)} envs can be restarted at their final state"
    return out, usable
