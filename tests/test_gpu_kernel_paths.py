"""Every evaluation path on the B200 against the oracle over the full joint range (`pytest -m gpu`), and the scenarios
that tests/test_kernel_emul.py runs under the warp emulator, on real warps (nvcc's multiply-add contraction, the CUDA
library's sin / cos, real shuffles and votes)."""
import json
import os

import numpy as np
import pytest

from jiminy_b200 import robots as R
from jiminy_b200.core import BatchedEngine
from oracle.oracle import OracleBatch

import kernel_paths_common as kpc
import parity_common as pc
import test_kernel_emul as tke

pytestmark = pytest.mark.gpu

def _record(name, data):
    """Measured deviations, printed and, when JB_DEVIATIONS_DIR names a directory, kept there as JSON."""
    print(name, json.dumps(data))
    out = os.environ.get("JB_DEVIATIONS_DIR")
    if out and os.path.isdir(out):
        with open(os.path.join(out, f"kernel_paths_{name}.json"), "w") as fh:
            json.dump(data, fh, indent=1)


@pytest.mark.parametrize("n_env", [4096, 4093])
@pytest.mark.parametrize("solver", ["euler_explicit", "runge_kutta_4"])
def test_hot_path_evaluation_matches_oracle_on_device(n_env, solver):
    """Every path (default composite-rigid-body hot path, ABA sweeps, dynamic plan, per-lane descriptors, full kernel
    only, one and two lanes per env): one evaluation at the device's final state against the oracle, all envs; and the
    paths end their step in the same state."""
    devs, states, failures = {}, {}, []
    for path in kpc.PATH_NAMES:
        try:
            devs[path], states[path] = kpc.hot_path_probe(None, path, solver, n_env)
        except AssertionError as e:
            failures.append(f"{path}: {e}")
    cross = {}
    if "crba" in states:
        for path, st in states.items():
            cross[path] = {k: kpc.rel_dev(x1, x0) for k, x1, x0 in zip(("q", "v"), st, states["crba"])}
            worst = max(cross[path].values())
            if worst > kpc.PATH_TOL:
                failures.append(f"{path} differs from the default path by {worst:.3e}")
    _record(f"{solver}_{n_env}", {"vs_oracle": devs, "vs_default_path": cross,
                                  "max_vs_oracle": {p: max(d.values()) for p, d in devs.items()}})
    assert not failures, failures


@pytest.mark.parametrize("name", R.ROBOT_NAMES)
def test_full_range_compute_dynamics_on_device(name):
    """The full-range sampler (joint angles over their own bounds and on multiples of pi/4, tilted base, none / some / all
    feet in the ground, fast joints, saturated motors) through `compute_dynamics` at the automatic lane plan."""
    robot, opt = R.load_robot(name)
    opt = R.baseline_options(name, opt)
    rng = np.random.default_rng(11)
    n = 100
    q, v, _ = kpc.full_range_states(robot, n, rng)
    cmd = kpc.over_limit_commands(robot, n, rng)
    with kpc.switches({}):
        eng = BatchedEngine(robot, opt, n)
    a1, f1, u1 = eng.compute_dynamics(q, v, cmd)
    a0, f0, u0 = OracleBatch(robot, opt, n).compute_dynamics(q, v, cmd)
    dev = {k: kpc.rel_dev(x1, x0) for k, x1, x0 in (("a", a1, a0), ("f_external", f1, f0), ("u", u1, u0))}
    _record(f"compute_dynamics_{name}", dev)
    assert max(dev.values()) <= kpc.RHS_TOL, dev


def test_structured_quadruped_solver_without_uniform_warps(monkeypatch):
    """JB_NO_UNIFORM_SOLVER=1: the structured quadruped contact solver uses its group-masked collectives even when the
    whole warp is converged (the path the emulator always takes, never run on a real warp by the rest of the suite)."""
    with kpc.switches({"JB_NO_UNIFORM_SOLVER": "1"}):
        eng, orc, sc = pc.robot_constraint_scenario("anymal", 40, 3, seed=2)
    assert "structured quadruped solver" in eng.describe()
    assert (eng.get_state()[1][:, 2] > 0.4).all()


# ---- bodies of tests/test_kernel_emul.py on the CUDA library (api=None).  They set JB_LANES through os.environ and reset
# it on success only: `switches` restores the environment whatever happens.
@pytest.mark.parametrize("name,lanes", [("anymal", 1), ("anymal", 2), ("atlas", 8)])
def test_single_rhs_matches_oracle_on_device(name, lanes):
    with kpc.switches({}):
        tke.test_single_rhs_matches_oracle(None, name, lanes)


@pytest.mark.parametrize("body", ["test_all_joint_models_and_internal_branching", "test_dopri_free_flyer_contact_and_unbounded_joint",
                                  "test_masked_restart_and_odd_env_count", "test_status_flags", "test_anymal_torque_mode_euler",
                                  "test_constraint_contact_on_trunk_body", "test_compute_dynamics_leaves_the_running_state_alone",
                                  "test_centroidal_terms_of_a_massless_subtree_are_finite", "test_flexibility_on_a_trunk_joint_of_atlas"])
def test_emulator_scenario_on_device(body):
    fn = getattr(tke, body)
    with kpc.switches({}):
        if body == "test_constraint_contact_on_trunk_body":
            fn(None, False, "lane-block")
            fn(None, True, "body-space")
        else:
            fn(None)


@pytest.mark.parametrize("toggle", [None, "JB_NO_STRUCTURED_CONS"])
def test_external_forces_with_constraint_contacts_on_device(monkeypatch, toggle):
    with kpc.switches({}):
        tke.test_external_forces_with_constraint_contacts(None, monkeypatch, toggle)


@pytest.mark.parametrize("lanes,toggle,solver", [(0, None, "body-space"), (0, "JB_NO_BODY_CONS", "lane-block"), (1, None, "generic")])
def test_constraint_contacts_all_joint_models_on_device(monkeypatch, lanes, toggle, solver):
    with kpc.switches({}):
        tke.test_constraint_contacts_all_joint_models(None, monkeypatch, lanes, toggle, solver)


@pytest.mark.parametrize("robot", ["atlas", "anymal"])
def test_dopri_with_constraint_contacts_on_device(robot):
    with kpc.switches({}):
        tke.test_dopri_with_constraint_contacts(None, robot)
