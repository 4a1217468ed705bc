"""Every evaluation path of the kernel source against the oracle over the full joint range (warp emulator of tests/emul),
and the accuracy of the hot path's inline sin / cos.  The same probe runs on the B200 in tests/test_gpu_kernel_paths.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from jiminy_b200 import robots as R
from oracle.oracle import OracleBatch

from emul import emul_api
import kernel_paths_common as kpc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_ENV = 9          # ANYmal: 8 envs per warp at the automatic plan, 16 at two lanes, 32 at one -- the last warp is partial


@pytest.fixture(scope="module")
def api():
    return emul_api()


def test_sampler_covers_the_full_range():
    """Inside the bounds; every quadrant of ANYmal's +-9.42 rad joints; angles on multiples of pi/4; none / some / all
    feet in the ground; velocities beyond the motors' velocity limits; commands beyond their effort limits."""
    robot, opt = kpc.probe_options("euler_explicit")
    rng = np.random.default_rng(0)
    q, v, modes = kpc.full_range_states(robot, 300, rng)
    qj = q[:, 7:]
    assert (qj >= robot.q_lower[7:]).all() and (qj <= robot.q_upper[7:]).all()
    np.testing.assert_allclose(np.linalg.norm(q[:, 3:7], axis=1), 1.0, atol=1e-15)
    wide = robot.q_upper[7:] > 9.0
    assert set(np.floor(qj[:, wide] / (np.pi / 2)).astype(int).ravel()) == set(range(-6, 6))
    off = np.abs(qj - np.round(qj / (np.pi / 4)) * (np.pi / 4))
    assert (off[:, wide] <= 1e-9).sum() > 100 and (np.abs(np.round(qj / (np.pi / 4))) >= 9).any()
    depth = np.array([[p.p[2] for p in R.frame_placements(robot, x, robot.contact_frame_names).values()] for x in q])
    touching = (depth < 0).sum(axis=1)
    for mode, want in (("none", {0}), ("some", {1, 2, 3}), ("all", {4})):
        assert set(touching[np.array(modes) == mode]) <= want
    assert (-depth.min(axis=1) < 3e-3).all()                     # no foot deeper than 2 mm (plus level error)
    vlim = np.array([m.velocity_limit for m in robot.motors])
    assert (np.abs(v[:, 6:]) > vlim).mean() > 0.5
    cmd = kpc.over_limit_commands(robot, 300, rng)
    assert (np.abs(cmd) > np.array([m.effort_limit for m in robot.motors])).mean() > 0.25
    v2 = kpc.clean_velocities(robot, opt, q, v, cmd, 2e-3)       # nearly all of them start and step as drawn
    assert (v2 == v).all(axis=1).mean() > 0.9


@pytest.mark.parametrize("solver", ["euler_explicit", "runge_kutta_4"])
@pytest.mark.parametrize("path", kpc.PATH_NAMES)
def test_hot_path_evaluation_matches_oracle(api, path, solver):
    """One evaluation of each path (the composite-rigid-body hot path by default) against the oracle at the state the
    device's step ended on: accelerations, efforts, contact forces, extra terms, centroidal terms, sensors."""
    dev, _ = kpc.hot_path_probe(api, path, solver, N_ENV)
    print(path, solver, " ".join(f"{k}={x:.1e}" for k, x in dev.items()))


@pytest.mark.parametrize("solver", ["euler_explicit", "runge_kutta_4"])
def test_kernel_paths_agree(api, solver):
    """The paths are reformulations of the same step: from the same full-range states they end in the same state."""
    _, base = kpc.hot_path_probe(api, "crba", solver, N_ENV)
    for path in kpc.PATH_NAMES[1:]:
        _, other = kpc.hot_path_probe(api, path, solver, N_ENV)
        for name, x1, x0 in zip(("q", "v"), other, base):
            e = kpc.rel_dev(x1, x0)
            assert e <= kpc.PATH_TOL, f"{path} / {solver}: {name} differs from the default path by {e:.3e}"


def test_switches_never_leak():
    """A failing body must not leave a switch behind for the next test."""
    os.environ.pop("JB_LANES", None)
    with pytest.raises(RuntimeError):
        with kpc.switches({"JB_LANES": "1"}):
            assert os.environ["JB_LANES"] == "1"
            raise RuntimeError
    assert "JB_LANES" not in os.environ


# ---- jb_sincos: the inline sin / cos of the hot path's joint angles
@pytest.fixture(scope="module")
def jb_sincos(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("sincos") / "jb_sincos_harness.so")
    subprocess.run(["/usr/bin/g++", "-O2", "-std=c++20", "-fPIC", "-shared", "-ffp-contract=off", "-DJB_HOST_EMUL=1",
                    "-I", os.path.join(ROOT, "tests", "emul"), "-I", os.path.join(ROOT, "jiminy_b200", "csrc"),
                    os.path.join(ROOT, "tests", "emul", "jb_sincos_harness.cpp"), "-o", lib], check=True)
    dll = C.CDLL(lib)
    P = C.POINTER(C.c_double)
    dll.jb_sincos_array.argtypes = [P, P, P, C.c_longlong]

    def f(x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        s, c = np.empty_like(x), np.empty_like(x)
        dll.jb_sincos_array(x.ctypes.data_as(P), s.ctypes.data_as(P), c.ctypes.data_as(P), x.size)
        return s, c
    return f


def _ulps(got, ref):
    """|got - ref| in units of the spacing of doubles at ref (ref in long double)."""
    r = np.abs(ref.astype(np.float64))
    return (np.abs(got.astype(np.longdouble) - ref) / np.spacing(r).astype(np.longdouble)).astype(np.float64)


@pytest.mark.skipif(np.finfo(np.longdouble).nmant < 63, reason="needs the x86 80-bit long double as the reference")
def test_jb_sincos_is_within_two_ulp(jb_sincos):
    """`jb_sincos` (jb_device.cuh) against sin / cos in long double: <= 2 ulp of double (DESIGN.md: <= 1.6 ulp over
    +-1e5 rad).  The function is built for the host with -ffp-contract=off from the unchanged device source; it is
    written with explicit fma(), products and exact subtractions only, so this build computes the device's bits.
    Sets: a dense grid over +-10 rad (ANYmal's joint range), the doubles nearest k pi/4 for |k| <= 1.3e5 (quadrant and
    octant boundaries, where the Cody-Waite reduction cancels), 1e6 seeded uniform points over +-1e5 rad, and +-0,
    subnormals and |x| < 2^-26."""
    pi = 4 * np.arctan(np.longdouble(1))
    k = np.arange(-130000, 130001).astype(np.longdouble)
    tiny = np.geomspace(5e-324, 2.0 ** -26, 2000)
    sets = {"grid +-10 rad": np.linspace(-10.0, 10.0, 2_000_001),
            "k pi/4": (k * pi / 4).astype(np.float64),
            "uniform +-1e5 rad": np.random.default_rng(0).uniform(-1e5, 1e5, 1_000_000),
            "0, subnormals, |x| < 2^-26": np.concatenate([[0.0, -0.0, 5e-324, -5e-324, 2.225e-308], tiny, -tiny])}
    worst = {}
    for name, x in sets.items():
        s, c = jb_sincos(x)
        xl = x.astype(np.longdouble)
        es, ec = _ulps(s, np.sin(xl)), _ulps(c, np.cos(xl))
        worst[name] = (float(es.max()), float(ec.max()))
        i = int(np.argmax(np.maximum(es, ec)))
        print(f"jb_sincos, {name}: max error sin {es.max():.3f} ulp, cos {ec.max():.3f} ulp (x = {x[i]!r})")
        assert es.max() <= 2.0 and ec.max() <= 2.0, (name, x[i], es[i], ec[i])
    print("jb_sincos: largest error found", max(max(w) for w in worst.values()), "ulp")
    tiny_x = sets["0, subnormals, |x| < 2^-26"]
    np.testing.assert_array_equal(jb_sincos(tiny_x)[0], tiny_x)  # sin x = x below 2^-26, exactly (up to the sign of 0)


# ---- the full-range sampler through the full kernel's `compute_dynamics`, every BASELINE robot
@pytest.mark.parametrize("name", R.ROBOT_NAMES)
def test_full_range_compute_dynamics(api, name):
    robot, opt = R.load_robot(name)
    opt = R.baseline_options(name, opt)
    rng = np.random.default_rng(11)
    n = 6
    q, v, _ = kpc.full_range_states(robot, n, rng)
    cmd = kpc.over_limit_commands(robot, n, rng)
    from jiminy_b200.core import BatchedEngine
    with kpc.switches({}):
        eng = BatchedEngine(robot, opt, n, api_=api)
    a1, f1, u1 = eng.compute_dynamics(q, v, cmd)
    a0, f0, u0 = OracleBatch(robot, opt, n).compute_dynamics(q, v, cmd)
    for k, x1, x0 in (("a", a1, a0), ("f_external", f1, f0), ("u", u1, u0)):
        assert kpc.rel_dev(x1, x0) <= kpc.RHS_TOL, (k, kpc.rel_dev(x1, x0))
