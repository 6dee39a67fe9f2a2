"""Cases of the axis-constrained plane models (SACMODEL_PERPENDICULAR_PLANE / SACMODEL_PARALLEL_PLANE): the axis test of
k_plane_score and plane_ransac_run (cm_plane.cu, cm_api.cu) at its decision boundaries, NaN models, searches where no
model passes, refits that leave the cone, settings that constrain nothing, degenerate axes and multi-cloud mixes.

A case is a dict like tests/plane_edges.py's (clouds, threshold, probability, max_iterations, seed, orders, optimizes)
plus model, axis, eps_angle. Boundary angles come from the numpy restatement (tests/plane_axis_np.py) of one draw's d."""
from __future__ import annotations

import math

import numpy as np

import plane_axis_oracle as PO
import plane_edges as P
from oracle import np_oracle as NP
import plane_axis_np as N

F32 = np.float32
PLANE, PERP, PAR = 0, 1, 2
TEN_DEG = math.radians(10.0)
Z = (0.0, 0.0, 1.0)


def case(name, clouds, model, eps, axis=Z, thr=0.3, prob=0.99, max_it=1000, seed=12345, orders=(0,), optimizes=(False, True),
         **kw):
    d = P._case(name, clouds, thr=thr, prob=prob, max_it=max_it, seed=seed, orders=orders, optimizes=optimizes, **kw)
    d.update(model=int(model), axis=tuple(float(v) for v in axis), eps_angle=float(eps))
    return d


def wall_zone(n_ground=600, n_wall=1200, n_clutter=300, seed=0, tilt=0.01, wall_x=6.0):
    """A ground zone (z = -1.8 + tilt * x, +-2 cm) whose wall (x = wall_x) holds more points than the ground."""
    rng = np.random.default_rng(seed)
    g = np.zeros((n_ground, 4), F32)
    g[:, 0] = rng.uniform(-6, 6, n_ground); g[:, 1] = rng.uniform(-4, 4, n_ground)
    g[:, 2] = -1.8 + tilt * g[:, 0] + rng.uniform(-0.02, 0.02, n_ground)
    w = np.zeros((n_wall, 4), F32)
    w[:, 0] = wall_x + rng.uniform(-0.02, 0.02, n_wall); w[:, 1] = rng.uniform(-4, 4, n_wall)
    w[:, 2] = rng.uniform(-1.7, 0.3, n_wall)
    c = np.zeros((n_clutter, 4), F32)
    c[:, 0] = rng.uniform(-6, 6, n_clutter); c[:, 1] = rng.uniform(-4, 4, n_clutter); c[:, 2] = rng.uniform(-1.5, 0.3, n_clutter)
    x = np.concatenate([g, w, c])
    x[:, 3] = rng.uniform(0, 255, len(x))
    return np.ascontiguousarray(x[rng.permutation(len(x))])


def walls_only(n=800, seed=1):
    """One exactly vertical wall (x = 5) and nothing else: every plane through three of its points has the normal
    (+-a, 0, 0), 90 degrees from z."""
    rng = np.random.default_rng(seed)
    x = np.zeros((n, 4), F32)
    x[:, 0] = 5.0
    x[:, 1] = rng.uniform(-4, 4, n)
    x[:, 2] = rng.uniform(-2, 2, n)
    x[:, 3] = 1.0
    return x


def nan_zone(seed=2, share=0.3):
    x = wall_zone(500, 300, 100, seed=seed)
    rng = np.random.default_rng(seed)
    bad = rng.random(len(x)) < share
    x[bad, rng.integers(0, 3, int(bad.sum()))] = np.nan
    return x


def first_good_draws(x, seed, order, count):
    """(draw index, model) of the first `count` good draws of PCL's sampler on x."""
    out = []
    s = P.draw_stream(len(x), seed, 4 * count + 8)
    for j, (a, b, c) in enumerate(s):
        good, m = NP.plane_of_sample(x[a], x[b], x[c], order)
        if good:
            out.append((j, m))
        if len(out) == count:
            break
    return out


def prev_double(v):
    return float(np.nextafter(np.float64(v), -np.inf))


def parallel_eps_for(d_abs):
    """The smallest double eps in (0, pi/2] with |sin(eps)| >= d_abs (libm sin): sin_angle_ just reaches |d|."""
    lo, hi = 0.0, math.pi / 2
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        if mid in (lo, hi):
            break
        if abs(math.sin(mid)) >= d_abs:
            hi = mid
        else:
            lo = mid
    e = hi
    while abs(math.sin(prev_double(e))) >= d_abs:   # libm sin may be flat over a few doubles
        e = prev_double(e)
    return e


def boundary_cases():
    """eps at one draw's own PCL angle (it passes) and one double below (it fails). PERPENDICULAR: one draw with d > 0
    (decided by c_pos) and one with d < 0 (decided by c_neg), each a draw whose d after getAngle3D's second normalize
    differs from d after one, so that the second normalize decides one of the two eps (about 1 % of the draws do)."""
    cases = []
    x = wall_zone(seed=11)
    for order in (0, 1, 2):
        draws = first_good_draws(x, 12345, order, 4000)
        for sign, tag_s in ((1, "pos"), (-1, "neg")):
            pick = None
            for j, m in draws:
                d2, d1 = N.plane_axis_dot(m, PERP, Z, order), N.plane_axis_dot(m, PAR, Z, order)
                if d1 != d2 and sign * float(d2) > 0 and N.perpendicular_angle(d2) < 1.2:
                    pick = (j, d2)
                    break
            assert pick is not None, "no draw of the scene separates one normalize from two (order %d, %s)" % (order, tag_s)
            j, d = pick
            a = N.perpendicular_angle(d)
            for tag, eps in (("at", a), ("below", prev_double(a))):
                cases.append(case("A-bound:perp:%d:%s:%s" % (order, tag_s, tag), [x], PERP, eps, prob=1.0, max_it=j + 5,
                                  orders=(order,), draw=j, draw_valid=(tag == "at"), draw_sign=sign))
        # parallel: sin_angle_ brackets |d| of a draw of the wall (normal near x: |d| small)
        for j, m in draws:
            dp = abs(float(N.plane_axis_dot(m, PAR, Z, order)))
            if 0.01 < dp < 0.5:
                break
        e = parallel_eps_for(dp)
        for tag, eps in (("at", e), ("below", prev_double(e))):
            cases.append(case("A-bound:par:%d:%s" % (order, tag), [x], PAR, eps, prob=1.0, max_it=j + 5, orders=(order,),
                              draw=j, draw_valid=(tag == "at")))
    return cases


def nan_cases():
    x = nan_zone()
    return [case("A-nan:%d" % m, [x], m, TEN_DEG, prob=1.0, max_it=200, orders=(0, 1, 2)) for m in (PERP, PAR)]


def none_valid_cases():
    """PERPENDICULAR at 10 degrees on walls only: every draw fails, k stays huge, the search runs to the cap."""
    x = walls_only()
    return [case("A-none:%d" % it, [x], PERP, TEN_DEG, max_it=it, optimizes=(False, True), no_valid=True)
            for it in (31, 32, 287, 288, 1000, 1311, 1312)]


def refit_cone_cases():
    """eps between the RANSAC model's angle and the refitted model's angle: the refit leaves the cone."""
    cases = []
    for seed in range(40):
        rng = np.random.default_rng(500 + seed)
        n = 600
        x = np.zeros((n, 4), F32)
        x[:, 0] = rng.uniform(-10, 10, n); x[:, 1] = rng.uniform(-10, 10, n)
        x[:, 2] = 0.17 * x[:, 0] + rng.uniform(-0.25, 0.25, n)
        x[:, 3] = 1.0
        r = PO.plane_ransac_model(x, 0.3, 0.99, 1000, True, 12345, 0, PLANE)
        ar = N.perpendicular_angle(N.plane_axis_dot(r["coeff_ransac"], PERP, Z, 0))
        af = N.perpendicular_angle(N.plane_axis_dot(r["coeff"], PERP, Z, 0))
        if ar < af:
            cases.append(case("A-refit:%d" % seed, [x], PERP, 0.5 * (ar + af), optimizes=(True,), refit_leaves=True))
        if len(cases) == 2:
            break
    return cases


def unconstrained_cases():
    """Settings that constrain nothing: results bit-identical to SACMODEL_PLANE (and 0 rejected)."""
    x = wall_zone(seed=21)
    out = []
    for m, eps in ((PERP, 0.0), (PERP, -0.1), (PERP, float("nan")), (PERP, math.pi / 2), (PERP, 2.0), (PERP, 1e300),
                   (PAR, 0.0), (PAR, -0.1), (PAR, float("nan")), (PLANE, TEN_DEG), (PLANE, float("nan"))):
        out.append(case("A-free:%d:%r" % (m, eps), [x], m, eps, orders=(0, 1, 2), same_as_plane=True))
    out.append(case("A-free:plane-axis", [x], PLANE, TEN_DEG, axis=(1e-30, 7.0, float("nan")), same_as_plane=True))
    return out


def axis_cases():
    x = wall_zone(seed=31)
    out = []
    for name, ax in (("zero", (0.0, 0.0, 0.0)), ("long", (0.0, 0.0, 5.0)), ("tilted", (0.3, 0.1, 2.0)),
                     ("underflow", (0.0, 0.0, 1e-30)), ("x", (1.0, 0.0, 0.0))):
        for m in (PERP, PAR):
            out.append(case("A-axis:%s:%d" % (name, m), [x], m, TEN_DEG, axis=ax, orders=(0, 2)))
    return out


def multi_cases():
    e = np.zeros((0, 4), F32)
    clouds = [wall_zone(seed=41), walls_only(500, 42), e, nan_zone(43), wall_zone(300, 100, 50, seed=44),
              P.ground(2, 45, 1.0), P.ground(1500, 46, 0.7), wall_zone(200, 900, 100, seed=47)]
    return [case("A-multi:%d" % m, clouds, m, TEN_DEG, max_it=1400) for m in (PERP, PAR)]


def axis_plane_cases() -> dict:
    out = {}
    for c in boundary_cases() + nan_cases() + none_valid_cases() + refit_cone_cases() + unconstrained_cases() + axis_cases() + multi_cases():
        out[c["name"]] = c
    return out
