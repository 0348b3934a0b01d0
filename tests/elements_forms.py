"""Host restatement of the element-set branches of satellite_function.py that the C oracle does not cover, and the seeded
inputs that land exactly on each branch. Test infrastructure only.

calculate_orbital_elements (:161-255) is oracle.orbital_elements on every branch: it returns 6 elements
[a, e, i, omega, Omega, f], 5 on the parabolic branch (energy == 0) [p, i, omega, Omega, f], or 4 on the circular branch
(e == 0) [a, i, u, Omega]. calculate_state_information (:257-315) takes the six-element form (oracle.state_information)
and the two forms those branches return. The 5- and 4-element forms below run the six-element form's tail (:303-315) with
e = 1 and the given p, or with e = 0, p = a and the given argument of latitude u (omega = 0, f = u).

The arithmetic is python floats and the `math` module, i.e. individually rounded IEEE operations and the host libm's
sin, cos and pow, the same calls the reference makes and the C oracle makes (compiled with -ffp-contract=off).
"""
from __future__ import annotations

import math

import numpy as np

MU = 3.986e14


def _div(a, b):
    """IEEE a / b (python floats raise on b == 0; numpy scalars give +-inf / nan like the device)"""
    with np.errstate(divide="ignore", invalid="ignore"):
        return float(np.float64(a) / np.float64(b))


def state_from_form(el, miu=MU):
    """calculate_state_information(el, miu) for len(el) == 5 or 4 -> (R[3], V[3])."""
    el = [float(x) for x in el]
    if len(el) == 5:
        p, i, omega, Omega, f = el
        e = 1.0
        u = omega + f
    elif len(el) == 4:
        a, i, u, Omega = el
        e, p, omega, f = 0.0, a, 0.0, u
    else:
        raise ValueError("the 5- and 4-element forms only; the six-element form is oracle.state_information")
    k = _div(p, 1 + e * math.cos(f))                                            # :303
    R = [k * (math.cos(Omega) * math.cos(u) - math.sin(Omega) * math.sin(u) * math.cos(i)),
         k * (math.sin(Omega) * math.cos(u) + math.cos(Omega) * math.sin(u) * math.cos(i)),
         k * (math.sin(i) * math.sin(u))]
    s = math.pow(_div(miu, p), 0.5)                                             # :309
    V = [s * (-math.cos(Omega) * (math.sin(u) + e * math.sin(omega))
              - math.sin(Omega) * (math.cos(u) + e * math.cos(omega)) * math.cos(i)),
         s * (-math.sin(Omega) * (math.sin(u) + e * math.sin(omega))
              + math.cos(Omega) * (math.cos(u) + e * math.cos(omega)) * math.cos(i)),
         s * (math.sin(i) * (math.cos(u) + e * math.cos(omega)))]
    return np.array(R), np.array(V)


def states_from_forms(el, miu=MU):
    """[n, 5] or [n, 4] -> [n, 6] (R, V)."""
    return np.array([np.concatenate(state_from_form(row, miu)) for row in np.asarray(el, dtype=np.float64)])


def elements_padded(oracle, rv, miu=MU):
    """oracle.orbital_elements on rows rv [n, 6] -> (elements [n, 6] zero-padded, kind [n] = number of elements)."""
    rv = np.asarray(rv, dtype=np.float64)
    out = np.zeros((len(rv), 6))
    kind = np.zeros(len(rv), dtype=np.int32)
    for k, row in enumerate(rv):
        el = oracle.orbital_elements(miu, row[:3], row[3:])
        out[k, :len(el)] = el
        kind[k] = len(el)
    return out, kind


# ---------------------------------------------------------------------------------------------------- seeded inputs
def _axis_state(rng, r, v, phi, equatorial):
    """R = r on one coordinate axis (random sign); V of speed v perpendicular to it, at angle phi in the plane of the other
    two axes (equatorial: R and V both in the x-y plane). np.dot(R, V) is then exactly zero."""
    if equatorial:
        ax = int(rng.integers(0, 2))
        R = np.zeros(3); R[ax] = r * rng.choice([-1.0, 1.0])
        V = np.zeros(3); V[1 - ax] = v * rng.choice([-1.0, 1.0])
        return np.concatenate([R, V])
    ax = int(rng.integers(0, 3))
    others = [k for k in range(3) if k != ax]
    R = np.zeros(3); R[ax] = r * rng.choice([-1.0, 1.0])
    V = np.zeros(3); V[others[0]] = v * math.cos(phi); V[others[1]] = v * math.sin(phi)
    return np.concatenate([R, V])


def _search(rng, oracle, want, n, make, max_tries=200000):
    rows = []
    tries = 0
    while len(rows) < n:
        tries += 1
        assert tries < max_tries, f"found {len(rows)} of {n} rows on the {want}-element branch"
        rv = make()
        if rv is not None and len(oracle.orbital_elements(MU, rv[:3], rv[3:])) == want:
            rows.append(rv)
    return np.array(rows)


def circular_states(rng, oracle, n, equatorial=False):
    """states on the circular branch (e == 0 exactly): v_norm ** 2 / miu == 1 / r_norm in floating point and r.v == 0."""
    def make():
        r = rng.uniform(6.6e6, 4.3e7)
        v = math.sqrt(MU / r) * (1 + int(rng.integers(-2, 3)) * 2.0 ** -52)
        return _axis_state(rng, r, v, rng.uniform(0.05, 2 * math.pi - 0.05), equatorial)
    return _search(rng, oracle, 4, n, make)


def parabolic_states(rng, oracle, n):
    """states on the parabolic branch (energy == 0 exactly). Half of them axis-aligned with v = sqrt(2 miu / r) exactly
    representable (r = 2 miu / v**2 for a short-mantissa v), half at a random flight-path angle."""
    def make():
        if rng.random() < 0.5:
            v = float(int(rng.integers(2000, 11000)))                # v ** 2 exact
            r = 2 * MU / v ** 2
            return _axis_state(rng, r, v, rng.uniform(0.05, 2 * math.pi - 0.05), False)
        r = rng.uniform(6.6e6, 4.3e7)
        v = math.sqrt(2 * MU / r) * (1 + int(rng.integers(-2, 3)) * 2.0 ** -52)
        d = rng.normal(size=3)
        R = r * d / np.linalg.norm(d)
        w = rng.normal(size=3)
        return np.concatenate([R, v * w / np.linalg.norm(w)])
    return _search(rng, oracle, 5, n, make)


def near_miss_states(oracle, circ, para):
    """each branch state with its largest velocity component moved by the fewest ulps (up and down) that make the branch's
    equality test fail: six-element states as close to the circular / parabolic branches as doubles allow."""
    out = []
    for rv in np.concatenate([circ, para]):
        k = int(np.argmax(np.abs(rv[3:]))) + 3
        for d in (np.inf, -np.inf):
            x = rv.copy()
            for _ in range(64):
                x[k] = np.nextafter(x[k], d)
                if len(oracle.orbital_elements(MU, x[:3], x[3:])) == 6:
                    out.append(x)
                    break
    return np.array(out)


def general_states(rng, n):
    """near-GEO states like the env's (six-element branch)."""
    return np.concatenate([np.array([27098000.0, 32306000.0, 0.0]) + rng.normal(0, 1e5, (n, 3)),
                           np.array([-2350.0, 1970.0, 0.0]) + rng.normal(0, 20, (n, 3))], axis=1)


def five_forms(rng, n):
    """[p, i, omega, Omega, f] with the special angles 0, pi/2, pi mixed in."""
    p = rng.uniform(6.6e6, 5e7, n)
    ang = rng.uniform(0, 2 * math.pi, (n, 4))
    ang[:, 0] /= 2                                                          # i in [0, pi)
    special = rng.random((n, 4)) < 0.1
    ang[special] = rng.choice([0.0, math.pi / 2, math.pi], size=int(special.sum()))
    ang[:, 3] = np.where(np.abs(ang[:, 3] - math.pi) < 1e-3, 1.0, ang[:, 3])   # 1 + cos(f) == 0 at f = pi
    return np.concatenate([p[:, None], ang], axis=1)


def four_forms(rng, n):
    """[a, i, u, Omega] with the special angles 0, pi/2, pi mixed in."""
    a = rng.uniform(6.6e6, 5e7, n)
    ang = rng.uniform(0, 2 * math.pi, (n, 3))
    ang[:, 0] /= 2
    special = rng.random((n, 3)) < 0.1
    ang[special] = rng.choice([0.0, math.pi / 2, math.pi], size=int(special.sum()))
    return np.concatenate([a[:, None], ang], axis=1)


def exact_round_trip_forms(rng, oracle, n_el, n):
    """5- or 4-element sets [x, i, 0, 0, (0)] (random x and inclination) whose state lies exactly on the branch they came
    from, so that the way back returns n_el finite elements (the oracle decides)."""
    rows = []
    while len(rows) < n:
        el = [rng.uniform(6.6e6, 5e7), rng.uniform(0.05, math.pi - 0.05)] + [0.0] * (n_el - 2)
        R, V = state_from_form(el)
        back = oracle.orbital_elements(MU, R, V)
        if len(back) == n_el and np.all(np.isfinite(back)):
            rows.append(el)
    return np.array(rows)
