"""The host restatement of calculate_orbital_elements' circular / parabolic branches (oracle.orbital_elements) and of the
5- and 4-element forms of calculate_state_information (tests/elements_forms.py), pinned against the reference
(tests/golden/elements_branches_golden.npz, written by make_golden_branches.py from the upstream reference) and checked for
consistency with the six-element form. CPU only."""
import math
import os

import numpy as np
import pytest

import elements_forms as F

FIXTURE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "elements_branches_golden.npz")
needs_fixture = pytest.mark.skipif(not os.path.exists(FIXTURE),
                                   reason="elements_branches_golden.npz not recorded (make_golden_branches.py)")


def same_bits(a, b):
    """bit-identical, NaN matching NaN (the circular equatorial u is 0 / 0 in the reference too)"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(np.all((a.view(np.int64) == b.view(np.int64)) | (np.isnan(a) & np.isnan(b))))


@needs_fixture
def test_orbital_elements_branches_match_reference(golden, oracle):
    g = golden("elements_branches_golden.npz")
    el, kind = F.elements_padded(oracle, g["rv"])
    assert np.array_equal(kind, g["kind"])
    assert set(np.unique(kind)) == {4, 5, 6}
    for k in range(len(kind)):
        assert same_bits(el[k, :kind[k]], g["elements"][k, :kind[k]]), (k, el[k], g["elements"][k])


@needs_fixture
@pytest.mark.parametrize("n_el", [5, 4])
def test_state_information_forms_match_reference(golden, n_el):
    g = golden("elements_branches_golden.npz")
    assert same_bits(F.states_from_forms(g[f"form{n_el}"]), g[f"state{n_el}"])


def test_generated_states_take_the_intended_branch(oracle):
    rng = np.random.default_rng(5)
    circ, circ_eq, para = F.circular_states(rng, oracle, 16), F.circular_states(rng, oracle, 8, True), F.parabolic_states(rng, oracle, 16)
    assert list(F.elements_padded(oracle, circ)[1]) == [4] * 16
    el_eq, k_eq = F.elements_padded(oracle, circ_eq)
    assert list(k_eq) == [4] * 8 and np.all(np.isnan(el_eq[:, 2]))          # equatorial: u = acos(0 / 0)
    assert list(F.elements_padded(oracle, para)[1]) == [5] * 16
    near = F.near_miss_states(oracle, np.concatenate([circ, circ_eq]), para)
    assert len(near) == 2 * 40 and set(F.elements_padded(oracle, near)[1]) == {6}


def test_four_element_form_is_the_six_element_form_at_zero_eccentricity(oracle):
    """[a, i, u, Omega] gives the bits of the six-element form (the C oracle) at [a, 0, i, 0, Omega, u]."""
    for a, i, u, Om in F.four_forms(np.random.default_rng(6), 500):
        R, V = F.state_from_form([a, i, u, Om])
        R6, V6 = oracle.state_information([a, 0.0, i, 0.0, Om, u], F.MU)
        assert same_bits(np.concatenate([R, V]), np.concatenate([R6, V6])), (a, i, u, Om)


def test_five_element_form_is_a_parabola_with_the_given_elements(oracle):
    """[p, i, omega, Omega, f] -> state -> elements: energy 0 to rounding, and p, i, omega, Omega, f recovered."""
    rng = np.random.default_rng(7)
    for p, i, om, Om, f in F.five_forms(rng, 300):
        if not (0.1 < i < math.pi - 0.1 and abs(math.cos(f)) < 0.9 and abs(math.cos(om)) < 0.99 and abs(math.cos(Om)) < 0.99):
            continue                                                      # node / apse angles ill-defined near 0, pi
        R, V = F.state_from_form([p, i, om, Om, f])
        r, v = np.linalg.norm(R), np.linalg.norm(V)
        assert abs(2 / r - v * v / F.MU) * r < 1e-13
        el = oracle.orbital_elements(F.MU, R, V)
        assert abs(el[1] - 1) < 1e-12 if len(el) == 6 else len(el) == 5
        got = [np.linalg.norm(np.cross(R, V)) ** 2 / F.MU] + list(el[-4:])
        want = [p, i, om % (2 * math.pi), Om % (2 * math.pi), f % (2 * math.pi)]
        d = np.abs(np.array(got) - np.array(want))
        d[2:] = np.minimum(d[2:], 2 * math.pi - d[2:])
        assert d[0] < 1e-12 * p and np.all(d[1:] < 1e-7), (want, got)
