"""calculate_orbital_elements on its circular / parabolic branches and calculate_state_information on its 5- and
4-element forms, on the device (sat_orbital_elements_all, sat_state_from_elements_n and the drop-in classes), against the
reference fixture and the host restatement, bit for bit. Run on the B200 box: pytest -m gpu."""
import os

import numpy as np
import pytest

import elements_forms as F

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

MU = F.MU
FIXTURE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "elements_branches_golden.npz")
needs_fixture = pytest.mark.skipif(not os.path.exists(FIXTURE),
                                   reason="elements_branches_golden.npz not recorded (make_golden_branches.py)")


def same_bits(a, b):
    """bit-identical, NaN matching NaN (the circular equatorial u is 0 / 0 on both sides)"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(np.all((a.view(np.int64) == b.view(np.int64)) | (np.isnan(a) & np.isnan(b))))


@pytest.fixture(scope="module")
def L():
    from ppo_rl_satellite_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def sf():
    from ppo_rl_satellite_b200.dropin import satellite_function
    return satellite_function


def elements_all(L, rv):
    d = torch.from_numpy(np.ascontiguousarray(rv, dtype=np.float64)).cuda()
    out = torch.full_like(d, 7.0)                          # padding must be written, not left over
    kind = torch.empty(d.shape[0], dtype=torch.int32, device="cuda")
    L.check(L.load().sat_orbital_elements_all(d.data_ptr(), d.shape[0], MU, out.data_ptr(), kind.data_ptr(), L.stream_ptr()),
            "sat_orbital_elements_all")
    return out.cpu().numpy(), kind.cpu().numpy()


def elements_old(L, rv):
    d = torch.from_numpy(np.ascontiguousarray(rv, dtype=np.float64)).cuda()
    out = torch.zeros_like(d)
    kind = torch.empty(d.shape[0], dtype=torch.int32, device="cuda")
    L.check(L.load().sat_orbital_elements(d.data_ptr(), d.shape[0], MU, out.data_ptr(), kind.data_ptr(), L.stream_ptr()),
            "sat_orbital_elements")
    return out.cpu().numpy(), kind.cpu().numpy()


def state_n(L, el, n_el=None):
    d = torch.from_numpy(np.ascontiguousarray(el, dtype=np.float64)).cuda()
    out = torch.empty((d.shape[0], 6), dtype=torch.float64, device="cuda")
    n_el = d.shape[1] if n_el is None else n_el
    return L.load().sat_state_from_elements_n(d.data_ptr(), d.shape[0], n_el, MU, out.data_ptr(), L.stream_ptr()), out.cpu().numpy()


@pytest.fixture(scope="module")
def pools(oracle):
    """branch states (circular inclined / equatorial, parabolic, one-ulp near misses), general states, and the oracle's
    elements of all of them; 5- and 4-element sets and the host restatement's states"""
    rng = np.random.default_rng(11)
    circ, circ_eq, para = F.circular_states(rng, oracle, 384), F.circular_states(rng, oracle, 128, True), F.parabolic_states(rng, oracle, 384)
    near = F.near_miss_states(oracle, np.concatenate([circ, circ_eq]), para)
    rv = np.concatenate([circ, circ_eq, para, near, F.general_states(rng, 1024)])
    el, kind = F.elements_padded(oracle, rv)
    forms = {}
    for n_el, gen in ((5, F.five_forms), (4, F.four_forms)):
        f = np.concatenate([gen(rng, 1536), el[kind == n_el, :n_el]])
        forms[n_el] = (f, F.states_from_forms(f))
    return dict(rv=rv, el=el, kind=kind, forms=forms)


# ---------------------------------------------------------------------------------------------------- reference fixture
@needs_fixture
def test_device_matches_reference_fixture(golden, L, sf):
    g = golden("elements_branches_golden.npz")
    el, kind = elements_all(L, g["rv"])
    assert np.array_equal(kind, g["kind"])
    T = sf.Time_window_of_danger_zone
    for k in range(len(kind)):
        assert same_bits(el[k, :kind[k]], g["elements"][k, :kind[k]]), k
        assert np.all(el[k, kind[k]:] == 0)
        if k % 7 == 0:                                      # the drop-in class, one row per call
            assert same_bits(T.calculate_orbital_elements(MU, g["rv"][k, :3], g["rv"][k, 3:]), g["elements"][k, :kind[k]])
    b_el, b_kind = sf.orbital_elements_batch(MU, g["rv"])
    assert np.array_equal(b_kind, g["kind"]) and same_bits(b_el, el)
    for n_el in (5, 4):
        rc, st = state_n(L, g[f"form{n_el}"])
        assert rc == 0 and same_bits(st, g[f"state{n_el}"])
        assert same_bits(sf.state_information_batch(g[f"form{n_el}"]), g[f"state{n_el}"])
        for k in range(0, len(st), 17):
            R, V = T.calculate_state_information(list(g[f"form{n_el}"][k]), miu=MU)
            assert same_bits(np.concatenate([R, V]), g[f"state{n_el}"][k])


# ---------------------------------------------------------------------------------------------------- host restatement
def test_branches_bit_identical_to_oracle(L, sf, pools):
    el, kind = elements_all(L, pools["rv"])
    assert np.array_equal(kind, pools["kind"]) and set(np.unique(kind)) == {4, 5, 6}
    assert same_bits(el, pools["el"])                       # valid columns and the zero padding
    T = sf.Time_window_of_danger_zone
    for k in range(0, len(kind), 23):
        assert same_bits(T.calculate_orbital_elements(MU, pools["rv"][k, :3], pools["rv"][k, 3:]), pools["el"][k, :kind[k]])
    for n_el in (5, 4):
        f, want = pools["forms"][n_el]
        rc, st = state_n(L, f)
        assert rc == 0 and same_bits(st, want)
        for k in range(0, len(f), 97):
            R, V = T.calculate_state_information(list(f[k]), miu=MU)
            assert same_bits(np.concatenate([R, V]), want[k])


@pytest.mark.parametrize("n", [1 << 20, (1 << 20) + 37])
def test_mixed_batch_bit_identical_row_by_row(L, pools, n):
    """every branch (and every form) in a seeded random order: lanes of a warp on different branches"""
    rng = np.random.default_rng(n)
    idx = rng.integers(0, len(pools["rv"]), n)
    el, kind = elements_all(L, pools["rv"][idx])
    assert np.array_equal(kind, pools["kind"][idx])
    assert same_bits(el, pools["el"][idx])
    for n_el in (5, 4):
        f, want = pools["forms"][n_el]
        j = rng.integers(0, len(f), n)
        rc, st = state_n(L, f[j])
        assert rc == 0 and same_bits(st, want[j])


def test_round_trip_keeps_kind(L, oracle):
    """element set -> state -> element set. The 5- and 4-element sets are [x, i, 0, 0, (0)] whose state lies exactly on its
    branch (any other set's state is six-element to rounding). x and i agree to the six-element round trip's tolerance
    (rtol 1e-12, atol 1e-8); the angles set to 0 come back through acos(1 - 1 ulp) = 1.5e-8 at worst, as in the reference."""
    rng = np.random.default_rng(12)
    for n_el in (5, 4):
        f = F.exact_round_trip_forms(rng, oracle, n_el, 256)
        rc, st = state_n(L, f)
        assert rc == 0
        el, kind = elements_all(L, st)
        assert np.all(kind == n_el)
        back = el[:, :n_el]
        np.testing.assert_allclose(back[:, :2], f[:, :2], rtol=1e-12, atol=1e-8)
        zero = np.minimum(np.abs(back[:, 2:]), np.abs(back[:, 2:] - 2 * np.pi))
        assert zero.max() <= 2 * 2.0 ** -26, zero.max()
    f6 = np.column_stack([rng.uniform(7e6, 4.3e7, 512), rng.uniform(1e-3, 0.5, 512), rng.uniform(0.1, 3.0, 512),
                          rng.uniform(0.1, 6.1, (512, 3))])
    rc, st = state_n(L, f6)
    el, kind = elements_all(L, st)
    assert rc == 0 and np.all(kind == 6)
    np.testing.assert_allclose(el, f6, rtol=1e-12, atol=1e-8)


# ---------------------------------------------------------------------------------------------------- unchanged paths
def test_existing_entry_points_unchanged(L, golden, pools):
    from ppo_rl_satellite_b200 import engine
    branch = pools["kind"] != 6
    _, kind_old = elements_old(L, pools["rv"][branch])
    assert np.all(kind_old == 0)                            # sat_orbital_elements: kind 0 on these rows, as before
    rv = pools["rv"][branch]
    pair = np.concatenate([rv, rv[::-1]], axis=1)           # both craft on a circular / parabolic element set
    mixed = np.concatenate([rv, pools["rv"][~branch][:len(rv)]], axis=1)
    for states in (pair, mixed):
        cnt = engine.danger_zone_count(torch.from_numpy(np.ascontiguousarray(states)).cuda(),
                                       torch.full((len(states),), 2.0, dtype=torch.float64, device="cuda"))
        assert np.all(cnt.cpu().numpy() == -1)
    ge = golden("elements_golden.npz")
    rv841 = np.concatenate([ge["R"], ge["V"]], axis=1)
    el_old, k_old = elements_old(L, rv841)
    el_new, k_new = elements_all(L, rv841)
    assert np.all(k_old == 6) and np.array_equal(k_old, k_new) and same_bits(el_old, el_new)
    d = torch.from_numpy(ge["elements_live"]).cuda()
    out = torch.empty_like(d)
    L.check(L.load().sat_state_from_elements(d.data_ptr(), d.shape[0], MU, out.data_ptr(), L.stream_ptr()), "state")
    rc, st = state_n(L, ge["elements_live"], 6)
    assert rc == 0 and same_bits(st, out.cpu().numpy())


@pytest.mark.parametrize("n_el", [3, 7, 0, -1])
def test_state_from_elements_n_rejects_other_counts(L, n_el):
    rc, _ = state_n(L, np.zeros((4, 6)), n_el)
    assert rc == -2                                         # SAT_ERR_SIZE
