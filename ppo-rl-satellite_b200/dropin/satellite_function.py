"""satellite_function -- drop-in for the hot-path subset of the reference's satellite_function.py.

Clohessy_Wiltshire.State_transition_matrix, Time_window_of_danger_zone.{calculate_orbital_elements,
calculate_state_information, calculate_number_of_hanger_area} run as CUDA kernels (batch of one, or batched when
given arrays with a leading axis); the first two cover every branch and element-set form of the reference. Numerical_calculation_method.numerical_calculation (the RK45 propagator the env has
commented out) is a per-state adaptive kernel. Out of scope (never called by the env or the driver, SURVEY.md s2): the
time-window sweep, Lagrange propagation, Danger_index_and_TW_matching_index.
"""
import numpy as np

try:
    from ._boot import engine as _eng, _lib as _L
except ImportError:  # imported as a top-level module (dropin/ on sys.path, the CPPO_main.py case)
    from _boot import engine as _eng, _lib as _L


def _dev(a):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device="cuda")


class Clohessy_Wiltshire:
    def __init__(self, R0_c=None, V0_c=None, R0_t=None, V0_t=None):
        self.R0_c, self.V0_c, self.R0_t, self.V0_t = R0_c, V0_c, R0_t, V0_t
        self.u = 3.986e14

    def State_transition_matrix(self, t):
        """satellite_function.py:753-781 -> (state_c_new[6], state_t_new[6])."""
        import torch
        self.t = t
        M = _eng.cw_stm(t)
        x, _buf = _eng.alloc_soa(6, 2, torch.float64, "cuda")
        x[:, 0] = _dev(np.concatenate([np.asarray(self.R0_c, dtype=np.float64), np.asarray(self.V0_c, dtype=np.float64)]))
        x[:, 1] = _dev(np.concatenate([np.asarray(self.R0_t, dtype=np.float64), np.asarray(self.V0_t, dtype=np.float64)]))
        import ctypes as C
        Mh = (C.c_double * 36)(*M.ravel())
        _L.check(_L.load().sat_cw_propagate(x.data_ptr(), 2, x.stride(0), Mh, _L.stream_ptr()), "sat_cw_propagate")
        out = x.cpu().numpy()
        return out[:, 0].copy(), out[:, 1].copy()


class Time_window_of_danger_zone:
    def __init__(self, R0_c=None, V0_c=None, R0_t=None, V0_t=None, c_args=None, t_args=None, Delta_V_c=None,
                 Delta_V_t=None, time_step=None, u=3.986e14):
        assert ((R0_c is not None and V0_c is not None) or c_args is not None) and \
               ((R0_t is not None and V0_t is not None) or t_args is not None), \
            "At least one of the speed, position, and elements not be None"
        self.time_step, self.u, self.Delta_V_c, self.Delta_V_t = time_step, u, Delta_V_c, Delta_V_t
        self.fai, self.num_td = 0, 0
        if R0_c is not None:
            assert isinstance(R0_c, np.ndarray) and isinstance(V0_c, np.ndarray)
            self.R0_c, self.V0_c = R0_c, V0_c
        else:
            self.R0_c, self.V0_c = self.calculate_state_information(c_args, miu=3.986e14)
        if R0_t is not None:
            assert isinstance(R0_t, np.ndarray) and isinstance(V0_t, np.ndarray)
            self.R0_t, self.V0_t = R0_t, V0_t
        else:
            self.R0_t, self.V0_t = self.calculate_state_information(t_args, miu=3.986e14)
        ec = self.calculate_orbital_elements(self.u, self.R0_c, self.V0_c)
        et = self.calculate_orbital_elements(self.u, self.R0_t, self.V0_t)
        self.a_c, self.e_c, self.i_c, self.omega_c, self.Omega_c, self.f0_c = ec
        self.a_t, self.e_t, self.i_t, self.omega_t, self.Omega_t, self.f0_t = et
        self.r_c = self.a_c * (1 - self.e_c ** 2) / (1 + self.e_c * np.cos(self.f0_c))
        self.p_c = self.a_c * (1 - self.e_c ** 2)
        self.r_t = self.a_t * (1 - self.e_t ** 2) / (1 + self.e_t * np.cos(self.f0_t))
        self.p_t = self.a_t * (1 - self.e_t ** 2)

    @staticmethod
    def calculate_orbital_elements(miu, R0, V0):
        """satellite_function.py:161-255 -> [a, e, i, omega, Omega, f]; on the parabolic branch (energy == 0)
        [p, i, omega, Omega, f], on the circular branch (e == 0) [a, i, u, Omega]."""
        rv = np.concatenate([np.asarray(R0, dtype=np.float64), np.asarray(V0, dtype=np.float64)]).reshape(1, 6)
        out, kind = orbital_elements_batch(miu, rv)
        return [float(v) for v in out[0, :int(kind[0])]]

    @staticmethod
    def calculate_state_information(data, miu=3.986e14):
        """satellite_function.py:257-315 -> (Coordinate[3], V[3]) from [a, e, i, omega, Omega, f], [p, i, omega, Omega, f]
        or [a, i, u, Omega]."""
        o = state_information_batch(np.asarray(data, dtype=np.float64).reshape(1, -1), miu=miu)[0]
        return o[:3].copy(), o[3:].copy()

    def calculate_number_of_hanger_area(self):
        """satellite_function.py:341-373 -> 0 / 1 / 2."""
        rv = _dev(np.concatenate([self.R0_c, self.V0_c, self.R0_t, self.V0_t]).reshape(1, 12))
        dv = _dev(np.array([float(self.Delta_V_c)]))
        n = int(_eng.danger_zone_count(rv, dv, u=self.u)[0])
        if n < 0:
            raise AttributeError("circular / parabolic element set: the reference raises here as well")
        self.num_td = n
        return n


class Numerical_calculation_method:
    """satellite_function.py:783-839: RK45 (scipy solve_ivp semantics) on the CW ODE for both craft."""

    def __init__(self, R0_c=None, V0_c=None, R0_t=None, V0_t=None):
        self.R0_c, self.V0_c, self.R0_t, self.V0_t = R0_c, V0_c, R0_t, V0_t
        self.u = 3.986e5
        self.pursuer_initial_state = np.concatenate((self.R0_c, self.V0_c))
        self.escaper_initial_state = np.concatenate((self.R0_t, self.V0_t))

    @staticmethod
    def _constants():
        import math
        mu, r = 398600, 35786                                  # :796,799 (python ints: r ** 3 is exact)
        omega = math.sqrt(mu / (r ** 3))                       # :801
        return 2 * omega, 3 * omega ** 2, omega ** 2           # :818-820

    def numerical_calculation(self, t):
        import torch
        if t <= 0 or t % 50 != 0:
            raise ValueError("Values in `t_eval` are not within `t_span`.")     # what solve_ivp raises for arange(0, t+50, 50)
        w2, w3, wz = self._constants()
        x, _buf = _eng.alloc_soa(6, 2, torch.float64, "cuda")
        x[:, 0] = _dev(self.pursuer_initial_state)
        x[:, 1] = _dev(self.escaper_initial_state)
        _L.check(_L.load().sat_cw_ode_rk45(x.data_ptr(), 2, x.stride(0), float(t), w2, w3, wz, 1e-3, 1e-6, None,
                                           _L.stream_ptr()), "sat_cw_ode_rk45")
        out = x.cpu().numpy()
        self.R0_c, self.V0_c = out[:3, 0].copy(), out[3:, 0].copy()
        self.R0_t, self.V0_t = out[:3, 1].copy(), out[3:, 1].copy()
        return out[:, 0].copy(), out[:, 1].copy()


def orbital_elements_batch(miu, rv):
    """rv: [n, 6] array (R, V) -> elements [n, 6], kind [n] (batched helper, CUDA). Row k holds the list
    calculate_orbital_elements returns, zero-padded; kind[k] is its length: 6, 5 (parabolic) or 4 (circular)."""
    import torch
    rv = _dev(rv)
    out = torch.empty_like(rv)
    kind = torch.empty(rv.shape[0], dtype=torch.int32, device="cuda")
    _L.check(_L.load().sat_orbital_elements_all(rv.data_ptr(), rv.shape[0], float(miu), out.data_ptr(), kind.data_ptr(),
                                                _L.stream_ptr()), "sat_orbital_elements_all")
    return out.cpu().numpy(), kind.cpu().numpy()


def state_information_batch(el, miu=3.986e14):
    """el: [n, 6], [n, 5] or [n, 4] element sets (the forms calculate_state_information takes) -> [n, 6] (R, V)."""
    import torch
    el = _dev(el)
    if el.dim() != 2 or el.shape[1] not in (6, 5, 4):
        raise ValueError(f"element sets must be [n, 6], [n, 5] or [n, 4], got {tuple(el.shape)}")
    out = torch.empty((el.shape[0], 6), dtype=torch.float64, device="cuda")
    _L.check(_L.load().sat_state_from_elements_n(el.data_ptr(), el.shape[0], el.shape[1], float(miu), out.data_ptr(),
                                                 _L.stream_ptr()), "sat_state_from_elements_n")
    return out.cpu().numpy()
