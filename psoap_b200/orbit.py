"""Drop-in for psoap.orbit's get_velocities() (psoap/orbit.py): SB1, SB2, ST1, ST2, ST3 and `models`.

Constructors take the reference's positional parameters; get_velocities(dates=None) returns the reference's
[n_components, n_dates] numpy array.  The Kepler solve and the velocity formulae run in one CUDA kernel
(csrc/orbit.cuh); in the chunk farm the same kernel feeds the covariance fill without leaving the device.
"""
import numpy as np

from . import _lib


# orbital parameter names in positional order (psoap/utils.py:4-8, up to and including gamma)
PARAM_NAMES = {
    "SB1": ["K", "e", "omega", "P", "T0", "gamma"],
    "SB2": ["q", "K", "e", "omega", "P", "T0", "gamma"],
    "ST1": ["K_in", "e_in", "omega_in", "P_in", "T0_in", "K_out", "e_out", "omega_out", "P_out", "T0_out", "gamma"],
    "ST2": ["q_in", "K_in", "e_in", "omega_in", "P_in", "T0_in", "K_out", "e_out", "omega_out", "P_out", "T0_out",
            "gamma"],
    "ST3": ["q_in", "K_in", "e_in", "omega_in", "P_in", "T0_in", "q_out", "K_out", "e_out", "omega_out", "P_out",
            "T0_out", "gamma"],
}


class _Orbit:
    model = None

    def __init__(self, *args, obs_dates=None, **kwargs):
        # reference call styles: models[m](*p_orb, date1D) (sample_parallel.py:183) and
        # models[m](**pars, obs_dates=date1D) (sample_parallel.py:166; extra keys ignored via **kwargs)
        names = PARAM_NAMES[self.model]
        args = list(args)
        if len(args) == len(names) + 1 and obs_dates is None:
            obs_dates = args.pop()
        if len(args) > len(names):
            raise TypeError("%s takes %d orbital parameters" % (self.model, len(names)))
        vals = dict(zip(names, args))
        for k in names[len(args):]:
            if k not in kwargs:
                raise TypeError("%s() missing required argument '%s'" % (self.model, k))
            vals[k] = kwargs[k]
        self.params = np.array([vals[k] for k in names], dtype=np.float64)
        for k in names:
            setattr(self, k, vals[k])
        self._check()
        self.obs_dates = obs_dates

    def _check(self):
        names = {"SB1": [1], "SB2": [2], "ST1": [1, 6], "ST2": [2, 7], "ST3": [2, 8]}[self.model]
        for k in names:
            e = self.params[k]
            assert (e >= 0.0) and (e < 1.0), "Eccentricity must be between [0, 1)"  # orbit.py:33,:192-193

    def get_velocities(self, dates=None):
        if dates is None and self.obs_dates is None:
            raise RuntimeError("Must provide input dates or specify observation dates upon creation of orbit object.")
        if dates is None:
            dates = self.obs_dates
        dates = np.atleast_1d(np.asarray(dates, dtype=np.float64))
        return velocities(self.model, self.params, dates).cpu().numpy()


def velocities(model, p_orb, dates):
    """Device evaluation: returns a CUDA tensor [ncomp, n_dates]."""
    lib = _lib.load()
    torch = _lib.torch_cuda()
    p = _lib.dev_f64(p_orb)
    d = _lib.dev_f64(dates)
    ncomp = _lib.NCOMP[model]
    out = torch.empty((ncomp, d.numel()), dtype=torch.float64, device="cuda")
    _lib.check(lib.psoap_orbit_velocities(_lib.MODELS[model], _lib.ptr(p), _lib.ptr(d), d.numel(), _lib.ptr(out),
                                          _lib.vp(None), _lib.stream_ptr()))
    return out


def velocity_jacobian(model, p_orb, dates):
    """d v_c[ep] / d p_orb[k] of `velocities` on the device: CUDA tensor [ncomp, n_dates, n_orb] (p_orb in
    utils.registered_params order)."""
    lib = _lib.load()
    torch = _lib.torch_cuda()
    p = _lib.dev_f64(p_orb)
    d = _lib.dev_f64(np.atleast_1d(np.asarray(dates, dtype=np.float64)) if not isinstance(dates, torch.Tensor) else dates)
    norb = _lib.N_ORB[model]
    if p.numel() != norb:
        raise ValueError("%s takes %d orbital parameters" % (model, norb))
    out = torch.empty((_lib.NCOMP[model], d.numel(), norb), dtype=torch.float64, device="cuda")
    _lib.check(lib.psoap_orbit_jacobian(_lib.MODELS[model], _lib.ptr(p), _lib.ptr(d), d.numel(), _lib.ptr(out),
                                        _lib.stream_ptr()))
    return out


class SB1(_Orbit):
    """orbit.py:20-115: SB1(K, e, omega, P, T0, gamma, obs_dates=None)"""
    model = "SB1"


class SB2(_Orbit):
    """orbit.py:117-170: SB2(q, K, e, omega, P, T0, gamma, obs_dates=None)"""
    model = "SB2"


class ST1(_Orbit):
    """orbit.py:172-320"""
    model = "ST1"


class ST2(_Orbit):
    """orbit.py:323-417"""
    model = "ST2"


class ST3(_Orbit):
    """orbit.py:420-487"""
    model = "ST3"


models = {"SB1": SB1, "SB2": SB2, "ST1": ST1, "ST2": ST2, "ST3": ST3}  # orbit.py:490
