"""Chunk-farm sampler driver: the B200 replacement of `psoap-sample-parallel`
(psoap/sample_parallel.py:40-92 set-up, :331-390 priors and lnprob, :396-443 Metropolis-Hastings run).

The likelihood of a proposal is one `ChunkFarm.lnprob` call (all chunks, one CUDA graph per GPU, one all-reduce).
emcee is not a dependency: `MHSampler` below keeps the part of emcee.MHSampler the reference uses (Gaussian
proposals with a fixed covariance, `sample(p0, iterations)` generator, `flatchain`, `lnprobability`,
`acceptance_fraction`).  Under torchrun every rank runs the same chain from the same seed (the proposals and the
all-reduced likelihoods are identical on all ranks, so are the accept decisions); rank 0 writes the outputs.
"""
import collections
import os
import shutil

import numpy as np

from . import utils


# --------------------------------------------------------------------------------------------------
# Priors — psoap/sample_parallel.py:331-356 (bounds only)
# --------------------------------------------------------------------------------------------------
def prior_SB1(p_orb, p_GP):
    K, e, omega, P, T0, gamma = p_orb
    amp_f, l_f = p_GP
    if K < 0.0 or e < 0.0 or e > 1.0 or P < 0.0 or omega < -90 or omega > 450 or amp_f < 0.0 or l_f < 0.0:
        return -np.inf
    return 0.0


def prior_SB2(p_orb, p_GP):
    q, K, e, omega, P, T0, gamma = p_orb
    amp_f, l_f, amp_g, l_g = p_GP
    if (q < 0.0 or K < 0.0 or e < 0.0 or e > 1.0 or P < 0.0 or omega < -90 or omega > 450 or amp_f < 0.0 or l_f < 0.0
            or amp_g < 0.0 or l_g < 0.0):
        return -np.inf
    return 0.0


def prior_ST3(p_orb, p_GP):
    q_in, K_in, e_in, omega_in, P_in, T0_in, q_out, K_out, e_out, omega_out, P_out, T0_out, gamma = p_orb
    if (q_in < 0.0 or K_in < 0.0 or e_in < 0.0 or e_in > 1.0 or P_in < 0.0 or omega_in < -90 or omega_in > 450
            or q_out < 0.0 or K_out < 0.0 or e_out < 0.0 or e_out > 1.0 or P_out < 0.0 or omega_out < -90
            or omega_out > 450 or np.any(np.asarray(p_GP) < 0.0)):
        return -np.inf
    return 0.0


priors = {"SB1": prior_SB1, "SB2": prior_SB2, "ST3": prior_ST3}  # sample_parallel.py:368


# --------------------------------------------------------------------------------------------------
# Metropolis-Hastings (the subset of emcee.MHSampler used at sample_parallel.py:434-443)
# --------------------------------------------------------------------------------------------------
class MHSampler:
    def __init__(self, cov, dim, lnprobfn, seed=None):
        self.cov = np.atleast_2d(np.asarray(cov, dtype=np.float64))
        self.dim = dim
        self.lnprobfn = lnprobfn
        self.rng = np.random.default_rng(seed)
        self._chain = np.empty((0, dim))
        self._lnprob = np.empty(0)
        self.naccepted = 0
        self.iterations = 0

    @property
    def flatchain(self):
        return self._chain

    chain = flatchain

    @property
    def lnprobability(self):
        return self._lnprob

    @property
    def acceptance_fraction(self):
        return self.naccepted / max(1, self.iterations)

    def sample(self, p0, lnprob0=None, iterations=1):
        p = np.array(p0, dtype=np.float64)
        lnprob = self.lnprobfn(p) if lnprob0 is None else lnprob0
        i0 = len(self._chain)
        self._chain = np.concatenate((self._chain, np.zeros((iterations, self.dim))), axis=0)
        self._lnprob = np.append(self._lnprob, np.zeros(iterations))
        for i in range(i0, i0 + iterations):
            self.iterations += 1
            q = self.rng.multivariate_normal(p, self.cov)
            newlnprob = self.lnprobfn(q)
            diff = newlnprob - lnprob
            if diff < 0:
                diff = np.exp(diff) - self.rng.random()
            if diff > 0:  # accept (also covers diff == +inf from a -inf starting point)
                p, lnprob = q, newlnprob
                self.naccepted += 1
            self._chain[i] = p
            self._lnprob[i] = lnprob
            yield p, lnprob

    def run_mcmc(self, p0, N, **kwargs):
        result = None
        for result in self.sample(p0, iterations=N, **kwargs):
            pass
        return result


# --------------------------------------------------------------------------------------------------
# Chunk files.  The reference stores chunks as HDF5 (psoap/data.py:149-197: datasets wl, fl, sigma, date, mask of
# shape [n_epochs, n_pix]); h5py is optional here, the same arrays in an .npz are accepted too.
# --------------------------------------------------------------------------------------------------
def load_chunk(fname, limit=100):
    """-> dict(lwl, fl, sigma, mask, date1D) after apply_mask() (psoap/data.py:120-147), first `limit` epochs."""
    from .data import Chunk
    if fname.endswith(".npz"):
        with np.load(fname) as f:
            arr = {k: f[k][:limit] for k in Chunk.DATASETS}
    else:
        import h5py  # optional dependency
        with h5py.File(fname, "r") as f:
            arr = {k: f[k][:limit] for k in Chunk.DATASETS}
    ch = Chunk(arr["wl"].astype(np.float64), arr["fl"].astype(np.float64), arr["sigma"].astype(np.float64),
               arr["date"].astype(np.float64), np.array(arr["mask"], dtype=bool))
    ch.apply_mask()
    return ch.as_farm_chunk()


def load_config(path="config.yaml"):
    """The run's YAML configuration (sample_parallel.py:11-17; keys as in psoap/data/config.SB2.yaml)."""
    import yaml
    try:
        with open(path) as f:
            return yaml.safe_load(f)
    except FileNotFoundError:
        print("You need to copy a config.yaml file to this directory, and then edit the values to your particular case.")
        raise


def load_user_prior(directory="."):
    """sample_parallel.py:362-369: a file `prior.py` in the run directory defining `prior(p)` (p = the SAMPLED
    parameter vector, fixed parameters left out) overrides the default bounds-only prior.  Returns None if absent."""
    import importlib.util
    path = os.path.join(directory, "prior.py")
    if not os.path.exists(path):
        return None
    spec = importlib.util.spec_from_file_location("prior", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.prior


def make_lnprob(farm, model, fix_params, pars, prior=None, user_prior=None):
    """sample_parallel.py:371-390 with the farm in place of the worker processes.  `prior(p_orb, p_GP)` replaces the
    default for the model; `user_prior(p)` is the reference's prior.py convention and takes precedence."""
    prior = prior or priors[model]

    def lnprob(p):
        p_orb, p_GP = utils.convert_vector(p, model, fix_params, **pars)
        lnprior = user_prior(p) if user_prior is not None else prior(p_orb, p_GP)
        if lnprior == -np.inf:
            return -np.inf
        return farm.lnprob(np.concatenate([p_orb, p_GP])) + lnprior
    return lnprob


def fisher_jump(F, model, fix_params):
    """Gaussian jump covariance for MHSampler from the expected Fisher information F [n_params, n_params] of the full
    registered vector (ChunkFarm.fisher): 2.38^2/d * inv(F_fit), F_fit = F restricted to the d sampled parameters
    (registry order, fix_params left out), the scaling utils.estimate_covariance gives a pilot chain's covariance.
    Raises ValueError when F_fit has an exactly zero row (the likelihood does not depend on that parameter: gamma,
    whose row is zero because the covariance depends on velocity differences only) or is not positive definite."""
    names = [n for n in utils.registered_params[model] if n not in fix_params]
    idx = [utils.registered_params[model].index(n) for n in names]
    F = np.asarray(F, dtype=np.float64)
    F_fit = F[np.ix_(idx, idx)]
    zero = [n for n, row in zip(names, F_fit) if not np.any(row)]
    if zero:
        raise ValueError("the Fisher information has an exactly zero row for %s: the likelihood does not depend on %s; "
                         "fix it (fix_params)" % (", ".join(zero), "it" if len(zero) == 1 else "them"))
    try:
        np.linalg.cholesky(F_fit)
    except np.linalg.LinAlgError as e:
        raise ValueError("the Fisher information of the sampled parameters %s is not positive definite" % names) from e
    return 2.38 ** 2 / len(idx) * np.linalg.inv(F_fit)


# --------------------------------------------------------------------------------------------------
# Per-epoch radial velocities without an orbit (ChunkFarm(..., free_velocities=True))
# --------------------------------------------------------------------------------------------------
# fit_epoch_velocities' result: v [ncomp, Ng] (km/s, at farm.epochs), gp [2 ncomp], cov (the Cramer-Rao covariance of
# the fitted entries, in the order of `free`), free (their positions in the farm's vector), sigma_v [ncomp, Ng] (the
# square root of cov's diagonal at each velocity; 0 at the reference epoch), lnprob, and scipy's OptimizeResult
EpochFit = collections.namedtuple("EpochFit", "v gp cov free sigma_v lnprob opt")


def epoch_fit_free(ncomp, Ng, ref_epoch=0, fix_gp=False):
    """Positions in the free vector [v_0[0..Ng), .., GP] that fit_epoch_velocities varies: every velocity except each
    component's v_c[ref_epoch] (the gauge: the likelihood depends on velocity differences within a component only),
    and the 2 ncomp GP values unless fix_gp."""
    if not 0 <= ref_epoch < Ng:
        raise ValueError("ref_epoch must lie in [0, %d)" % Ng)
    fixed = {c * Ng + ref_epoch for c in range(ncomp)}
    n = ncomp * Ng + (0 if fix_gp else 2 * ncomp)
    return np.array([k for k in range(n) if k not in fixed], dtype=np.int64)


def fit_epoch_velocities(farm, v0, gp0, ref_epoch=0, fix_gp=False, options=None):
    """Maximum-likelihood radial velocity of every component at every epoch, without an orbit: L-BFGS-B (scipy) on
    farm.lnprob_and_grad for a ChunkFarm built with free_velocities=True.  v0: [ncomp, Ng] starting velocities (km/s,
    at farm.epochs), gp0: the 2 ncomp GP values.  Each component's v_c[ref_epoch] is held at its v0 value, which fixes
    the gauge (a constant added to all of a component's velocities leaves the likelihood unchanged); with fix_gp the GP
    values are held too.  The GP values are bounded below by 0.  Returns an EpochFit; its covariance is the inverse of
    farm.fisher at the optimum with the fixed rows and columns removed (the Cramer-Rao bound)."""
    from scipy.optimize import minimize
    from . import _lib
    if not getattr(farm, "free", False):
        raise ValueError("fit_epoch_velocities needs a ChunkFarm built with free_velocities=True")
    ncomp, Ng = _lib.NCOMP[farm.model], len(farm.epochs)
    v0 = np.asarray(v0, dtype=np.float64)
    gp0 = np.asarray(gp0, dtype=np.float64).reshape(-1)
    if v0.shape != (ncomp, Ng) or gp0.size != 2 * ncomp:
        raise ValueError("v0 must be [%d, %d] and gp0 hold %d values" % (ncomp, Ng, 2 * ncomp))
    p0 = np.concatenate([v0.reshape(-1), gp0])
    free = epoch_fit_free(ncomp, Ng, ref_epoch, fix_gp)
    nv = ncomp * Ng

    def full(x):
        p = p0.copy()
        p[free] = x
        return p

    def f(x):
        lnp, g = farm.lnprob_and_grad(full(x))
        if not np.isfinite(lnp):
            return np.inf, np.zeros_like(x)
        return -lnp, -g[free]

    bounds = [(None, None) if k < nv else (0.0, None) for k in free]
    opt = minimize(f, p0[free], jac=True, method="L-BFGS-B", bounds=bounds, options=options or {})
    p = full(opt.x)
    F = np.asarray(farm.fisher(p), dtype=np.float64)[np.ix_(free, free)]
    cov = np.linalg.inv(F)
    sig = np.zeros(nv)
    vfree = free < nv
    sig[free[vfree]] = np.sqrt(np.diag(cov)[vfree])
    return EpochFit(p[:nv].reshape(ncomp, Ng), p[nv:], cov, free, sig.reshape(ncomp, Ng), -float(opt.fun), opt)


def fit_sb1_epoch_velocities(chunks, v0, amp_f, l_f, ref_epoch=0, mu_GP=1.0, soften=1.0, fix_gp=False, **farm_kw):
    """Single-lined per-epoch velocities on the dense GP: the counterpart of the reference's celerite per-epoch fit
    (psoap/covariance.py:426-494), with the velocities at the sorted unique dates of all chunks.  v0: [Ng] starting
    velocities (km/s).  Builds a one-component free-velocity farm, runs fit_epoch_velocities and releases the farm."""
    from .farm import ChunkFarm
    farm = ChunkFarm("SB1", chunks, mu_GP=mu_GP, soften=soften, free_velocities=True, **farm_kw)
    try:
        return fit_epoch_velocities(farm, np.asarray(v0, dtype=np.float64).reshape(1, -1), [amp_f, l_f], ref_epoch,
                                    fix_gp)
    finally:
        farm.close()


def run(config, chunks, run_index=0, seed=0, rank=0, world_size=1, process_group=None, verbose=True, workdir=None):
    """Run the chain described by a PSOAP config (a dict, or the path of a config.yaml; psoap/data/config.SB2.yaml
    keys: model, parameters, jumps, fix_params, samples, opt_jump, outdir, soften; `fisher_jump: true` takes the jump
    covariance from fisher_jump(farm.fisher(p0), ...) instead of opt_jump / jumps).  A `prior.py` in `workdir`
    (default: the current directory, as in the reference) overrides the default prior.  Returns the sampler."""
    from .farm import ChunkFarm
    if isinstance(config, str):
        config = load_config(config)
    model, pars, fix = config["model"], config["parameters"], config["fix_params"]
    user_prior = load_user_prior(workdir or ".")
    if verbose and rank == 0:
        print("Loaded user defined prior." if user_prior is not None else "Using default prior.")
    farm = ChunkFarm(model, chunks, soften=config.get("soften", 1.0), rank=rank, world_size=world_size,
                     process_group=process_group)
    lnprob = make_lnprob(farm, model, fix, pars, user_prior=user_prior)
    dim = len(utils.registered_params[model]) - len(fix)
    p0 = utils.convert_dict(model, fix, **pars)
    lnp0 = lnprob(p0)
    if lnp0 == -np.inf:  # sample_parallel.py:406-422
        farm.close()
        raise RuntimeError("Starting position for Markov Chain evaluates to -np.inf")
    if config.get("fisher_jump"):  # the local shape of the posterior at p0, without a pilot chain
        try:
            cov = fisher_jump(farm.fisher(np.concatenate(utils.convert_vector(p0, model, fix, **pars))), model, fix)
        except Exception:
            farm.close()
            raise
    else:
        try:
            cov = np.load(config.get("opt_jump", ""))  # sample_parallel.py:427-432
        except Exception:
            cov = utils.convert_dict(model, fix, **config["jumps"]) ** 2 * np.eye(dim)
    sampler = MHSampler(cov, dim, lnprob, seed=seed)
    for i, _ in enumerate(sampler.sample(p0, lnprob0=lnp0, iterations=config["samples"])):
        if verbose and rank == 0 and (i + 1) % 20 == 0:
            print("Iteration", i + 1)
    if rank == 0 and config.get("outdir"):
        routdir = os.path.join(config["outdir"], "run{:0>2}".format(run_index))
        if os.path.exists(routdir):
            shutil.rmtree(routdir)
        os.makedirs(routdir)
        np.save(os.path.join(routdir, "lnprob.npy"), sampler.lnprobability)      # sample_parallel.py:442-443
        np.save(os.path.join(routdir, "flatchain.npy"), sampler.flatchain)
    farm.close()
    return sampler
