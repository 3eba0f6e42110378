"""Small synthetic hierarchical logistic-regression problems for the tests."""
import numpy as np

from oracle import density as dens
from oracle import fakes


def make_site(model, n, D, J, seed):
    """One site's data + a plausible cavity.  Returns dict(X, y, j_ind, J, mu, Omega)."""
    rng = np.random.RandomState(seed)
    X = rng.standard_normal((n, D)) * 0.7 + 0.2 * rng.standard_normal(D)
    sizes = np.full(J, n // J)
    sizes[:n - sizes.sum()] += 1
    j_ind = np.repeat(np.arange(J), sizes)
    beta = rng.standard_normal(D) * 0.8
    alpha = rng.standard_normal(J) * 0.7
    bj = np.repeat(beta[None, :], J, axis=0) + (0.0 if model == 'm1b' else 0.4 * rng.standard_normal((J, D)))
    f = alpha[j_ind] + np.einsum('nd,nd->n', X, bj[j_ind])
    y = (rng.uniform(size=n) < 1 / (1 + np.exp(-f))).astype(np.int64)
    d = dens.dphi(model, D)
    Omega = fakes.random_spd(rng, d, scale=1.5)
    mu = 0.3 * rng.standard_normal(d)
    return dict(X=X, y=y, j_ind=j_ind, J=J, mu=mu, Omega=Omega, d=d, sizes=sizes)


def oracle_density(model, site):
    return dens.TiltedDensity(model, site['X'], site['y'], site['mu'], site['Omega'],
                              j_ind=site['j_ind'], J=site['J'])


def bf16_round(x):
    """round-to-nearest-even fp32 -> bf16 -> fp64 (what the tensor-core path stores)"""
    u = np.asarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return u.astype(np.uint32).view(np.float32).astype(np.float64)


def tc_stored_X(X):
    """The design matrix as the tensor-core pass holds it (csrc/epg_sampler.cu k_convert_xb): centred on the
    site's column means (fp64 mean stored as fp32), the remainder rounded to bf16; the means re-enter
    exactly through the intercept coefficient / chain rule, so the effective inputs are mean + bf16(x - mean)."""
    X = np.asarray(X, dtype=np.float64)
    c = X.mean(axis=0).astype(np.float32)
    dev = X.astype(np.float32) - c
    return c.astype(np.float64) + bf16_round(dev)


def tc_oracle(model, site):
    """fp64 oracle of the tensor-core passes (csrc/epg_lik_tc.cuh, epg_lik_tcw.cuh): the design matrix as
    tc_stored_X holds it, and the residuals E = y - sigmoid(f) rounded to bf16 as the epilogue stores them for
    the gradient product G = E'X.  Returns lp_grad(q) -> (lp, grad)."""
    td = oracle_density(model, dict(site, X=tc_stored_X(site['X'])))
    return lambda q: td.lp_grad(q, e_map=bf16_round)
