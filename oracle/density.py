"""fp64 NumPy restatement of the tilted log-densities and their gradients.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

The tilted density of a site is   cavity N(phi; mu, Omega^-1)  x  N(eta;0,I)
[x N(etb;0,I)]  x  prod_n Bernoulli-logit(y_n; f_n), as written in the
reference's Stan programs (all sampled parameters are unconstrained, so there
are no Jacobian terms; Stan drops additive constants):

  m1b[_sg]  experiment/models/m1b.stan:21-42, m1b_sg.stan:19-35
            phi = [log sigma_a, beta(D)];  alpha_j = eta_j sigma_a;  f = alpha_j + x'beta
  m3b[_sg]  m3b.stan:21-49, m3b_sg.stan:19-39
            phi = [log sigma_a, log sigma_b(D)];  beta_j = etb_j * sigma_b
  m4b[_sg]  m4b.stan:21-53, m4b_sg.stan:19-43
            phi = [mu_a, log sigma_a, mu_b(D), log sigma_b(D)]
            alpha_j = mu_a + eta_j sigma_a;  beta_j = mu_b + etb_j * sigma_b
  m2b[_sg]  m2b.stan:21-46, m2b_sg.stan:19-38
            phi = [log sigma_a, log sigma_b];  alpha_j = eta_j sigma_a;  beta = etb sigma_b
            (ONE slope vector etb(D) for all groups of the site, a site-local latent)
  m5b[_sg]  m5b.stan:21-53, m5b_sg.stan:19-45
            m4b with Laplace latents: eta, etb ~ double_exponential(0, 1)  ->  -|eta| - sum|etb|

Parameter vector layout used by this repo (oracle and CUDA alike):
    q = [ phi (d) | eta (J) | etb (J x D, group-major) ]   (etb only for m3b/m4b/m5b; m2b: etb (D))

Parity status: UNPINNED against Stan (PyStan 2.17.0.0 is an un-vendored
dependency, not installed here).  tests/test_oracle_density.py pins the
gradient against central finite differences of the log-density and the
log-density against an independent scalar evaluation of the Stan model block.
"""

import numpy as np

MODELS = ('m1b', 'm2b', 'm3b', 'm4b', 'm5b')


def dphi(model, D):
    return {'m1b': D + 1, 'm2b': 2, 'm3b': D + 1, 'm4b': 2 * D + 2, 'm5b': 2 * D + 2}[model]


def num_params(model, D, J):
    return dphi(model, D) + J + {'m1b': 0, 'm2b': D}.get(model, J * D)


class TiltedDensity(object):
    def __init__(self, model, X, y, mu, Omega, j_ind=None, J=1):
        assert model in MODELS
        self.model = model
        self.X = np.asarray(X, dtype=np.float64)
        self.y = np.asarray(y, dtype=np.float64)
        self.N, self.D = self.X.shape
        self.J = int(J)
        self.j_ind = np.zeros(self.N, dtype=np.int64) if j_ind is None else np.asarray(j_ind, dtype=np.int64)
        self.mu = np.asarray(mu, dtype=np.float64)
        self.Omega = np.asarray(Omega, dtype=np.float64)
        self.d = dphi(model, self.D)
        self.p = num_params(model, self.D, self.J)
        # one-hot group membership for segmented sums
        self.G = np.zeros((self.J, self.N))
        self.G[self.j_ind, np.arange(self.N)] = 1.0

    def split(self, q):
        d, J, D = self.d, self.J, self.D
        phi = q[..., :d]
        eta = q[..., d:d + J]
        if self.model == 'm1b':
            etb = None
        elif self.model == 'm2b':
            etb = q[..., d + J:]                                       # (.., D): shared by the site's groups
        else:
            etb = q[..., d + J:].reshape(q.shape[:-1] + (J, D))
        return phi, eta, etb

    def lp_grad(self, q, e_map=None):
        """q: (nq, p) -> (lp (nq,), grad (nq, p)).  e_map: applied to the residuals e = y - sigmoid(f) before
        they enter the gradient (e.g. the rounding a kernel stores them with); None: exact fp64."""
        q = np.atleast_2d(np.asarray(q, dtype=np.float64))
        nq = q.shape[0]
        D, J, d = self.D, self.J, self.d
        phi, eta, etb = self.split(q)
        if self.model == 'm1b':
            mu_a = 0.0
            sig_a = np.exp(phi[:, 0])
            beta = np.repeat(phi[:, None, 1:1 + D], J, axis=1)          # (nq,J,D)
            sig_b = None
        elif self.model == 'm2b':
            mu_a = 0.0
            sig_a = np.exp(phi[:, 0])
            sig_b = np.exp(phi[:, 1])                                   # scalar scale of the slopes
            beta = np.repeat((etb * sig_b[:, None])[:, None, :], J, axis=1)
        elif self.model == 'm3b':
            mu_a = 0.0
            sig_a = np.exp(phi[:, 0])
            sig_b = np.exp(phi[:, 1:1 + D])
            beta = etb * sig_b[:, None, :]
        else:
            mu_a = phi[:, 0]
            sig_a = np.exp(phi[:, 1])
            sig_b = np.exp(phi[:, 2 + D:2 + 2 * D])
            beta = phi[:, None, 2:2 + D] + etb * sig_b[:, None, :]
        four = self.model in ('m4b', 'm5b')
        laplace = self.model == 'm5b'
        alpha = (mu_a[:, None] if four else 0.0) + eta * sig_a[:, None]   # (nq,J)
        # f[q,n] = alpha[q, j(n)] + x_n . beta[q, j(n)]
        if J == 1:
            f = alpha + beta[:, 0, :] @ self.X.T                       # BLAS path (single group)
        else:
            f = alpha[:, self.j_ind] + np.einsum('nd,qnd->qn', self.X, beta[:, self.j_ind, :])
        with np.errstate(over='ignore', invalid='ignore'):
            lp_lik = np.sum(self.y * f - np.logaddexp(0.0, f), axis=1)
            e = self.y - 1.0 / (1.0 + np.exp(-f))                      # (nq,N)
        if e_map is not None:
            e = e_map(e)
        if J == 1:
            s = e.sum(axis=1, keepdims=True)
            g = (e @ self.X)[:, None, :]
        else:
            s = e @ self.G.T                                           # (nq,J) per-group sum of e
            g = np.einsum('qn,jn,nd->qjd', e, self.G, self.X)          # (nq,J,D) per-group X'e
        dev = phi - self.mu
        c = dev @ self.Omega.T                                     # Omega symmetric
        lp = -0.5 * np.sum(dev * c, axis=1) + lp_lik
        lp -= np.sum(np.abs(eta), axis=1) if laplace else 0.5 * np.sum(eta ** 2, axis=1)
        grad = np.zeros((nq, self.p))
        gphi = -c.copy()
        geta = sig_a[:, None] * s - (np.sign(eta) if laplace else eta)
        if self.model == 'm1b':
            gphi[:, 0] += sig_a * np.sum(eta * s, axis=1)
            gphi[:, 1:1 + D] += g.sum(axis=1)
        elif self.model == 'm2b':
            gs = g.sum(axis=1)                                          # (nq,D) X'e over the whole site
            lp -= 0.5 * np.sum(etb ** 2, axis=1)
            gphi[:, 0] += sig_a * np.sum(eta * s, axis=1)
            gphi[:, 1] += sig_b * np.sum(etb * gs, axis=1)
            grad[:, d + J:] = sig_b[:, None] * gs - etb
        elif self.model == 'm3b':
            lp -= 0.5 * np.sum(etb ** 2, axis=(1, 2))
            gphi[:, 0] += sig_a * np.sum(eta * s, axis=1)
            gphi[:, 1:1 + D] += sig_b * np.sum(etb * g, axis=1)
            grad[:, d + J:] = (sig_b[:, None, :] * g - etb).reshape(nq, -1)
        else:
            lp -= np.sum(np.abs(etb), axis=(1, 2)) if laplace else 0.5 * np.sum(etb ** 2, axis=(1, 2))
            gphi[:, 0] += s.sum(axis=1)
            gphi[:, 1] += sig_a * np.sum(eta * s, axis=1)
            gphi[:, 2:2 + D] += g.sum(axis=1)
            gphi[:, 2 + D:2 + 2 * D] += sig_b * np.sum(etb * g, axis=1)
            grad[:, d + J:] = (sig_b[:, None, :] * g - (np.sign(etb) if laplace else etb)).reshape(nq, -1)
        grad[:, :d] = gphi
        grad[:, d:d + J] = geta
        return lp, grad

    def lp_scalar(self, q):
        """Independent, loop-level evaluation that reads like the Stan model block."""
        q = np.asarray(q, dtype=np.float64)
        phi, eta, etb = self.split(q)
        D = self.D
        lp = -0.5 * (phi - self.mu) @ self.Omega @ (phi - self.mu)      # multi_normal_prec
        if self.model == 'm5b':
            lp += -np.sum(np.abs(eta)) - np.sum(np.abs(etb))            # double_exponential(0,1)
        else:
            lp += -0.5 * np.sum(eta ** 2)                               # eta ~ normal(0,1)
            if etb is not None:
                lp += -0.5 * np.sum(etb ** 2)                           # etb ~ normal(0,1)
        for n in range(self.N):
            j = self.j_ind[n]
            if self.model == 'm1b':
                a = eta[j] * np.exp(phi[0])
                b = phi[1:1 + D]
            elif self.model == 'm2b':
                a = eta[j] * np.exp(phi[0])
                b = etb * np.exp(phi[1])
            elif self.model == 'm3b':
                a = eta[j] * np.exp(phi[0])
                b = etb[j] * np.exp(phi[1:1 + D])
            else:
                a = phi[0] + eta[j] * np.exp(phi[1])
                b = phi[2:2 + D] + etb[j] * np.exp(phi[2 + D:2 + 2 * D])
            fn = a + self.X[n] @ b
            lp += self.y[n] * fn - np.log1p(np.exp(fn))                 # bernoulli_logit
        return lp
