"""CPU test double of epstan._lib.Context, built on the oracle, so that the
HOST-side logic of the multi-rank Master (site sharding, the natural-parameter
all-reduce, flag consensus, gathering of the mirrors) can run over gloo in a
container without a GPU.  Lives under tests/: the product never imports it."""

import numpy as np
import torch

from epstan._lib import EpgError
from oracle import ep_linalg as orc

(Q, R, Q0, R0, QI, RI, QI2, RI2, DQI, DRI, CAVQ, CAVM, S, M, PARTIAL, TMEAN, DSUM) = range(17)
XCHG_SLOTS = 64
_SITE3 = (QI, QI2, DQI, CAVQ)
_SITE2 = (RI, RI2, DRI, CAVM, TMEAN)


class OracleContext(object):
    def __init__(self, device=0, stream=None):
        self.device = device
        self.K = self.d = 0
        self._launches = 0

    def init_state(self, K, d):
        self.K, self.d = K, d
        self.a = {}
        for i in _SITE3:
            self.a[i] = np.zeros((d, d, K))
        for i in _SITE2:
            self.a[i] = np.zeros((d, K))
        for i in (Q, Q0, S):
            self.a[i] = np.zeros((d, d))
        for i in (R, R0, M):
            self.a[i] = np.zeros(d)
        self.a[PARTIAL] = np.zeros(d * d + d + 1)
        self._partial_t = torch.from_numpy(self.a[PARTIAL])
        self.a[DSUM] = np.zeros(d * d + d + 2 + XCHG_SLOTS)
        self._qprev = None
        self._dsum_t = torch.from_numpy(self.a[DSUM])
        self._ok = np.zeros(K, dtype=bool)    # (epg_init_state clears the site flags)
        self.draws = None
        self.U = None

    def upload(self, array, host, k0=0, k1=None):
        k1 = self.K if k1 is None else k1
        host = np.asarray(host, dtype=np.float64)
        if array in _SITE3:
            self.a[array][:, :, k0:k1] = host.reshape(self.d, self.d, k1 - k0, order='F')
        elif array in _SITE2:
            self.a[array][:, k0:k1] = host.reshape(self.d, k1 - k0, order='F')
        else:
            self.a[array][...] = host.reshape(self.a[array].shape, order='F')

    def download(self, array, out, k0=0, k1=None):
        k1 = self.K if k1 is None else k1
        if array in _SITE3:
            src = self.a[array][:, :, k0:k1]
        elif array in _SITE2:
            src = self.a[array][:, k0:k1]
        else:
            src = self.a[array]
        out[...] = src.reshape(out.shape, order='F')
        return out

    def partial_tensor(self):
        return self._partial_t

    def dsum_tensor(self):
        return self._dsum_t

    def delta_sums(self, with_norms=True, slots=None):
        d = self.d
        S2 = sum(orc.fisher_norm2(self.a[Q], self.a[R], self.a[DQI][:, :, k], self.a[DRI][:, k])
                 for k in range(self.K) if self._ok[k]) if with_norms else 0.0
        self._qprev = (self.a[Q].copy(), self.a[R].copy())
        self.a[DSUM][d * d + d + 2:] = 0.0
        if slots is not None:
            self.a[DSUM][d * d + d + 2:d * d + d + 2 + len(slots)] = slots
        self.a[DSUM][:d * d] = self.a[DQI].sum(axis=2).ravel(order='F')
        self.a[DSUM][d * d:d * d + d] = self.a[DRI].sum(axis=1)
        self.a[DSUM][d * d + d] = S2
        self.a[DSUM][d * d + d + 1] = self._ok.sum()

    def _sums(self, what):
        if self._qprev is None:
            raise EpgError(what + ": call epg_delta_sums(_ex) first")
        return self._qprev

    def delta_snr(self):
        # (the Fisher metric of the (Q, r) that delta_sums snapshotted, as epg_delta_snr)
        d = self.d
        Qp, rp = self._sums('epg_delta_snr')
        T2 = orc.fisher_norm2(Qp, rp, self.a[DSUM][:d * d].reshape(d, d, order='F'),
                              self.a[DSUM][d * d:d * d + d])
        return T2, float(self.a[DSUM][d * d + d]), int(round(self.a[DSUM][d * d + d + 1]))

    def read_exchange(self):
        d = self.d
        b = self.a[DSUM]
        return float(b[d * d + d]), int(round(b[d * d + d + 1])), b[d * d + d + 2:].copy()

    def mix_phi_sums(self, n):
        d = self.d
        out = np.zeros(d + 2 * d * d)
        for k in range(self.K):
            x = self.draws[k]
            mk = x.mean(axis=1)
            xc = x - mk[:, None]
            out[:d] += mk
            out[d:d + d * d] += (xc @ xc.T).ravel(order='F')
            out[d + d * d:] += np.outer(mk, mk).ravel(order='F')
        return out

    def update_from_sums(self, df):
        d = self.d
        Qp, rp = self._sums('epg_update_from_sums')
        self.a[PARTIAL][:d * d] = ((Qp - self.a[Q0]) + df * self.a[DSUM][:d * d].reshape(d, d, order='F')).ravel(order='F')
        self.a[PARTIAL][d * d:d * d + d] = (rp - self.a[R0]) + df * self.a[DSUM][d * d:d * d + d]

    def on_torch_stream(self):
        return True

    def launch_count(self):
        return self._launches

    def cavity(self, k0=0, k1=None, proposal=False):
        k1 = self.K if k1 is None else k1
        Qs, rs = (self.a[QI2], self.a[RI2]) if proposal else (self.a[QI], self.a[RI])
        flags = np.zeros(k1 - k0, dtype=bool)
        for k in range(k0, k1):
            ok, P, mu = orc.cavity(self.a[Q], self.a[R], Qs[:, :, k], rs[:, k])
            flags[k - k0] = ok
            self.a[CAVQ][:, :, k] = P
            self.a[CAVM][:, k] = mu
        self._ok[k0:k1] = flags             # epg_cavity owns the site flags too (include/epgpu.h)
        return flags, bool(flags.all())

    def set_draws(self, draws, n, k0=0, k1=None):
        k1 = self.K if k1 is None else k1
        if self.draws is None or self.draws.shape[2] != n:
            self.draws = np.zeros((self.K, self.d, n))
        self.draws[k0:k1] = np.asarray(draws).reshape(k1 - k0, self.d, n)

    def get_draws(self, n, k0=0, k1=None):
        return self.draws[k0:(self.K if k1 is None else k1)].copy()

    def moments(self, n, prec_estim='sample', k0=0, k1=None):
        k1 = self.K if k1 is None else k1
        flags = np.zeros(k1 - k0, dtype=bool)
        for k in range(k0, k1):
            ok, dQ, dr = orc.tilted_moments(self.draws[k].T, self.a[Q], self.a[R], prec_estim)
            flags[k - k0] = ok
            self.a[DQI][:, :, k], self.a[DRI][:, k] = dQ, dr
            self.a[TMEAN][:, k] = self.draws[k].mean(axis=1)
        self._ok[k0:k1] = flags
        return flags, int(flags.sum())

    def fail_sites(self, sites):
        for k in sites:
            self.a[DQI][:, :, k] = 0.0
            self.a[DRI][:, k] = 0.0
            self._ok[k] = False

    def reinit_sites(self, sites):
        self.reinit_marks = getattr(self, 'reinit_marks', []) + [int(k) for k in sites]

    def update_partial(self, df):
        self.a[QI2][...] = self.a[QI] + df * self.a[DQI]
        self.a[RI2][...] = self.a[RI] + df * self.a[DRI]
        d = self.d
        self.a[PARTIAL][:d * d] = self.a[QI2].sum(axis=2).ravel(order='F')
        self.a[PARTIAL][d * d:d * d + d] = self.a[RI2].sum(axis=1)

    def update_finish(self):
        d = self.d
        self.a[Q][...] = self.a[Q0] + self.a[PARTIAL][:d * d].reshape(d, d, order='F')
        self.a[R][...] = self.a[R0] + self.a[PARTIAL][d * d:d * d + d]
        try:
            self.U = orc._chol_upper(self.a[Q])
            return True
        except orc.NotPosDef:
            return False

    def accept(self):
        self.a[QI], self.a[QI2] = self.a[QI2], self.a[QI]
        self.a[RI], self.a[RI2] = self.a[RI2], self.a[RI]

    def global_moments(self, m_out=None, S_out=None):
        Sm, mm = orc.invert_normal_params(self.U, self.a[R], cho_form=True)
        self.a[S][...], self.a[M][...] = Sm, mm
        if m_out is not None:
            m_out[...] = mm
        if S_out is not None:
            S_out[...] = Sm

    def force_pd(self, thr, min_eig):
        forced = np.zeros(self.K, dtype=bool)
        lam = np.zeros(self.K)
        for k in range(self.K):
            lam[k] = orc.min_eig(self.a[QI2][:, :, k])
            if lam[k] < thr:
                self.a[QI][np.arange(self.d), np.arange(self.d), k] += min_eig - lam[k]
                forced[k] = True
        self._ok[:] = forced                # (so does epg_force_pd)
        return forced, lam

    def set_option(self, name, value):
        pass

    def close(self):
        pass
