"""Row-by-row restatement of the reference's translation-symmetric spin-1/2 sectors, for halves of up to 18 bits.

TEST INFRASTRUCTURE ONLY.  tests/repr_builders.py enumerates a whole sector, which stops at 32 sites.  This module
builds only the sublattice tables (2^(N/2) entries per translation) and applies the same convention to given rows:
whether a state is its orbit's representative, its norm, and the row of the matrix-free product
    (H x)_r = diag_r x_r + sum_bonds sqrt(nu_r / nu_j) * (J/2) * exp(2 pi i k.disp_i / L) * x_j
(model<T>::MultMv2, repr branch, src/model.cc:1016-1107; rows of zero norm: fake_pos + r/dim).  The rules (canon, zip,
unzip, translations of the halves) are repr_builders.Sector's own methods, run on these tables.
"""
import cmath
import math

import numpy as np

import repr_builders as R


class SectorTables(R.Sector):
    """repr_builders.Sector without the enumeration: tables and per-state rules of one (lattice, k)."""

    def __init__(self, L, k):                     # noqa: super().__init__ would enumerate the sector
        par = self.par = R.Lattice(L)
        sub = self.sub = par.child()
        self.k = [int(x) for x in k]
        N, Ns = par.N, par.N // 2
        self.N, self.Ns = N, Ns
        u = np.uint64
        allsub = np.arange(1 << Ns, dtype=u)
        splans = [sub.plan(d) for d in sub.disps]
        self.subT = np.stack([R._apply_plan(allsub, p) for p in splans])
        rep = self.subT.min(axis=0).astype(np.int64)                 # first state of the orbit in integer order
        dist = np.zeros(1 << Ns, dtype=np.int64)
        for jd in range(len(splans) - 1, -1, -1):                     # first displacement that reaches the state
            dist[self.subT[jd][rep] == allsub] = jd
        self.rep, self.dist = rep, dist
        self.ntrans = len(par.disps)
        sp_index = {tuple(p): j for j, p in enumerate(splans)}
        self.fwd = []
        for d in par.disps:
            p = par.plan(d)
            if p[0] % 2 == 0:
                self.fwd.append((False, sp_index[tuple(p[2 * t] // 2 for t in range(Ns))],
                                 sp_index[tuple((p[2 * t + 1] - 1) // 2 for t in range(Ns))]))
            else:
                self.fwd.append((True, sp_index[tuple(p[2 * t + 1] // 2 for t in range(Ns))],
                                 sp_index[tuple((p[2 * t] - 1) // 2 for t in range(Ns))]))
        dindex = {d: i for i, d in enumerate(par.disps)}
        self.inv = [self.fwd[dindex[tuple((-x) % l for x, l in zip(d, par.L))]] for d in par.disps]
        self.compat = [sum(self.k[q] % par.L[q] * d[q] * (N // par.L[q]) for q in range(par.dim)) % N for d in par.disps]
        self.phase = []
        for d in par.disps:                                           # src/model.cc:808-814
            e = 0.0
            for q in range(par.dim):
                e += self.k[q] * d[q] / float(par.L[q])
            self.phase.append(cmath.exp(complex(0.0, 2.0 * math.pi * e)))

    def representative_and_norm(self, states):
        """(is the state its orbit's representative under the reference's rule, norm_trans_repr of the state)."""
        st = np.asarray(states, dtype=np.uint64)
        a, b = self.unzip(st)
        _, ca, cb = self.canon(a, b)
        is_rep = (ca == a) & (cb == b)
        cnt = np.zeros(st.size, dtype=np.int64)
        ok = np.ones(st.size, dtype=bool)
        for i in range(self.ntrans):
            ai, bi = self._move(self.fwd[i], a, b)
            fixed = (ai == a) & (bi == b)
            cnt += fixed
            if self.compat[i] != 0:
                ok &= ~fixed
        return is_rep, np.where(ok, (self.ntrans // np.maximum(cnt, 1)).astype(np.float64), 0.0)

    def rows_times(self, states, nu, bonds, rows, x, J=1.0, fake_pos=100.0):
        """(H x)[rows] of the matrix-free product; states / nu: the whole sector in row order (any order of bit patterns)."""
        u = np.uint64
        states = np.asarray(states, dtype=u)
        byval = np.argsort(states, kind="stable")
        srt = states[byval]
        n = states.size
        rows = np.asarray(rows, dtype=np.int64)
        st = states[rows]
        bonds = sorted((min(p, q), max(p, q)) for (p, q) in bonds)
        live = nu[rows] > 0
        diag = np.zeros(rows.size)
        for (p, q) in bonds:
            par = ((st >> u(p)) & u(1)) == ((st >> u(q)) & u(1))
            diag = diag + np.where(par, 0.25 * J, -0.25 * J)
        diag = np.where(live, diag, fake_pos + rows / float(n))
        y = diag * x[rows]
        ph = np.asarray(self.phase)
        for (p, q) in bonds:
            act = np.nonzero(live & (((st >> u(p)) & u(1)) != ((st >> u(q)) & u(1))))[0]
            if act.size == 0:
                continue
            s2 = st[act] ^ u((1 << p) | (1 << q))
            i, ca, cb = self.canon(*self.unzip(s2))
            t = self.zip(ca, cb)
            pos = np.minimum(np.searchsorted(srt, t), n - 1)
            found = srt[pos] == t
            j = byval[pos]
            keep = found & (nu[j] > 0)
            act, i, j = act[keep], i[keep], j[keep]
            w = np.sqrt(nu[rows[act]] / nu[j]) * (0.5 * J)
            np.add.at(y, act, w * ph[i] * x[j])
        return y
