"""numpy restatement of model::moprXvec_repr (src/model.cc:1716-1846) for one-site electron operators between the momentum
sectors of tests/repr_builders_fermion.py, and an independent full-basis computation to check it against.

TEST INFRASTRUCTURE ONLY.  Operators, A = sum_r c_r O_r:
  * density     O_r = cu_r n_up,r + cd_r n_dn,r (S^z_q: cd = -cu; charge n_q: cd = cu);
  * spin flip   O_r = c+_{r,dn} c_{r,up} (S^-) or c+_{r,up} c_{r,dn} (S^+);
  * fermion     O_r = c_{r,s} or c+_{r,s}.
Sign of a single-electron operator: oprXphi's rule (src/basis.cc:2717-2731; the two halves of the device's el_hop): the parity
of the electrons below site r (bits below 2r), and for spin down also the up electron of site r itself, counted on the state
before the operator acts.  The reference's scatter (`apply_scatter`): every term acts on the OLD representative j, the
produced state is T_t (representative i of the NEW sector) and
    y_i += sqrt(nu_old[j] / nu_new[i]) * x_j * c_r * conj(phase_new[t]) * (-1)^(operator sign + translation sign of (rep_i, t)).
`apply_gather` is the form the device computes (every output row written once, terms in site order): A^+ = sum conj(c_r) O_r^+
acts on the NEW representative i, the result is mapped into the OLD sector by the same rule, and y_i takes the conjugate of
that element times x_j.  For coefficients e^{+i q.r} (a vector at momentum K goes to K + q) the two are the same matrix.
"""
import numpy as np

import repr_builders as R
import repr_builders_fermion as F

PREC = 2e-12                      # lanczos_precision, src/miscellaneous.cc:47
u = np.uint64


def _sign_below(st, r, sp):
    """oprXphi's sign for an operator on (r, sp), counted on the state it acts on."""
    sg = F._fermions_below(st, r)
    if sp == 1:
        sg = sg ^ ((st >> u(2 * r)) & u(1)).astype(np.int64)
    return sg


def _one(st, r, sp, create):
    """c_{r,sp} (create=False) or c+_{r,sp}: (applicable, new state, sign)."""
    b = u(1 << (2 * r + sp))
    ok = ((st & b) == 0) if create else ((st & b) != 0)
    return ok, st ^ b, _sign_below(st, r, sp)


def term(kind, st, r, lower=True, create=False, spin=0):
    """O_r on the patterns st: (applicable, new state, sign).  kind: "flip" (lower: S^- = c+_dn c_up, else S^+) or "fermion"."""
    if kind == "flip":
        a_sp, c_sp = (0, 1) if lower else (1, 0)
        ok1, s1, g1 = _one(st, r, a_sp, False)
        ok2, s2, g2 = _one(s1, r, c_sp, True)
        return ok1 & ok2, s2, g1 ^ g2
    return _one(st, r, spin, create)


def adjoint(kind, lower=True, create=False, spin=0):
    """Keyword arguments of the adjoint term."""
    if kind == "flip":
        return dict(lower=not lower)
    return dict(create=not create, spin=spin)


def _map(S_src, S_tgt, kind, coef, x, kw, conj_phase):
    """y_i += sqrt(nu_src[j]/nu_tgt[i]) x_j c_r phase(t) (-1)^(...) over the terms acting on the representatives of S_src."""
    y = np.zeros(S_tgt.n, dtype=np.complex128)
    rows = np.nonzero((np.abs(x) >= PREC) & (S_src.nu >= PREC))[0]
    ph = np.asarray(S_tgt.phase)
    ph = np.conj(ph) if conj_phase else ph
    for r in range(S_src.N):
        ok, s2, sg = term(kind, S_src.states[rows], r, **kw)
        act, s2, sg = rows[ok], s2[ok], sg[ok]
        if act.size == 0:
            continue
        a2, b2 = S_tgt.unzip(s2)
        i, ca, cb = S_tgt.canon(a2, b2)
        tgt = S_tgt.index(ca, cb)
        keep = S_tgt.nu[tgt] >= PREC
        act, i, tgt, sg, ca, cb = act[keep], i[keep], tgt[keep], sg[keep], ca[keep], cb[keep]
        tsg = np.zeros(act.size, dtype=np.int64)
        cst = S_tgt.zip(ca, cb)
        for ti in np.unique(i):
            sel = i == ti
            tsg[sel] = S_tgt.translation_sign(cst[sel], int(ti))
        val = np.sqrt(S_src.nu[act] / S_tgt.nu[tgt]) * x[act] * coef[r] * ph[i]
        val = np.where((sg ^ tsg) == 1, -val, val)
        np.add.at(y, tgt, val)
    return y


def apply_scatter(S_old, S_new, kind, coef, x, **kw):
    """The reference's off-diagonal branch (src/model.cc:1762-1834) for kind "flip" or "fermion"."""
    return _map(S_old, S_new, kind, np.asarray(coef, dtype=np.complex128), np.asarray(x, dtype=np.complex128), kw, True)


def apply_gather(S_old, S_new, kind, coef, x, **kw):
    """The same operator row by row of the new sector, through the adjoint: the matrix element (i, j) is the conjugate of the
    element (j, i) of A^+ = sum conj(c_r) O_r^+ mapped from S_new into S_old.  Only rows j with |x_j| >= PREC count."""
    coef = np.asarray(coef, dtype=np.complex128)
    x = np.asarray(x, dtype=np.complex128)
    y = np.zeros(S_new.n, dtype=np.complex128)
    live = np.nonzero(S_new.nu >= PREC)[0]
    akw = adjoint(kind, **kw)
    ph = np.asarray(S_old.phase)
    for r in range(S_new.N):
        ok, s2, sg = term(kind, S_new.states[live], r, **akw)
        act, s2, sg = live[ok], s2[ok], sg[ok]
        if act.size == 0:
            continue
        a2, b2 = S_old.unzip(s2)
        t, ca, cb = S_old.canon(a2, b2)
        j = S_old.index(ca, cb)
        keep = (S_old.nu[j] >= PREC) & (np.abs(x[j]) >= PREC)
        act, t, j, sg, ca, cb = act[keep], t[keep], j[keep], sg[keep], ca[keep], cb[keep]
        tsg = np.zeros(act.size, dtype=np.int64)
        cst = S_old.zip(ca, cb)
        for ti in np.unique(t):
            sel = t == ti
            tsg[sel] = S_old.translation_sign(cst[sel], int(ti))
        val = np.sqrt(S_new.nu[act] / S_old.nu[j]) * coef[r] * ph[t] * x[j]
        val = np.where((sg ^ tsg) == 1, -val, val)
        np.add.at(y, act, val)
    return y


def apply_density(S_old, S_new, cu, cd, x):
    """Diagonal branch (src/model.cc:1758-1761): y_j = sqrt(nu_old[j]/nu_new[j]) x_j sum_r (cu_r n_up,r + cd_r n_dn,r)(state_j)."""
    assert S_old.n == S_new.n and np.array_equal(S_old.states, S_new.states)
    x = np.asarray(x, dtype=np.complex128)
    ok = (np.abs(x) >= PREC) & (S_old.nu >= PREC) & (S_new.nu >= PREC)
    t = np.zeros(S_old.n, dtype=np.complex128)
    t[ok] = np.sqrt(S_old.nu[ok] / S_new.nu[ok]) * x[ok]
    d = np.zeros(S_old.n, dtype=np.complex128)
    st = S_old.states
    for r in range(S_old.N):
        d += cu[r] * ((st >> u(2 * r)) & u(1)).astype(float) + cd[r] * ((st >> u(2 * r + 1)) & u(1)).astype(float)
    return t * d


def plane_wave(L, k, sign=+1):
    """e^{sign i 2 pi k.r / L} per site (site numbering of the reference's lattice: first even direction fastest)."""
    lat = R.Lattice(L)
    c = np.zeros(lat.N, dtype=np.complex128)
    for s in range(lat.N):
        e = sum(k[d] * lat.coor[s][d] / float(L[d]) for d in range(len(L)))
        c[s] = np.exp(sign * 2j * np.pi * e)
    return c


def dense_sector(L, nup, ndn, k, t=1.0, U=1.1):
    """(restated sector, dense Hermitian H) from tests/repr_builders_fermion.py's upper-triangle csr_mat."""
    S, ia, ja, val = F.hubbard_sector_upper_csr(L, nup, ndn, k, F.square_hops(*L), t, U)
    rows = np.repeat(np.arange(S.n), np.diff(ia))
    A = np.zeros((S.n, S.n), dtype=np.complex128)
    A[rows, ja] = val
    return S, A + np.triu(A, 1).conj().T


# ------------------------------------------------------------------ independent full basis: occupation numbers, own mode order
class FullBasis:
    """Hubbard model on the Lx x Ly torus (site x + y Lx) in plain occupation numbers; Jordan-Wigner mode order: all up modes
    (site order), then all down modes -- not the reference's interleaved order, so nothing is shared with the restatement
    but the model."""

    def __init__(self, L, nup, ndn, t=1.0, U=1.1):
        from itertools import combinations
        self.L, self.N = list(L), int(np.prod(L))
        N = self.N
        ups = [sum(1 << s for s in c) for c in combinations(range(N), nup)]
        dns = [sum(1 << s for s in c) for c in combinations(range(N), ndn)]
        self.states = np.array(sorted(a | (b << N) for a in ups for b in dns), dtype=np.int64)
        self.index = {int(s): i for i, s in enumerate(self.states)}
        self.nup, self.ndn = nup, ndn
        self.t, self.U = t, U

    def mode(self, r, sp):
        return r + sp * self.N

    def apply_mode(self, s, m, create):
        """c_m / c+_m on one pattern: (new pattern, sign) or None."""
        if bool((s >> m) & 1) == create:
            return None
        sg = -1 if bin(s & ((1 << m) - 1)).count("1") & 1 else 1
        return s ^ (1 << m), sg

    def hamiltonian(self):
        Lx, Ly = self.L
        n = self.states.size
        H = np.zeros((n, n))
        bonds = []
        for x in range(Lx):
            for y in range(Ly):
                i = x + y * Lx
                bonds += [(i, (x + 1) % Lx + y * Lx), (i, x + ((y + 1) % Ly) * Lx)]
        for col, s in enumerate(self.states):
            s = int(s)
            H[col, col] += self.U * bin(s & (s >> self.N) & ((1 << self.N) - 1)).count("1")
            for i, j in bonds:
                for sp in (0, 1):
                    for a, b in ((i, j), (j, i)):
                        r1 = self.apply_mode(s, self.mode(b, sp), False)
                        if r1 is None:
                            continue
                        r2 = self.apply_mode(r1[0], self.mode(a, sp), True)
                        if r2 is None:
                            continue
                        H[self.index[r2[0]], col] += -self.t * r1[1] * r2[1]
        return H

    def apply_fermion(self, target, coef, x, create, spin):
        """sum_r coef[r] c(+)_{r,spin} x -> vector of `target` (a FullBasis with the matching particle numbers)."""
        y = np.zeros(target.states.size, dtype=np.complex128)
        for col, s in enumerate(self.states):
            if x[col] == 0:
                continue
            for r in range(self.N):
                res = self.apply_mode(int(s), self.mode(r, spin), create)
                if res is not None:
                    y[target.index[res[0]]] += coef[r] * res[1] * x[col]
        return y

    def plane_wave(self, k, sign=+1):
        Lx, Ly = self.L
        return np.array([np.exp(sign * 2j * np.pi * (k[0] * (r % Lx) / Lx + k[1] * (r // Lx) / Ly)) for r in range(self.N)])
