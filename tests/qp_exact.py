"""Exact optimum of a dense convex QP, certified by its KKT conditions (test infrastructure only).

The problem is the OPT operator's (lopt.cpp:35-66):

    minimise 0.5 x'Hx + c'x   subject to   a_i.x = b_i (i < neq),   a_i.x <= b_i (neq <= i < nrows)

with L = [A | b] of shape [nrows, 31] and H the lower triangle of Q mirrored, which is all the solver reads.  This module
shares no code with the solver (csrc/qp_warp.cuh) or with the reference ALGLIB: it is a textbook primal active-set method
on the KKT system in numpy, whose final KKT solve is refined with residuals in extended precision (np.longdouble), and
whose result is certified (strict convexity, stationarity, feasibility, dual feasibility, complementarity) before it is
returned.  A result that fails a check raises CertificationError, so a wrong reference can never pass silently.
"""
import numpy as np

N = 30

# The tolerance rule a solver result must meet against x* (see passes()):
TOL_EXACT = 1e-7        # err <= 1e-7 ...
V_FLOOR = 1e-6          # ... or the solver stopped with a violation v(x) > 1e-6 ...
K_VIOL = 1.0            # ... and err <= K * v(x)
MAX_SECOND = 0.005      # at most 0.5 % of the instances of a group may use the second branch


class CertificationError(AssertionError):
    pass


def sym_lower(Q):
    """H: the lower triangle of Q mirrored onto the upper one."""
    Q = np.asarray(Q, dtype=np.float64)
    return np.tril(Q) + np.tril(Q, -1).T


def _kkt_solve(H, c, Aw, bw, refine=3):
    """Solve [H Aw'; Aw 0] [x; lam] = [-c; bw] in float64, refining with residuals in np.longdouble."""
    n, m = H.shape[0], Aw.shape[0]
    K = np.zeros((n + m, n + m))
    K[:n, :n] = H
    K[:n, n:] = Aw.T
    K[n:, :n] = Aw
    rhs = np.concatenate([-c, bw])
    # symmetric diagonal scaling: the controller's Q spans 1 .. 1e8 (slack weight)
    d = np.ones(n + m)
    dh = np.sqrt(np.abs(np.diag(H)))
    d[:n] = 1.0 / np.where(dh > 0, dh, 1.0)
    if m:
        an = np.linalg.norm(Aw * d[None, :n], axis=1)
        d[n:] = 1.0 / np.where(an > 0, an, 1.0)
    Ks = K * d[:, None] * d[None, :]
    Kl = K.astype(np.longdouble)
    rl = rhs.astype(np.longdouble)
    z = d * np.linalg.solve(Ks, d * rhs)
    for _ in range(refine):
        r = rl - Kl @ z.astype(np.longdouble)
        dz = d * np.linalg.solve(Ks, d * np.asarray(r, dtype=np.float64))
        z = z + dz
    return z[:n], z[n:]


def _independent(Aw, a, tol=1e-10):
    """Is row a linearly independent of the rows of Aw?"""
    if Aw.shape[0] == 0:
        return np.linalg.norm(a) > 0
    if Aw.shape[0] >= Aw.shape[1]:
        return False
    coef, *_ = np.linalg.lstsq(Aw.T, a, rcond=None)
    return np.linalg.norm(Aw.T @ coef - a) > tol * np.linalg.norm(a)


def violation(x, L, neq):
    """v(x): largest |a.x - b| over equality rows and (a.x - b)+ over inequality rows, each divided by max(1, |b_i|)."""
    L = np.asarray(L, dtype=np.float64)
    if L.shape[0] == 0:
        return 0.0
    r = (L[:, :N] @ x - L[:, N]) / np.maximum(1.0, np.abs(L[:, N]))
    r[:neq] = np.abs(r[:neq])
    r[neq:] = np.maximum(r[neq:], 0.0)
    return float(r.max())


def objective(Q, c, x):
    H = sym_lower(Q)
    return float(0.5 * x @ H @ x + c @ x)


def exact_qp(Q, c, L, neq, x0=None, maxit=500):
    """x*, the multipliers lam [nrows] (>= 0 on inequality rows), the active set (row indices) and the certificate dict.

    A primal active-set method warm-started from x0 (the solver's x is a good guess).  While the iterate is infeasible,
    the most violated row (scaled by max(1, |b_i|)) joins the working set; once feasible, the classic method runs: step to
    the working set's minimiser with a ratio test, drop the row with the most negative multiplier at a minimiser."""
    H = sym_lower(Q)
    c = np.asarray(c, dtype=np.float64)
    L = np.asarray(L, dtype=np.float64).reshape(-1, N + 1)
    nrows = L.shape[0]
    A, b = L[:, :N], L[:, N]
    bs = np.maximum(1.0, np.abs(b))
    try:
        np.linalg.cholesky(H)
    except np.linalg.LinAlgError:
        raise CertificationError("H is not positive definite: the optimum is not unique")
    x = np.zeros(N) if x0 is None else np.asarray(x0, dtype=np.float64).copy()
    W = list(range(neq))
    for i in range(neq, nrows):
        if A[i] @ x - b[i] >= -1e-9 * bs[i] and _independent(A[W], A[i]):
            W.append(i)
    feasible = False
    for _ in range(maxit):
        xw, lw = _kkt_solve(H, c, A[W], b[W])
        if not feasible:
            r = (A @ xw - b) / bs
            r[:neq] = 0.0
            r[W] = 0.0
            j = int(np.argmax(r)) if nrows else -1
            if nrows and r[j] > 1e-12:
                if not _independent(A[W], A[j]):
                    # drop the working row with the most negative multiplier to make room
                    ineq = [k for k, i in enumerate(W) if i >= neq]
                    if not ineq:
                        raise CertificationError("infeasible equality-constrained QP")
                    W.pop(min(ineq, key=lambda k: lw[k]))
                    continue
                W.append(j)
                continue
            feasible = True
            x = xw
            continue
        p = xw - x
        if np.abs(p).max() <= 1e-14 * max(1.0, np.abs(x).max()):
            x = xw
            neg = [(lw[k], k) for k, i in enumerate(W) if i >= neq and lw[k] < 0.0]
            if not neg or min(neg)[0] >= -1e-13 * max(1.0, np.abs(lw).max()):
                break
            W.pop(min(neg)[1])
            continue
        ap = A @ p
        alpha, block = 1.0, -1
        for i in range(neq, nrows):
            if i in W or ap[i] <= 1e-15 * np.abs(A[i]).max() * np.abs(p).max():
                continue
            t = (b[i] - A[i] @ x) / ap[i]
            if t < alpha:
                alpha, block = max(t, 0.0), i
        x = x + alpha * p
        if block >= 0:
            W.append(block)
    else:
        raise CertificationError("active-set method did not converge in %d iterations" % maxit)
    x, lw = _kkt_solve(H, c, A[W], b[W])
    lam = np.zeros(nrows)
    lam[W] = lw
    cert = certify(H, c, A, b, neq, x, lam)
    return x, lam, sorted(W), cert


def certify(H, c, A, b, neq, x, lam, tol=1e-10):
    """Check the KKT conditions in extended precision; raise CertificationError if one fails.  Returns the residuals."""
    Hl, cl, Al, bl = (np.asarray(v, dtype=np.longdouble) for v in (H, c, A, b))
    xl, ll = np.asarray(x, dtype=np.longdouble), np.asarray(lam, dtype=np.longdouble)
    g = Hl @ xl + cl + Al.T @ ll
    gscale = max(1.0, float(np.abs(c).max()) if c.size else 1.0, float((np.abs(H) @ np.abs(x)).max()),
                 float((np.abs(A.T) @ np.abs(lam)).max()) if A.shape[0] else 0.0)
    stat = float(np.abs(g).max()) / gscale
    r = np.asarray(Al @ xl - bl, dtype=np.float64)
    rscale = np.maximum(1.0, np.maximum(np.abs(b), np.abs(A) @ np.abs(x))) if A.shape[0] else np.ones(0)
    feas_eq = float((np.abs(r[:neq]) / rscale[:neq]).max()) if neq else 0.0
    feas_in = float((np.maximum(r[neq:], 0.0) / rscale[neq:]).max()) if A.shape[0] > neq else 0.0
    lscale = max(1.0, float(np.abs(lam).max()) if lam.size else 0.0)
    dual = float(np.maximum(-lam[neq:], 0.0).max()) / lscale if A.shape[0] > neq else 0.0
    comp = float(np.abs(lam[neq:] * r[neq:] / rscale[neq:]).max()) / lscale if A.shape[0] > neq else 0.0
    cert = dict(stationarity=stat, feas_eq=feas_eq, feas_ineq=feas_in, dual=dual, complementarity=comp)
    bad = {k: v for k, v in cert.items() if not v <= tol}
    if bad:
        raise CertificationError("KKT certificate failed: %s" % bad)
    return cert


def err(x, xs):
    """max|x - x*| / max(1, max|x*|)"""
    return float(np.abs(x - xs).max() / max(1.0, np.abs(xs).max()))


def passes(e, v, flat=False):
    """The tolerance rule: (passes, used_second_branch).  flat=True: err <= 1e-7 with no second branch."""
    if e <= TOL_EXACT:
        return True, False
    if flat:
        return False, False
    return (v > V_FLOOR and e <= K_VIOL * v), True


class Tally:
    """Applies the tolerance rule over a group of instances and reports what the printout of the group needs."""

    def __init__(self, what, flat=False):
        self.what, self.flat = what, flat
        self.n = 0
        self.worst = 0.0
        self.second = []          # (instance, err, v)
        self.failed = []

    def add(self, i, e, v):
        ok, second = passes(e, v, self.flat)
        self.n += 1
        self.worst = max(self.worst, e)
        if not ok:
            self.failed.append((i, e, v))
        elif second:
            self.second.append((i, e, v))

    def report(self):
        ratio = max((e / v for _, e, v in self.second), default=0.0)
        return ("%s: %d instances, worst err %.3e, second branch %d (worst err/v %.3f), failed %d"
                % (self.what, self.n, self.worst, len(self.second), ratio, len(self.failed)))

    def check(self):
        print(self.report())
        assert not self.failed, "%s: outside the tolerance rule: %s" % (self.what, self.failed[:5])
        assert len(self.second) <= MAX_SECOND * self.n, "%s: %d of %d instances needed the violation branch" % (
            self.what, len(self.second), self.n)


def known_answer_qp(rng, nrows, neq, nact=None, cond=1e3):
    """A QP whose optimum is known by construction: pick x*, an active set and multipliers lam > 0, derive c and b.
    Returns (Q, c, L, x*, lam, active rows) with Q = H symmetric."""
    nin = nrows - neq
    if nact is None:
        nact = int(rng.integers(0, min(nin, N - neq) + 1)) if nin else 0
    U, _ = np.linalg.qr(rng.standard_normal((N, N)))
    ev = np.exp(rng.uniform(0.0, np.log(cond), N))
    H = (U * ev) @ U.T
    H = 0.5 * (H + H.T)
    A = rng.standard_normal((nrows, N))
    xs = rng.uniform(-2.0, 2.0, N)
    act = list(range(neq)) + list(neq + rng.choice(nin, nact, replace=False)) if nrows else []
    lam = np.zeros(nrows)
    if neq:
        lam[:neq] = rng.standard_normal(neq)
    ina = [i for i in act if i >= neq]
    lam[ina] = rng.uniform(0.1, 2.0, len(ina))
    b = A @ xs if nrows else np.zeros(0)
    slack = rng.uniform(0.1, 2.0, nrows)
    inactive = np.ones(nrows, dtype=bool)
    inactive[act] = False
    b[inactive] += slack[inactive]
    c = -(H @ xs + A.T @ lam)
    L = np.hstack([A, b[:, None]]) if nrows else np.zeros((0, N + 1))
    return H, c, L, xs, lam, sorted(act)
