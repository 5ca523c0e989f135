"""The certified optimum of tests/qp_exact.py, hardened for QPs whose limits bind (test infrastructure only).

Near the controller's joint and torque limits, qp_exact.exact_qp can fail to return a certified optimum:

  * its first phase (the most violated row joins the working set) is a heuristic, and where more rows than variables meet at
    a vertex it cycles, dropping and re-adding the same rows, or reaches a working set whose KKT matrix is singular;
  * its final KKT solve refines three times; at a vertex of nearly dependent rows (multipliers of 1e13) that leaves row
    residuals of 1e-10, and an x 2e-9 from one that meets the rows to 1e-16.

certified_qp settles both.  It decides feasibility first with a linear program (lp_margin, scipy's HiGHS), which shares no code
with any QP solver here.  It restarts the classic primal active-set method from the LP's point, which meets every inequality
row with slack, where exact_qp fails.  It always re-solves the final working set's KKT system with ten refinement steps.
Whichever way x was found, it must pass qp_exact.certify, whose checks and tolerance are unchanged.
"""
import numpy as np

from tests import qp_exact as E

N = E.N
REFINE = 10


def lp_margin(L, neq):
    """Feasibility of the rows of L decided by a linear program:

        t* = min t   subject to   a_i.x = b_i (i < neq),   (a_i.x - b_i) / max(1, |b_i|) <= t (inequality rows),   t >= -1.

    t* > 0: no point meets the rows, the QP is infeasible, and t* is the least row-scaled violation any point can have.
    t* <= 0: the returned x meets the equality rows and every inequality row with a row-scaled slack of at least -t*.
    Returns (t*, x); (inf, None) when the equality rows alone admit no point."""
    from scipy.optimize import linprog
    L = np.asarray(L, dtype=np.float64).reshape(-1, N + 1)
    A, b = L[:, :N], L[:, N]
    s = np.maximum(1.0, np.abs(b))
    nin = L.shape[0] - neq
    cost = np.zeros(N + 1)
    cost[N] = 1.0
    r = linprog(cost, A_ub=np.hstack([A[neq:] / s[neq:, None], -np.ones((nin, 1))]) if nin else None,
                b_ub=b[neq:] / s[neq:] if nin else None,
                A_eq=np.hstack([A[:neq] / s[:neq, None], np.zeros((neq, 1))]) if neq else None, b_eq=b[:neq] / s[:neq] if neq else None,
                bounds=[(None, None)] * N + [(-1.0, None)], method="highs")
    if r.status == 2:
        return np.inf, None
    if r.status != 0:
        raise E.CertificationError("the feasibility LP did not solve: %s" % r.message)
    return float(r.fun), r.x[:N]


def _from_feasible(H, c, A, b, neq, x, maxit):
    """The classic primal active-set method from a point x that meets every row (exact_qp's second phase): step to the working
    set's minimiser with a ratio test, drop the row with the most negative multiplier at a minimiser.  Returns the working set."""
    nrows = A.shape[0]
    W = list(range(neq))
    for _ in range(maxit):
        xw, lw = E._kkt_solve(H, c, A[W], b[W])
        p = xw - x
        if np.abs(p).max() <= 1e-14 * max(1.0, np.abs(x).max()):
            x = xw
            neg = [(lw[k], k) for k, i in enumerate(W) if i >= neq and lw[k] < 0.0]
            if not neg or min(neg)[0] >= -1e-13 * max(1.0, np.abs(lw).max()):
                return W
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
    raise E.CertificationError("active-set method from the LP's point did not converge in %d iterations" % maxit)


def certified_qp(Q, c, L, neq, x0=None, maxit=500):
    """x*, the multipliers lam [nrows], the working set and the certificate dict, as qp_exact.exact_qp; an LP-infeasible QP
    raises CertificationError.  Also returns how x* was found: "exact_qp" or "lp restart"."""
    H = E.sym_lower(Q)
    c = np.asarray(c, dtype=np.float64)
    L = np.asarray(L, dtype=np.float64).reshape(-1, N + 1)
    A, b = L[:, :N], L[:, N]
    try:
        W = E.exact_qp(Q, c, L, neq, x0=x0, maxit=maxit)[2]
        how = "exact_qp"
    except (E.CertificationError, np.linalg.LinAlgError):
        t, xf = lp_margin(L, neq)
        if t > 0.0:
            raise E.CertificationError("infeasible QP: the least row-scaled violation of any point is %.3e" % t)
        W = _from_feasible(H, c, A, b, neq, xf, maxit)
        how = "lp restart"
    x, lw = E._kkt_solve(H, c, A[W], b[W], refine=REFINE)
    lam = np.zeros(L.shape[0])
    lam[W] = lw
    return x, lam, sorted(W), E.certify(H, c, A, b, neq, x, lam), how
