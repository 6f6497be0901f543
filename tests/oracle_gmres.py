"""amgb_solve_gmres in numpy: restarted GMRES(m) on A x = b, right-preconditioned by prec(v) (one V-cycle from
a zero guess: oracle_sa.precondition composed with any of the three oracle Multigrids), Arnoldi by classical
Gram-Schmidt with one reorthogonalisation, Givens rotations and back substitution on the host.  The device
solver follows the same steps; its dot products are summed in another order, so its step counts agree to
about one step, not its bits (include/amgb.h)."""
import numpy as np


def gmres(A, b, prec, rel_tol, restart=30, max_iters=1000, x0=None):
    """Returns (steps, true ||b - A x|| / ||b||, x, history of the |g_{j+1}| / ||b|| estimates)."""
    A = A.to_scipy() if hasattr(A, "to_scipy") else A
    b = np.ascontiguousarray(b, np.float64)
    x = np.zeros_like(b) if x0 is None else np.array(x0, np.float64)
    m = restart
    bnorm = np.linalg.norm(b)
    it, hist = 0, []
    if bnorm == 0.0:
        return 0, 0.0, x, hist
    r = b - A @ x
    beta = np.linalg.norm(r)
    rel = beta / bnorm
    failed = False
    while not failed and it < max_iters and rel > rel_tol:
        V = np.zeros((m + 1, b.size))
        H = np.zeros((m + 1, m))
        cs, sn, g = np.zeros(m), np.zeros(m), np.zeros(m + 1)
        V[0] = r / beta
        g[0] = beta
        k = 0
        for j in range(m):
            if it >= max_iters:
                break
            w = A @ prec(V[j])
            h = V[: j + 1] @ w
            w = w - h @ V[: j + 1]
            h2 = V[: j + 1] @ w
            w = w - h2 @ V[: j + 1]
            H[: j + 1, j] = h + h2
            hnext = np.linalg.norm(w)
            H[j + 1, j] = hnext
            if not (np.all(np.isfinite(H[: j + 1, j])) and np.isfinite(hnext)):
                failed = True  # abandon the cycle: x stays that of the last completed one
                break
            if hnext != 0.0:
                V[j + 1] = w / hnext
            for i in range(j):
                t = cs[i] * H[i, j] + sn[i] * H[i + 1, j]
                H[i + 1, j] = -sn[i] * H[i, j] + cs[i] * H[i + 1, j]
                H[i, j] = t
            d = np.hypot(H[j, j], hnext)
            if d == 0.0:  # A M v_j = 0
                failed = True
                break
            cs[j], sn[j] = H[j, j] / d, hnext / d
            H[j, j], H[j + 1, j] = d, 0.0
            g[j + 1] = -sn[j] * g[j]
            g[j] = cs[j] * g[j]
            k = j + 1
            it += 1
            est = abs(g[j + 1]) / bnorm
            hist.append(est)
            if est <= rel_tol or hnext == 0.0:
                break
        if failed or k == 0:
            break
        y = np.zeros(k)
        for i in range(k - 1, -1, -1):
            y[i] = (g[i] - H[i, i + 1:k] @ y[i + 1:]) / H[i, i]
        x = x + prec(y @ V[:k])
        r = b - A @ x
        beta = np.linalg.norm(r)
        rel = beta / bnorm
    return it, rel, x, hist
