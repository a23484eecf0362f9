"""One Levenberg-Marquardt feasibility step (twb_batch_lm_step_device) for ONE instance, written plainly in numpy:

    r  = violation of g against [g_lower, g_upper]
    Js = diag(s) J,  rs = s r,   s_i = 1 / max(1, max_k |J_ik|)
    (Js^T Js + mu I) dx = -Js^T rs          cg_iters conjugate-gradient iterations (alpha = 0 if p^T A p <= 0,
                                            beta = 0 if r^T r <= 0)
    x <- clip(x + dx min(1, cap / max|dx|), x_lower, x_upper)

in float64 or in np.longdouble.  It states the maths, not the kernel: the sparse products are numpy gathers and segment
sums over the CSR pattern and its transpose, in numpy's summation order.  g and the Jacobian values are inputs, so it
needs neither the evaluation nor the oracle.  A NaN in the inputs stays a NaN in the outputs, as on paper."""
import numpy as np

# np.longdouble is an extended type only on some platforms (x86-64: 64-bit mantissa, eps 1.08e-19); elsewhere it may be
# float64 itself, and a comparison against it would prove nothing
LONGDOUBLE_IS_WIDER = bool(np.finfo(np.longdouble).eps < np.finfo(np.float64).eps)


def _segments(ufunc, vals, ptr, empty):
    """ufunc over vals[ptr[i]:ptr[i + 1]] for every segment i; `empty` for an empty segment (np.ufunc.reduceat would return
    vals[ptr[i]] there).  Segments are contiguous and in order, so reduceat at the starts of the non-empty ones is exact."""
    starts, ends = ptr[:-1], ptr[1:]
    out = np.full(len(starts), empty, dtype=vals.dtype)
    full = ends > starts
    if full.any():
        out[full] = ufunc.reduceat(vals, starts[full])
    return out


class Pattern:
    """The CSR pattern (row_ptr, col_idx) of an m x n Jacobian and its transpose."""

    def __init__(self, row_ptr, col_idx, n):
        self.row_ptr = np.asarray(row_ptr, np.int64)
        self.col_idx = np.asarray(col_idx, np.int64)
        self.m, self.n = len(self.row_ptr) - 1, int(n)
        self.row_of = np.repeat(np.arange(self.m), np.diff(self.row_ptr))       # row of every CSR slot
        self.by_col = np.argsort(self.col_idx, kind="stable")                  # slots grouped by column
        self.row_t = self.row_of[self.by_col]                                   # their rows
        self.col_ptr = np.concatenate([[0], np.cumsum(np.bincount(self.col_idx, minlength=self.n))])

    def row_max_abs(self, vals):
        return _segments(np.maximum, np.abs(vals), self.row_ptr, 0)

    def matvec(self, vals, v):
        """J v"""
        return _segments(np.add, vals * v[self.col_idx], self.row_ptr, 0)

    def rmatvec(self, vals_t, u):
        """J^T u, with vals_t = vals[by_col] (the values in the transpose's order)"""
        return _segments(np.add, vals_t * u[self.row_t], self.col_ptr, 0)


def violation(g, g_lower, g_upper):
    return np.where(g < g_lower, g - g_lower, np.where(g > g_upper, g - g_upper, np.zeros_like(g)))


def lm_capped_step(pat, g, jac, g_lower, g_upper, mu, cap, cg_iters, dtype=np.float64):
    """(dx, violation): the capped step dx min(1, cap / max|dx|) before the projection, and max_i |s_i r_i|, in `dtype`."""
    g, jac, g_lower, g_upper = (np.asarray(a, np.float64).astype(dtype) for a in (g, jac, g_lower, g_upper))
    mu, cap = dtype(mu), dtype(cap)
    s = 1 / np.maximum(pat.row_max_abs(jac), dtype(1))
    js = jac * s[pat.row_of]
    js_t = js[pat.by_col]
    rs = s * violation(g, g_lower, g_upper)
    b = -pat.rmatvec(js_t, rs)
    dx = np.zeros(pat.n, dtype)
    res, p = b.copy(), b.copy()
    rr = np.sum(res * res)
    for _ in range(cg_iters):
        ap = pat.rmatvec(js_t, pat.matvec(js, p)) + mu * p
        pap = np.sum(p * ap)
        alpha = rr / pap if pap > 0 else dtype(0)
        dx = dx + alpha * p
        res = res - alpha * ap
        rr_new = np.sum(res * res)
        p = res + (rr_new / rr if rr > 0 else dtype(0)) * p
        rr = rr_new
    big = np.max(np.abs(dx)) if pat.n else dtype(0)
    if big > cap:
        dx = dx * (cap / big)
    return dx, (np.max(np.abs(rs)) if pat.m else dtype(0))


def lm_step(x, g, jac, x_lower, x_upper, g_lower, g_upper, row_ptr, col_idx, mu, cap, cg_iters, dtype=np.float64, pat=None):
    """(x_new, violation) of one step for one instance, in `dtype` (np.float64 or np.longdouble).  `pat`: an optional
    Pattern of (row_ptr, col_idx), to build the transpose once for many instances."""
    x = np.asarray(x, np.float64)
    pat = Pattern(row_ptr, col_idx, len(x)) if pat is None else pat
    dx, viol = lm_capped_step(pat, g, jac, g_lower, g_upper, mu, cap, cg_iters, dtype)
    lo, up = (np.asarray(a, np.float64).astype(dtype) for a in (x_lower, x_upper))
    return np.minimum(np.maximum(x.astype(dtype) + dx, lo), up), viol


def relabelled_float64_steps(x, g, jac, x_lower, x_upper, g_lower, g_upper, row_ptr, col_idx, mu, cap, cg_iters, count, seed):
    """x_new of the float64 step on `count` relabellings of the same instance, mapped back to the original numbering: the
    identity, then random permutations of the rows, of the columns and of the entries inside each row.  The step does not
    depend on the numbering, its rounding does: the spread of these results is what float64 arithmetic alone leaves open.
    (On this project's problems the error of a 25-iteration step moves by up to two orders of magnitude with the order.)"""
    row_ptr, col_idx = np.asarray(row_ptr, np.int64), np.asarray(col_idx, np.int64)
    x, g, jac, x_lower, x_upper, g_lower, g_upper = (np.asarray(a, np.float64) for a in (x, g, jac, x_lower, x_upper, g_lower, g_upper))
    m, n = len(row_ptr) - 1, len(x)
    rng = np.random.default_rng(seed)
    out = []
    for k in range(count):
        rows, cols = (np.arange(m), np.arange(n)) if k == 0 else (rng.permutation(m), rng.permutation(n))
        slots = np.concatenate([np.arange(row_ptr[i], row_ptr[i + 1]) if k == 0 else rng.permutation(np.arange(row_ptr[i], row_ptr[i + 1]))
                                for i in rows] + [np.zeros(0, np.int64)])
        new_col = np.empty(n, np.int64)
        new_col[cols] = np.arange(n)
        rp = np.concatenate([[0], np.cumsum(np.diff(row_ptr)[rows])])
        xn, _ = lm_step(x[cols], g[rows], jac[slots], x_lower[cols], x_upper[cols], g_lower[rows], g_upper[rows], rp,
                        new_col[col_idx[slots]], mu, cap, cg_iters, np.float64)
        out.append(xn[new_col])
    return out
