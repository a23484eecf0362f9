"""The trust-region step rule of twb_batch_lm_solve_device (TWB_LM_STEP_TRUST) for ONE instance, written plainly in numpy:

    gamma   = Js^T s r                                     the gradient of 1/2 ||s r||^2 in the row-scaled problem
    frozen  = x_lower == x_upper  or  (x <= x_lower and gamma > 0)  or  (x >= x_upper and gamma < 0)
    CG on the free set: (Js^T Js + mu I) dx = -gamma with res, p, dx and A p zero at every frozen variable
    x_trial = clip(x + dx min(1, radius / max|dx|), x_lower, x_upper),   step_norm = max |x_trial - x|
    after the gain-ratio decision (lm_solve_reference.accept):
      rho < 0.25 or rejected:                   radius <- 0.25 step_norm
      rho > 0.75 and step_norm >= 0.99 radius:  radius <- min(2 radius, radius_max)
      stalled once radius < 1e-12 max(1, max |x|)

It states the maths in numpy's summation order, like lm_reference, so g and the Jacobian values are inputs."""
import numpy as np

import lm_reference as ref

SHRINK, LOW, HIGH, GROW, EDGE, COLLAPSE = 0.25, 0.25, 0.75, 2.0, 0.99, 1e-12


def gradient(pat, g, jac, g_lower, g_upper):
    """gamma = Js^T s r in float64."""
    s = 1 / np.maximum(pat.row_max_abs(jac), 1.0)
    js = jac * s[pat.row_of]
    return pat.rmatvec(js[pat.by_col], s * ref.violation(g, g_lower, g_upper))


def frozen(x, x_lower, x_upper, gamma):
    return (x_lower == x_upper) | ((x <= x_lower) & (gamma > 0)) | ((x >= x_upper) & (gamma < 0))


def trust_step(pat, x, g, jac, x_lower, x_upper, g_lower, g_upper, mu, radius, cg_iters, dtype=np.float64):
    """(x_trial, frozen mask, step_norm) of one trial step in `dtype` (np.float64 or np.longdouble)."""
    x, g, jac, x_lower, x_upper, g_lower, g_upper = (np.asarray(a, np.float64).astype(dtype)
                                                     for a in (x, g, jac, x_lower, x_upper, g_lower, g_upper))
    mu, radius = dtype(mu), dtype(radius)
    s = 1 / np.maximum(pat.row_max_abs(jac), dtype(1))
    js = jac * s[pat.row_of]
    js_t = js[pat.by_col]
    gamma = pat.rmatvec(js_t, s * ref.violation(g, g_lower, g_upper))
    fz = frozen(x, x_lower, x_upper, gamma)
    free = ~fz
    b = np.where(free, -gamma, dtype(0))
    dx = np.zeros(pat.n, dtype)
    res, p = b.copy(), b.copy()
    rr = np.sum(res * res)
    for _ in range(cg_iters):
        ap = np.where(free, pat.rmatvec(js_t, pat.matvec(js, p)) + mu * p, dtype(0))
        pap = np.sum(p * ap)
        alpha = rr / pap if pap > 0 else dtype(0)
        dx = dx + alpha * p
        res = res - alpha * ap
        rr_new = np.sum(res * res)
        p = res + (rr_new / rr if rr > 0 else dtype(0)) * p
        rr = rr_new
    big = np.max(np.abs(dx)) if pat.n else dtype(0)
    if big > radius:
        dx = dx * (radius / big)
    xt = np.minimum(np.maximum(x + dx, x_lower), x_upper)
    return xt, fz, (np.max(np.abs(xt - x)) if pat.n else dtype(0))


def radius_update(radius, step_norm, accepted, rho, radius_max, x_max_abs):
    """(new radius, collapsed) after a trial with gain ratio rho."""
    if not accepted or rho < LOW:
        r = SHRINK * step_norm
    elif rho > HIGH and step_norm >= EDGE * radius:
        r = min(GROW * radius, radius_max)
    else:
        r = radius
    return r, bool(r < COLLAPSE * max(1.0, x_max_abs))


def relabelled_trust_steps(x, g, jac, x_lower, x_upper, g_lower, g_upper, row_ptr, col_idx, mu, radius, cg_iters, count, seed):
    """x_trial of the float64 trust step on `count` relabellings of the same instance (rows, columns and the entries inside
    each row permuted), mapped back to the original numbering: the spread float64 rounding alone leaves open, as
    lm_reference.relabelled_float64_steps does for the cap rule."""
    row_ptr, col_idx = np.asarray(row_ptr, np.int64), np.asarray(col_idx, np.int64)
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
        pat = ref.Pattern(rp, new_col[col_idx[slots]], n)
        xt, _, _ = trust_step(pat, x[cols], g[rows], jac[slots], x_lower[cols], x_upper[cols], g_lower[rows], g_upper[rows], mu, radius,
                              cg_iters)
        out.append(xt[new_col])
    return out
