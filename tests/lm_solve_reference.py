"""What a solve iteration adds to the Levenberg-Marquardt step of lm_reference, for ONE instance, written plainly in numpy:

    merit      phi0 = 1/2 ||s r(g)||^2                         s: the row scales at x
    predicted  phi0 - 1/2 ||s r(g + J d)||^2,  d = x_trial - x  (the step after the cap and the projection)
    phi_t      1/2 ||s r(g_trial)||^2                          the same s
    rho        (phi0 - phi_t) / predicted
    accept     predicted > 0, g_trial and phi_t finite, rho > eta:  mu <- max(mu_min, mu max(1/3, 1 - (2 rho - 1)^3)), nu <- 2
    reject     otherwise:                                        mu <- mu nu, nu <- 2 nu, stalled if mu > mu_max

The mu / nu update is written in the kernel's order of operations (t * t * t, not a power), so that on the same decision
it gives the same bits."""
import numpy as np

import lm_reference as ref

RUNNING, CONVERGED, STALLED, NONFINITE = 0, 1, 2, 3


def row_scales(pat, jac, dtype=np.float64):
    return 1 / np.maximum(pat.row_max_abs(np.asarray(jac, np.float64).astype(dtype)), dtype(1))


def half_norm2(s, g, g_lower, g_upper):
    """1/2 ||s r(g)||^2"""
    v = s * ref.violation(g, g_lower, g_upper)
    return np.sum(v * v) / 2


def merit_and_predicted(pat, x, x_trial, g, jac, g_lower, g_upper, dtype=np.float64):
    """(merit, predicted) in `dtype` for the step from x to x_trial."""
    x, x_trial, g, jac, g_lower, g_upper = (np.asarray(a, np.float64).astype(dtype) for a in (x, x_trial, g, jac, g_lower, g_upper))
    s = row_scales(pat, jac, dtype)
    phi0 = half_norm2(s, g, g_lower, g_upper)
    return phi0, phi0 - half_norm2(s, g + pat.matvec(jac, x_trial - x), g_lower, g_upper)


def accept(merit, predicted, phi_t, g_trial_finite, mu, nu, eta, mu_min, mu_max):
    """(accepted, rho, mu, nu, stalled) in float64."""
    f = np.float64
    merit, predicted, phi_t, mu, nu = f(merit), f(predicted), f(phi_t), f(mu), f(nu)
    with np.errstate(all="ignore"):
        rho = (merit - phi_t) / predicted
        ok = bool(predicted > 0 and g_trial_finite and np.isfinite(phi_t) and rho > eta)
        if ok:
            t = f(2.0) * rho - f(1.0)
            return True, rho, np.maximum(f(mu_min), mu * np.maximum(f(1.0) / f(3.0), f(1.0) - t * t * t)), f(2.0), False
        mu_new = mu * nu
        return False, rho, mu_new, f(2.0) * nu, bool(mu_new > mu_max)
