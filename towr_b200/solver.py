"""Device-resident multi-start solver loop on top of the batched evaluation (BASELINE configs[0] / [4] name IPOPT solves;
neither IPOPT nor ifopt exists in this image, see DESIGN.md).

The stand-in is a deterministic Levenberg-Marquardt FEASIBILITY iteration on the NLP's constraints — what IPOPT's
restoration phase minimises — for every instance of a batch in lock step:

    r  = violation of g(x) against [g_lower, g_upper]              (twb_batch_eval_device: g and the CSR Jacobian values;
                                                                    the problem's bounds or one row per instance)
    Js = diag(s) J,  rs = s r,   s_i = 1 / max(1, max_k |J_ik|)    (row scaling)
    (Js^T Js + mu I) dx = -Js^T rs                                 (`cg_iters` conjugate-gradient iterations, matrix-free)
    x <- clip(x + dx * min(1, cap / max|dx|), x_lower, x_upper)

The iterates, g, the Jacobian values and all solver vectors stay on the GPU.  An iteration is two library calls:
`twb_batch_eval_device` (g and the CSR Jacobian values of all instances) and `twb_batch_lm_step_device`, or
`twb_batch_lm_step_bounds_device` with per-instance constraint bounds (towr_b200/csrc/lm_kernel.cu: CTA = instance, the
conjugate gradients run in shared memory on the problem's ONE shared CSR pattern and its transpose, fixed summation
orders, no atomics).  An instance whose x, g or Jacobian values hold a
non-finite entry (the evaluation flags it in `status` bit 0) is not stepped by the native step: its x stays exactly as it
was and its violation is NaN, so the caller can tell it apart instead of finding it clipped to its bounds.
`solve(X, max_iters, tol)` solves to a tolerance instead: per iteration `twb_batch_eval_device`, the trial step
`twb_batch_lm_trial_device` (the same step with a damping mu per instance, written to x_trial; merit 1/2 ||s r||^2, the
decrease the linear model predicts, status CONVERGED when max |s r| <= tol or NONFINITE), a g-only evaluation at x_trial and
`twb_batch_lm_accept_device` (gain ratio rho > eta: x <- x_trial and mu lowered, else x kept and mu raised, STALLED past
mu_max).  The host picks the budget and stops early once no instance is RUNNING; tests/test_lm_solve.py holds the
acceptance rule in numpy (tests/lm_solve_reference.py) and compares decisions on identical inputs.
`native=False` keeps the first implementation of the same step in PyTorch tensor algebra (padded ELL gathers) — 30 x
slower, used by the tests as a second opinion.
tests/test_solver_loop.py holds the same algorithm in numpy, driven one instance at a time like ifopt by the CPU
restatement of the reference; all three must walk the same iterates.
"""
import numpy as np


def ell_maps(row_ptr, col_idx, n):
    """Padded index maps of a CSR pattern: (rows, cols_of, rowsT, rows_of) with
    rows[i, k]   = slot of the k-th entry of row i            (pad: nnz)
    cols_of[i,k] = its column                                  (pad: 0)
    rowsT[j, k]  = slot of the k-th entry of column j          (pad: nnz)
    rows_of[j,k] = its row                                     (pad: 0)
    Slots index the CSR value array extended by one zero."""
    row_ptr = np.asarray(row_ptr, np.int64); col_idx = np.asarray(col_idx, np.int64)
    m, nnz = len(row_ptr) - 1, len(col_idx)
    lens = np.diff(row_ptr)
    W = int(lens.max()) if m else 0
    rows = np.full((m, W), nnz, np.int64); cols_of = np.zeros((m, W), np.int64)
    for i in range(m):
        k = np.arange(row_ptr[i], row_ptr[i + 1])
        rows[i, :len(k)] = k; cols_of[i, :len(k)] = col_idx[k]
    row_of_slot = np.repeat(np.arange(m), lens)
    order = np.argsort(col_idx, kind="stable")                 # slots grouped by column, ascending row inside a column
    counts = np.bincount(col_idx, minlength=n)
    Wc = int(counts.max()) if nnz else 0
    rowsT = np.full((n, Wc), nnz, np.int64); rows_of = np.zeros((n, Wc), np.int64)
    start = np.concatenate([[0], np.cumsum(counts)])
    for j in range(n):
        k = order[start[j]:start[j + 1]]
        rowsT[j, :len(k)] = k; rows_of[j, :len(k)] = row_of_slot[k]
    return rows, cols_of, rowsT, rows_of


class BatchedLevenbergMarquardt:
    """All instances of a `Batch` in lock step, everything on the batch's GPU."""

    def __init__(self, batch, x_lower=None, x_upper=None, g_lower=None, g_upper=None, mu=1e-2, cap=0.1, cg_iters=25, native=True):
        """x_lower / x_upper: variable bounds, (n,) or per instance (B, n); g_lower / g_upper: constraint bounds, (m,) or per
        instance (B, m) (e.g. the last two results of Batch.state_instances_device(..., want_g_bounds=True)); None: the
        problem's own."""
        import torch
        self.torch = torch
        self.native = native
        self.batch, p = batch, batch.problem
        self.p, self.B = p, batch.B
        self.dev = torch.device("cuda", batch.device)
        xl, xu, gl, gu = p.bounds()
        to = lambda a: a.to(self.dev, torch.float64) if torch.is_tensor(a) else torch.as_tensor(np.asarray(a, np.float64), device=self.dev)
        self.xl = to(xl if x_lower is None else x_lower); self.xu = to(xu if x_upper is None else x_upper)
        if (g_lower is None) != (g_upper is None):
            raise ValueError("g_lower and g_upper: both or neither")
        self.gl, self.gu = to(gl if g_lower is None else g_lower), to(gu if g_upper is None else g_upper)
        # per-instance constraint bounds go to the native step as (B, m) rows; without them it uses the problem's own
        self.gl_full = None if g_lower is None else self.gl.expand(self.B, p.m).contiguous()
        self.gu_full = None if g_upper is None else self.gu.expand(self.B, p.m).contiguous()
        rows, cols_of, rowsT, rows_of = ell_maps(p.row_ptr(), p.structure()[1], p.n)
        ti = lambda a: torch.as_tensor(a, device=self.dev)
        self.rows, self.cols_of, self.rowsT, self.rows_of = ti(rows), ti(cols_of), ti(rowsT), ti(rows_of)
        self.mu, self.cap, self.cg_iters = mu, cap, cg_iters
        B = self.B
        self.g = torch.empty((B, p.m), dtype=torch.float64, device=self.dev)
        self.jac = None if native else torch.empty((B, p.nnz + 1), dtype=torch.float64, device=self.dev)   # one extra zero: the pad slot
        self.jac_vals = torch.empty((B, p.nnz), dtype=torch.float64, device=self.dev)
        self.status = torch.zeros(B, dtype=torch.int32, device=self.dev)
        self.viol = torch.zeros(B, dtype=torch.float64, device=self.dev)
        self.xl_full = self.xl.expand(B, p.n).contiguous(); self.xu_full = self.xu.expand(B, p.n).contiguous()

    def _violation(self, g):
        t = self.torch
        return t.where(g < self.gl, g - self.gl, t.where(g > self.gu, g - self.gu, t.zeros_like(g)))

    def step(self, X):
        """One iteration for all instances.  X: (B, n) CUDA float64, updated in place.  Returns the largest scaled
        violation per instance BEFORE the step, (B,)."""
        t = self.torch
        from . import capi
        self.batch.eval_device(X, g=self.g, jac=self.jac_vals, status=self.status, flags=capi.EVAL_G | capi.EVAL_JAC)
        if self.native:
            self.batch.lm_step_device(X, self.g, self.jac_vals, self.xl_full, self.xu_full, self.mu, self.cap, self.cg_iters, self.viol,
                                      g_lower=self.gl_full, g_upper=self.gu_full)
            return self.viol.clone()
        self.jac[:, :-1] = self.jac_vals; self.jac[:, -1] = 0.0
        A = self.jac[:, self.rows]                                   # (B, m, W) rows of J
        s = 1.0 / t.clamp(A.abs().amax(dim=2), min=1.0)              # (B, m)
        A = A * s[:, :, None]
        AT = self.jac[:, self.rowsT] * s[:, self.rows_of]            # (B, n, Wc) columns of Js
        rs = s * self._violation(self.g)
        Jv = lambda v: (A * v[:, self.cols_of]).sum(dim=2)           # Js v
        JTu = lambda u: (AT * u[:, self.rows_of]).sum(dim=2)         # Js^T u
        b = -JTu(rs)
        dx = t.zeros_like(b); res = b.clone(); pdir = b.clone()
        rr = (res * res).sum(dim=1)
        for _ in range(self.cg_iters):
            Ap = JTu(Jv(pdir)) + self.mu * pdir
            pAp = (pdir * Ap).sum(dim=1)
            alpha = t.where(pAp > 0, rr / pAp, t.zeros_like(rr))
            dx += alpha[:, None] * pdir
            res -= alpha[:, None] * Ap
            rr_new = (res * res).sum(dim=1)
            beta = t.where(rr > 0, rr_new / rr, t.zeros_like(rr))
            pdir = res + beta[:, None] * pdir
            rr = rr_new
        big = dx.abs().amax(dim=1)
        dx *= t.where(big > self.cap, self.cap / big, t.ones_like(big))[:, None]
        X.copy_(t.minimum(t.maximum(X + dx, self.xl), self.xu))
        return rs.abs().amax(dim=1)

    def run(self, X, iters):
        """`iters` iterations; returns the violation history (iters, B) as a CUDA tensor."""
        hist = self.torch.empty((iters, self.B), dtype=self.torch.float64, device=self.dev)
        for it in range(iters):
            hist[it] = self.step(X)
        return hist

    def solve_state(self):
        """A fresh per-instance solve state for `iterate`: mu = the constructor's mu, nu = 2, status RUNNING, 0 iterations,
        and the trial buffers."""
        if not self.native:
            raise ValueError("solve / iterate run on the native path only")
        if not self.mu > 0:
            raise ValueError("solve needs an initial mu > 0")
        return SolveState(self)

    def iterate(self, X, st, tol, eta=1e-4, mu_min=1e-12, mu_max=1e10, cg_iters=None):
        """One solve iteration for every instance in lock step, four calls that only enqueue (graph-capturable after the
        first): evaluate g and J at X, the trial step (sets CONVERGED / NONFINITE), evaluate g at the trial point, accept or
        reject.  X (B, n) and the solve state `st` are updated in place."""
        from . import capi
        bt, f = self.batch, capi.EVAL_G | capi.EVAL_JAC
        bt.eval_device(X, g=self.g, jac=self.jac_vals, status=self.status, flags=f)
        bt.lm_trial_device(X, self.g, self.jac_vals, st.mu, st.status, st.x_trial, st.row_scale, st.merit, st.predicted,
                           self.xl_full, self.xu_full, self.gl_full, self.gu_full, self.cap,
                           self.cg_iters if cg_iters is None else cg_iters, tol, st.violation)
        if cg_iters == 0:
            return
        bt.eval_device(st.x_trial, g=st.g_trial, flags=capi.EVAL_G)
        bt.lm_accept_device(X, st.x_trial, st.g_trial, st.row_scale, st.merit, st.predicted, st.mu, st.nu, st.status, st.iterations,
                            self.gl_full, self.gu_full, eta, mu_min, mu_max)

    def solve(self, X, max_iters, tol, eta=1e-4, mu_min=1e-12, mu_max=1e10, check_every=4):
        """Solve every instance to max |s r| <= tol, at most `max_iters` iterations (native path only).  X (B, n) is updated
        in place.  The loop stops early once no instance is RUNNING (one host read of a flag every `check_every`
        iterations); afterwards one more evaluation and a trial without conjugate gradients make the status and the
        violation describe the returned X.  Returns (status, iterations, violation, mu), (B,) CUDA tensors: status LM_*
        (an instance still RUNNING has used up max_iters), iterations the trials taken, violation max |s r| at X."""
        import torch
        from . import capi
        st = self.solve_state()
        for it in range(max_iters):
            self.iterate(X, st, tol, eta, mu_min, mu_max)
            if (it + 1) % check_every == 0 and not bool(torch.any(st.status == capi.LM_RUNNING)):
                break
        self.iterate(X, st, tol, cg_iters=0)
        return st.status, st.iterations, st.violation, st.mu


class SolveState:
    """Per-instance state of BatchedLevenbergMarquardt.solve: damping mu and its growth factor nu, the solve status and the
    trials taken, plus the buffers of the trial point (x_trial, g_trial, row_scale, merit, predicted, violation)."""

    def __init__(self, lm):
        import torch
        from . import capi
        B, p, dev, f64 = lm.B, lm.p, lm.dev, torch.float64
        self.mu = torch.full((B,), float(lm.mu), dtype=f64, device=dev)
        self.nu = torch.full((B,), 2.0, dtype=f64, device=dev)
        self.status = torch.full((B,), capi.LM_RUNNING, dtype=torch.int32, device=dev)
        self.iterations = torch.zeros(B, dtype=torch.int32, device=dev)
        self.x_trial = torch.empty((B, p.n), dtype=f64, device=dev)
        self.g_trial = torch.empty((B, p.m), dtype=f64, device=dev)
        self.row_scale = torch.empty((B, p.m), dtype=f64, device=dev)
        self.merit = torch.empty(B, dtype=f64, device=dev)
        self.predicted = torch.empty(B, dtype=f64, device=dev)
        self.violation = torch.full((B,), float("nan"), dtype=f64, device=dev)
