"""ORACLE — TEST INFRASTRUCTURE ONLY.

scipy's `trf_no_bounds` (scipy/optimize/_lsq/trf.py, the solver behind calibration.py:209-210) restated with ONE change: the
regularised Gauss-Newton direction is solved exactly (dense normal equations) instead of by LSMR.  The loop is scipy's, and so are
`minimize_quadratic_1d`, `update_tr_radius` and `check_termination`, imported, not re-typed.  The step itself (`trf_step`) is a
high-precision statement of the same operation: the regularised system is solved in float64 with iterative refinement (residual in
long double), and the 2-D trust-region subproblem by a bracketed root of its secular equation instead of scipy's quartic.

The model runs from normal equations: `lin(x) -> (J^T J, J^T f, cost)`.  Tests drive it either with the oracle residual and a 3-point
finite-difference Jacobian (`fun`, `jac`) or with the device's own normal equations (`lin`), and compare the GPU solver's
per-iteration table, or one step, with it."""
import numpy as np
from numpy.linalg import norm
from scipy.optimize import brentq
from scipy.optimize._lsq.common import check_termination, minimize_quadratic_1d, update_tr_radius


def solve_refined(M, b, sweeps=2):
  """x with M x = b: LU in float64, then `sweeps` refinement steps whose residual b - M x is formed in long double."""
  Ml, bl = M.astype(np.longdouble), b.astype(np.longdouble)
  x = np.linalg.solve(M, b)
  for _ in range(sweeps):
    r = bl - Ml @ x.astype(np.longdouble)
    x = x + np.linalg.solve(M, r.astype(np.float64))
  return x


def solve_subproblem_2d(B, g, Delta):
  """argmin 0.5 p^T B p + g^T p over ||p|| <= Delta (B 2x2 symmetric) -> (p, on_boundary).

  Interior Newton point when B is positive definite and the point lies inside.  Otherwise the boundary minimiser
  p(s) = -(B + s I)^-1 g with s >= max(0, -l_min) the root of ||p(s)|| = Delta, found by brentq in the eigenbasis of B."""
  l, V = np.linalg.eigh(B)
  h = V.T @ g
  if l[0] > 0:
    p = -V @ (h / l)
    if norm(p) <= Delta: return p, False
  assert abs(h[0]) > 1e-12 * norm(h), "hard case of the 2-D subproblem: the model does not handle it"

  def secular(s):              # 1/||p(s)|| - 1/Delta: increasing in s, close to linear (the form Newton's method is usually run on)
    a = l[0] + s
    return (0.0 if a == 0 else 1.0 / np.hypot(h[0] / a, h[1] / (l[1] + s))) - 1.0 / Delta

  lo = max(0.0, -l[0])         # secular(lo) <= 0: the Newton point is outside, or B is singular / indefinite
  hi = max(lo, norm(h) / Delta - l[0])
  while secular(hi) < 0: hi = 2 * hi + 1e-300
  s = brentq(secular, lo, hi, xtol=1e-300, rtol=4 * np.finfo(float).eps, maxiter=500)
  p = -V @ (h / (l + s))
  return p * (Delta / norm(p)), True


def trf_step(JtJ, g, x, Delta, scale_inv, reg_Delta=None, reg_floor=1e-12):
  """One trial step of trf_no_bounds with x_scale='jac' and an exact inner solve, from the normal equations at x.

  scipy computes the damping `reg` once per outer iteration and keeps the subspace across rejected trials, shrinking only Delta:
  `reg_Delta` is the radius the iteration started with (default: Delta).  Returns a dict with
    step, step_h      the step in x and in the scaled variables (step = step_h / scale_inv)
    reg, predicted    the damping term and the predicted reduction of the quadratic model
    boundary          whether the 2-D step lies on the trust-region boundary
    cond              condition number of A + reg I (A = D J^T J D) over the live columns (diag(J^T J) > 0)
    gn_h, B_S, g_S    the regularised Gauss-Newton direction and the 2-D problem, p_S its solution (for checks against scipy)"""
  d = 1.0 / scale_inv
  g_h = d * g
  A = d[:, None] * JtJ * d[None, :]
  a, b = g_h @ A @ g_h, -(g_h @ g_h)
  Dr = Delta if reg_Delta is None else reg_Delta
  ag_value = minimize_quadratic_1d(a, b, 0, Dr / norm(g_h))[1]
  reg = max(-ag_value / Dr ** 2, reg_floor)
  M = A + reg * np.eye(A.shape[0])
  gn_h = solve_refined(M, g_h)
  Sb, _ = np.linalg.qr(np.vstack((g_h, gn_h)).T)
  B_S, g_S = Sb.T @ A @ Sb, Sb.T @ g_h
  p_S, boundary = solve_subproblem_2d(B_S, g_S, Delta)
  step_h = Sb @ p_S
  predicted = -(0.5 * p_S @ B_S @ p_S + g_S @ p_S)
  live = np.diag(JtJ) > 0
  ev = np.linalg.eigvalsh(M[np.ix_(live, live)]) if live.any() else np.ones(1)
  return dict(step=d * step_h, step_h=step_h, reg=reg, predicted=predicted, boundary=boundary, cond=ev[-1] / ev[0],
              gn_h=gn_h, B_S=B_S, g_S=g_S, p_S=p_S)


def jac_scale(JtJ, scale_inv_old=None):
  """x_scale='jac': column norms of J (sqrt of diag(J^T J)), zero columns scaled by 1; later iterations keep the running maximum."""
  s = np.sqrt(np.diag(JtJ)).copy()
  if scale_inv_old is None:
    s[s == 0] = 1
    return s
  return np.maximum(scale_inv_old, s)


def trf_exact(fun, jac, x0, ftol=1e-8, xtol=1e-8, gtol=1e-8, max_nfev=100, reg_floor=1e-12, lin=None, trace=None):
  """The trf loop.  `fun(x)` gives the residual (its cost judges a trial step); the normal equations come from `lin(x)`, by default
  J^T J, J^T f of `jac`.  `trace`, if a list, receives per trial step the state its control decisions were taken on."""
  if lin is None:
    def lin(x):
      J, f = jac(x), fun(x)
      return J.T @ J, J.T @ f, 0.5 * f @ f
  x = np.array(x0, float)
  f = fun(x); nfev = 1
  cost = 0.5 * f @ f
  JtJ, g, _ = lin(x); njev = 1
  scale_inv = jac_scale(JtJ)
  Delta = norm(x * scale_inv) or 1.0
  rows, it, status, step_norm, reduction = [], 0, None, None, None
  while True:
    g_norm = norm(g, np.inf)
    if g_norm < gtol: status = 1
    rows.append((it, nfev, cost, reduction, step_norm, g_norm))
    if status is not None or nfev >= max_nfev: break
    Delta_it = Delta
    reduction = -1
    while reduction <= 0 and nfev < max_nfev:
      st = trf_step(JtJ, g, x, Delta, scale_inv, reg_Delta=Delta_it, reg_floor=reg_floor)
      step, predicted = st["step"], st["predicted"]
      f_new = fun(x + step); nfev += 1
      cost_new = 0.5 * f_new @ f_new
      reduction = cost - cost_new
      shn = norm(st["step_h"])
      Delta_new, ratio = update_tr_radius(Delta, reduction, predicted, shn, shn > 0.95 * Delta)
      step_norm = norm(step)
      if trace is not None:
        trace.append(dict(st, x=x, Delta=Delta, cost=cost, cost_new=cost_new, reduction=reduction, ratio=ratio, step_norm=step_norm,
                          x_norm=norm(x), step_h_norm=shn))
      status = check_termination(reduction, cost, step_norm, norm(x), ratio, ftol, xtol)
      if status is not None: break
      Delta = Delta_new
    if reduction > 0:
      x = x + step; f = f_new; cost = cost_new
      JtJ, g, _ = lin(x); njev += 1
      scale_inv = jac_scale(JtJ, scale_inv)
    else:
      step_norm, reduction = 0, 0
    it += 1
  return x, cost, nfev, njev, (status or 0), rows
