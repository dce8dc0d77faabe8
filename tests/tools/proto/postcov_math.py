"""Numpy restatement of the posterior-covariance sweep K8 (csrc/postcov.cuh) on the reference's variables
(src/celerite_solver.jl): the full posterior covariance  C(x, x′) = k(x, x′) − k(x, t)ᵀ K̃⁻¹ k(t, x′)  of the latent f at
ascending τ, in O((N + M)·R² + M·(N + M)·R) without a matrix inverse.  Notation of postvar_math.py (K6).

Write C(x, x′) = k(x, x′) − α(x)ᵀ α(x′), α(x) = D^{−1/2} L⁻¹ k(t, x), and take x ≤ x′ (n₀ = n₀(x) ≤ n₀′ = n₀(x′)).

  n < n₀:  α_n(x) = √D_n W_nᵀ Φ(t_n → x) U(x) (the factor row of x inserted as a noise-free point), so the data before x give
           p(x)ᵀ Φ(x → x′) U(x′) with p(x) = S_x U(x), the filter state of K6 pass 1.  With k(x, x′) = V(x)ᵀ Φ(x → x′) U(x′)
           the prior term merges in:  k(x, x′) − Σ_{n<n₀} α_n α_n = −r(x)ᵀ v(x),  r(x) = p(x) − V(x),  v(x) = Φ(x → x′) U(x′).
  n ≥ n₀:  α_n(x) = −U_nᵀ A(n₀ → n) g_x / √D_n (K6's seed g_x = e_{x→t_{n₀}} ∘ r(x)), so the rest is g_xᵀ h_{n₀}(x′) with
               h_{n₀′}(x′) = Ξ_{n₀′} g_{x′},   h_n = A_nᵀ (φ_{n+1} ∘ h_{n+1}) − U_n (W_nᵀ v_n),   A_n = I − W_n U_nᵀ.
           Since g_x = e_{x→t_{n₀}} ∘ r(x), g_xᵀ h_{n₀} = r(x)ᵀ h̃(x) with h̃(x) = Φ(x → t_{n₀}) h_{n₀}: h carried down to x.

So one R-vector per column, w = v + h̃, walked backward from x′ over the merged grid G (the data times and τ, a τ point first
at a tie, so that a data point at τ counts as after it, as n₀ = #{t_n < τ} says):

    start at x′:     w = U(x′) + e_{x′→t_{n₀′}} ∘ (Ξ_{n₀′} g_{x′})         (U(x′) alone when n₀′ = N)
    each G step:     w ← φ^G_k ∘ w                                        (decay t^G_{k−1} → t^G_k, ≤ 1)
    data point n:    w ← w − U_n (W_nᵀ w)                                  (v and h̃ share the step: v_n + A_nᵀ h̃ − U_n W_nᵀ v_n)
    τ point x ≤ x′:  C(x, x′) = −r(x)ᵀ w

and the diagonal is −r(x)ᵀ U(x) − g_xᵀ Ξ_{n₀} g_x = D_x − g_xᵀ Ξ g_x, K6's variance.  K6 provides r(x) and the start vector
w₀(x) per τ point (its pass 1 has p and V, its pass 2 Ξ_{n₀}); the walk needs neither D nor V."""
import numpy as np
from scipy.linalg import cho_factor, cho_solve

from postvar_math import decay, factor, kernel, term_rows, uv


def merged_grid_tau_first(t, tau):
    """Merged order of t and τ, a τ point first at a tie: times [N + M] and codes (n ≥ 0: data point n, −m − 1: τ point m)."""
    t, tau = np.asarray(t, dtype=np.float64), np.asarray(tau, dtype=np.float64)
    code = np.concatenate([np.arange(len(t)), -np.arange(len(tau)) - 1])
    key = np.concatenate([np.ones(len(t)), np.zeros(len(tau))])
    order = np.lexsort((key, np.concatenate([t, tau])))   # stable: the τ points keep their order
    return np.concatenate([t, tau])[order], code[order]


def point_vectors(a, b, c, d, t, s2, tau):
    """What K6 adds per τ point for K8: r(x) = p(x) − V(x) and the start vector w₀(x), both [M × R]."""
    a, b, c, d, t, s2, tau = (np.asarray(x, dtype=np.float64) for x in (a, b, c, d, t, s2, tau))
    rows = term_rows(b, d)
    R = len(rows[0])
    N, M = len(t), len(tau)
    W, D = factor(a, b, c, d, t, s2)
    n0 = np.searchsorted(t, tau, side="left")
    r, w0, g = np.zeros((M, R)), np.zeros((M, R)), np.zeros((M, R))
    Q = np.zeros((R, R))   # K6 pass 1: the state just after absorbing point n − 1
    m = 0
    for n in range(N + 1):
        while m < M and n0[m] == n:
            U, V = uv(a, b, d, rows, tau[m])
            e = decay(c, rows, tau[m] - t[n - 1]) if n > 0 else np.zeros(R)
            r[m] = e * (Q @ (e * U)) - V
            w0[m] = U
            if n < N:
                g[m] = decay(c, rows, t[n] - tau[m]) * r[m]
            m += 1
        if n < N:
            ph = decay(c, rows, t[n] - t[n - 1]) if n > 0 else np.zeros(R)
            Q = np.outer(ph, ph) * Q + D[n] * np.outer(W[n], W[n])
    Xi = np.zeros((R, R))  # K6 pass 2
    m = M - 1
    while m >= 0 and n0[m] == N:
        m -= 1
    for n in range(N - 1, -1, -1):
        U, _ = uv(a, b, d, rows, t[n])
        ph = decay(c, rows, t[n + 1] - t[n]) if n + 1 < N else np.zeros(R)
        X = np.outer(ph, ph) * Xi
        p = X @ W[n]
        Xi = X - np.outer(U, p) - np.outer(p, U) + (W[n] @ p + 1.0 / D[n]) * np.outer(U, U)
        while m >= 0 and n0[m] == n:
            w0[m] += decay(c, rows, t[n] - tau[m]) * (Xi @ g[m])
            m -= 1
    return r, w0, W


def predict_cov(a, b, c, d, t, s2, tau):
    """Posterior covariance [M × M] of the latent f at ascending τ: the backward walk of every column at once."""
    a, b, c, d, t, s2, tau = (np.asarray(x, dtype=np.float64) for x in (a, b, c, d, t, s2, tau))
    rows = term_rows(b, d)
    R = len(rows[0])
    M = len(tau)
    r, w0, W = point_vectors(a, b, c, d, t, s2, tau)
    G, code = merged_grid_tau_first(t, tau)
    C = np.full((M, M), np.nan)
    w = np.zeros((M, R))   # row m′: the state of column m′ (zero until the walk reaches x′)
    for k in range(len(G) - 1, -1, -1):
        if k + 1 < len(G):
            w *= decay(c, rows, G[k + 1] - G[k])
        if code[k] >= 0:
            U, _ = uv(a, b, d, rows, G[k])
            w -= np.outer(w @ W[code[k]], U)
        else:
            m = -code[k] - 1
            w[m] = w0[m]
            C[m, m:] = -(w[m:] @ r[m])   # C(x_m, x_m′) for every column m′ ≥ m
    return np.where(np.isnan(C), C.T, C)   # the mirror: exactly symmetric


def dense_cov(a, b, c, d, t, s2, tau):
    """The same covariance with dense matrices and a Cholesky solve."""
    K = kernel(a, b, c, d, t[:, None] - t[None, :]) + np.diag(s2)
    k = kernel(a, b, c, d, tau[:, None] - t[None, :])
    return kernel(a, b, c, d, tau[:, None] - tau[None, :]) - k @ cho_solve(cho_factor(K, lower=True), k.T)


def _kernel_ld(a, b, c, d, lag):
    lag = np.abs(lag.astype(np.longdouble))
    out = np.zeros_like(lag)
    for aa, bb, cc, dd in zip(*(np.asarray(x).astype(np.longdouble) for x in (a, b, c, d))):
        out += np.exp(-cc * lag) * (aa * np.cos(dd * lag) + bb * np.sin(dd * lag))
    return out


def dense_cov_ld(a, b, c, d, t, s2, tau):
    """dense_cov in 80-bit arithmetic: Cholesky factor and forward substitution written out, C = K_ττ − ZᵀZ, Z = L⁻¹ K_tτ."""
    K = _kernel_ld(a, b, c, d, t[:, None] - t[None, :]) + np.diag(np.asarray(s2).astype(np.longdouble))
    L = np.zeros_like(K)
    for j in range(len(K)):
        v = K[j:, j] - L[j:, :j] @ L[j, :j]
        L[j, j] = np.sqrt(v[0])
        L[j + 1:, j] = v[1:] / L[j, j]
    Z = _kernel_ld(a, b, c, d, t[:, None] - tau[None, :])
    for i in range(len(t)):
        Z[i] = (Z[i] - L[i, :i] @ Z[:i]) / L[i, i]
    return _kernel_ld(a, b, c, d, tau[:, None] - tau[None, :]) - Z.T @ Z


def conditioned_error(got, a, b, c, d, t, s2, tau, tol):
    """(error of got against dense_cov / Σa, None) when within tol; otherwise the conditioning rule: the errors of got and of
    dense_cov against the 80-bit covariance (got must be at least as close to it as the FP64 dense route)."""
    want = dense_cov(a, b, c, d, t, s2, tau)
    err = float(np.max(np.abs(got - want))) / np.sum(a)
    if err <= tol:
        return err, None
    ld = dense_cov_ld(a, b, c, d, t, s2, tau)
    return err, tuple(float(np.max(np.abs(x - ld))) / np.sum(a) for x in (got, want))
