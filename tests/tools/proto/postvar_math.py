"""Numpy restatement of the posterior-variance sweep K6 (csrc/postvar.cuh) on the reference's variables
(src/celerite_solver.jl): the diagonal of the posterior covariance  k(0) − k(τ, t)ᵀ K̃⁻¹ k(τ, t),  K̃ = K + diag(σ̃²),
in O((N + M)·R²) without a matrix inverse.

Rows (celerite_solver.jl:51-64, absolute times): a complex term gives U = (a cos dt + b sin dt, a sin dt − b cos dt),
V = (cos dt, sin dt); a real term (b = d = 0) one row U = a, V = 1.  φ_n = e^{−c (t_n − t_{n−1})} per row.

Forward factor (what the STEP_STORE sweep leaves behind):
    S_n = (φ_n φ_nᵀ) ∘ (S_{n−1} + D_{n−1} W_{n−1} W_{n−1}ᵀ),   D_n = Σa + σ̃²_n − U_nᵀ S_n U_n,   W_n = (V_n − S_n U_n) / D_n

Prediction point τ with n₀ = #{t_n < τ} (searchsortedfirst(t, τ) − 1), e_τ the row decay t_{n₀−1} → τ:
    S_τ = (e_τ e_τᵀ) ∘ (S_{n₀−1} + D_{n₀−1} W_{n₀−1} W_{n₀−1}ᵀ)           (0 when n₀ = 0)
    D_τ = Σa − U(τ)ᵀ S_τ U(τ)                                              filter variance from the data before τ
    g_τ = e_{τ→t_{n₀}} ∘ (S_τ U(τ) − V(τ))
    Ξ_{N−1} = U U ᵀ / D_{N−1};   Ξ_n = U_n U_nᵀ / D_n + A_nᵀ ((φ_{n+1} φ_{n+1}ᵀ) ∘ Ξ_{n+1}) A_n,   A_n = I − W_n U_nᵀ
    var(τ) = D_τ − g_τᵀ Ξ_{n₀} g_τ                                          (no Ξ term when n₀ = N)

The backward step is applied as a rank-2 update: X = (φφᵀ) ∘ Ξ_{n+1}, p = X W_n, s = W_nᵀ p,
    Ξ_n = X − U_n pᵀ − p U_nᵀ + (s + 1/D_n) U_n U_nᵀ."""
import numpy as np


def term_rows(b, d):
    """Row map: the term of each row and its kind (0: cos row, 1: sin row, 2: real term, b = d = 0)."""
    tm, kind = [], []
    for m, (bb, dd) in enumerate(zip(b, d)):
        if bb == 0.0 and dd == 0.0:
            tm.append(m); kind.append(2)
        else:
            tm += [m, m]; kind += [0, 1]
    return np.array(tm), np.array(kind)


def uv(a, b, d, rows, x):
    tm, kind = rows
    co, si = np.cos(d[tm] * x), np.sin(d[tm] * x)
    U = np.where(kind == 0, a[tm] * co + b[tm] * si, np.where(kind == 1, a[tm] * si - b[tm] * co, a[tm]))
    V = np.where(kind == 0, co, np.where(kind == 1, si, 1.0))
    return U, V


def decay(c, rows, dt):
    return np.exp(-c[rows[0]] * dt)


def factor(a, b, c, d, t, s2):
    """The forward celerite factor: W [N × R], D [N]."""
    rows = term_rows(b, d)
    R = len(rows[0])
    N = len(t)
    W, D = np.zeros((N, R)), np.zeros(N)
    S = np.zeros((R, R))
    for n in range(N):
        U, V = uv(a, b, d, rows, t[n])
        if n > 0:
            ph = decay(c, rows, t[n] - t[n - 1])
            S = np.outer(ph, ph) * (S + D[n - 1] * np.outer(W[n - 1], W[n - 1]))
        D[n] = np.sum(a) + s2[n] - U @ S @ U
        W[n] = (V - S @ U) / D[n]
    return W, D


def predict_var(a, b, c, d, t, s2, tau):
    """Posterior variance of the latent f(τ) at ascending τ, by the two sweeps of K6."""
    a, b, c, d, t, s2, tau = (np.asarray(x, dtype=np.float64) for x in (a, b, c, d, t, s2, tau))
    rows = term_rows(b, d)
    R = len(rows[0])
    N, M = len(t), len(tau)
    suma = np.sum(a)
    W, D = factor(a, b, c, d, t, s2)
    n0 = np.searchsorted(t, tau, side="left")
    # (a) forward replay: Q = S_{n−1} + D_{n−1} W_{n−1} W_{n−1}ᵀ, the state just after absorbing point n − 1
    Dt, g = np.zeros(M), np.zeros((M, R))
    Q = np.zeros((R, R))
    m = 0
    for n in range(N + 1):
        while m < M and n0[m] == n:
            U, V = uv(a, b, d, rows, tau[m])
            e = decay(c, rows, tau[m] - t[n - 1]) if n > 0 else np.zeros(R)
            x = e * U
            y = Q @ x
            Dt[m] = suma - x @ y
            if n < N:
                g[m] = decay(c, rows, t[n] - tau[m]) * (e * y - V)
            m += 1
        if n < N:
            ph = decay(c, rows, t[n] - t[n - 1]) if n > 0 else np.zeros(R)
            Q = np.outer(ph, ph) * Q + D[n] * np.outer(W[n], W[n])
    # (b) backward sweep of Ξ
    var = Dt.copy()
    Xi = np.zeros((R, R))
    m = M - 1
    while m >= 0 and n0[m] == N:
        m -= 1
    for n in range(N - 1, -1, -1):
        U, _ = uv(a, b, d, rows, t[n])
        ph = decay(c, rows, t[n + 1] - t[n]) if n + 1 < N else np.zeros(R)
        X = np.outer(ph, ph) * Xi
        p = X @ W[n]
        s = W[n] @ p
        Xi = X - np.outer(U, p) - np.outer(p, U) + (s + 1.0 / D[n]) * np.outer(U, U)
        while m >= 0 and n0[m] == n:
            var[m] -= g[m] @ Xi @ g[m]
            m -= 1
    return var


def kernel(a, b, c, d, lag):
    lag = np.abs(np.asarray(lag, dtype=np.float64))
    return sum(np.exp(-cc * lag) * (aa * np.cos(dd * lag) + bb * np.sin(dd * lag)) for aa, bb, cc, dd in zip(a, b, c, d))
