"""Numpy restatement of the posterior-draw sweep K7 (csrc/postdraw.cuh) on the reference's variables
(src/celerite_solver.jl): draws of fp(τ, σ²_τ) conditioned on the data by Matheron's rule, in O((N + M)·R) per draw on two
factors computed once per coefficient set.

Merged grid G: the data times t and the prediction times τ, a data point first at a tie, the τ points in their order.
Noise on G: σ̃²_n = ν σ²_n at data points, σ²_τ at τ points.  Factors (the STEP_STORE sweep, postvar_math.factor):
(W^G, D^G) of K(G, G) + diag(noise), (W, D) of K̃ = K(t, t) + diag(ν σ²).  Per draw with standard normals q [N + M]
(merged-grid order), three passes over G, all decays taken per G step (φ_k: t_{k−1} → t_k):

  pass 1 (forward):   f ← φ_k ∘ f;  g ← φ_k ∘ g;  e = √D^G_k q_k;  u_k = U_kᵀ f + e;  f ← f + W^G_k e        (sim, :536-546)
                      data point n:  z_n = (ỹ_n − μ − u_k) − U_kᵀ g;  g ← g + W_n z_n                (solve_prec! forward)
                      τ point m:     out_m = μ + u_k
  pass 2 (backward):  P ← φ_{k+1} ∘ P  (P: Σ_{n absorbed} U(t_n) z_n decayed to t_k)
                      data point n:  z_n ← z_n / D_n − W_nᵀ P;  P ← P + U_k z_n                       (solve_prec! backward)
                      τ point m:     out_m += V(τ_m)ᵀ P                                              (pred backward sweep)
  pass 3 (forward):   Q ← φ_k ∘ Q;  data point n: Q ← Q + V_k z_n;  τ point m: out_m += U(τ_m)ᵀ Q      (pred forward sweep)

At a tie the data point precedes the τ point, so pass 3 absorbs it and pass 2 does not: every data point enters the
correction Σ_n k(|τ_m − t_n|) z_n once."""
import numpy as np
from scipy.linalg import cho_factor, cho_solve, cholesky

from postvar_math import factor, kernel, term_rows, uv


def merged_grid(t, tau):
    """Merged order of t and τ (data first at a tie): times [N + M] and codes (n ≥ 0: data point n, −m − 1: τ point m)."""
    t, tau = np.asarray(t, dtype=np.float64), np.asarray(tau, dtype=np.float64)
    code = np.concatenate([np.arange(len(t)), -np.arange(len(tau)) - 1])
    key = np.concatenate([np.zeros(len(t)), np.ones(len(tau))])
    order = np.lexsort((key, np.concatenate([t, tau])))   # stable: the τ points keep their order
    return np.concatenate([t, tau])[order], code[order]


def posterior_draws(a, b, c, d, t, y, s2, tau, q, mu=0.0, sigma2_tau=1e-18):
    """Draws [S × M] of the posterior at τ for the standard normals q [S × (N + M)] in merged-grid order."""
    a, b, c, d, t, y, s2, tau = (np.asarray(x, dtype=np.float64) for x in (a, b, c, d, t, y, s2, tau))
    q = np.atleast_2d(np.asarray(q, dtype=np.float64))
    rows = term_rows(b, d)
    R = len(rows[0])
    N, M = len(t), len(tau)
    G, code = merged_grid(t, tau)
    noise = np.where(code >= 0, s2[np.maximum(code, 0)], sigma2_tau)
    WG, DG = factor(a, b, c, d, G, noise)
    W, D = factor(a, b, c, d, t, s2)
    UV = [uv(a, b, d, rows, x) for x in G]
    phi = [np.zeros(R)] + [np.exp(-c[rows[0]] * (G[k] - G[k - 1])) for k in range(1, N + M)]
    sq = np.sqrt(DG)
    out = np.zeros((q.shape[0], M))
    for s, qs in enumerate(q):
        z = np.zeros(N)
        f, g = np.zeros(R), np.zeros(R)
        for k in range(N + M):   # pass 1
            U = UV[k][0]
            f, g = phi[k] * f, phi[k] * g
            e = sq[k] * qs[k]
            u = U @ f + e
            f = f + WG[k] * e
            if code[k] >= 0:
                n = code[k]
                z[n] = (y[n] - mu - u) - U @ g
                g = g + W[n] * z[n]
            else:
                out[s, -code[k] - 1] = mu + u
        P = np.zeros(R)
        for k in range(N + M - 1, -1, -1):   # pass 2
            if k + 1 < N + M:
                P = phi[k + 1] * P
            U, V = UV[k]
            if code[k] >= 0:
                n = code[k]
                z[n] = z[n] / D[n] - W[n] @ P
                P = P + U * z[n]
            else:
                out[s, -code[k] - 1] += V @ P
        Q = np.zeros(R)
        for k in range(N + M):   # pass 3
            U, V = UV[k]
            Q = phi[k] * Q
            if code[k] >= 0:
                Q = Q + V * z[code[k]]
            else:
                out[s, -code[k] - 1] += U @ Q
    return out


def dense_draws(a, b, c, d, t, y, s2, tau, q, mu=0.0, sigma2_tau=1e-18):
    """The same draws with dense matrices: the Cholesky factor of K(G, G) + diag(noise) times q, then a Cholesky solve for
    the correction.  In exact arithmetic the celerite factor L√D of the recursion is that Cholesky factor."""
    a, b, c, d, t, y, s2, tau = (np.asarray(x, dtype=np.float64) for x in (a, b, c, d, t, y, s2, tau))
    G, code = merged_grid(t, tau)
    noise = np.where(code >= 0, s2[np.maximum(code, 0)], sigma2_tau)
    L = cholesky(kernel(a, b, c, d, G[:, None] - G[None, :]) + np.diag(noise), lower=True)
    dat, pre = np.flatnonzero(code >= 0), np.flatnonzero(code < 0)
    dat, pre = dat[np.argsort(code[dat])], pre[np.argsort(-code[pre] - 1)]
    u = np.atleast_2d(q) @ L.T                                   # [S × (N + M)]
    K = cho_factor(kernel(a, b, c, d, t[:, None] - t[None, :]) + np.diag(s2), lower=True)
    z = cho_solve(K, (y - mu - u[:, dat]).T)                     # [N × S]
    return mu + u[:, pre] + (kernel(a, b, c, d, tau[:, None] - t[None, :]) @ z).T
