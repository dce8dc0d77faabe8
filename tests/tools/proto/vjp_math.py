"""Math-level prototype of the K5r step rule (csrc/vjp.cuh): the reverse-mode adjoint (vector-Jacobian product) of the
explicit-coefficient celerite sweep in the full-square state form of jvp_math.py.  One backward sweep returns ∂logL with respect
to a, b, c, d, μ, ν and the data row (y, σ²) at once (Foreman-Mackey 2018, RNAAS 2, 31).

Forward step n (jvp_math.logl_jvp):  gin = g + w z₋;  g = φ∘gin;  Tin = T + q wᵀ;  T = (φφᵀ)∘Tin;  p = T u;
    D = Σa + ν s2_n − uᵀp;  z = ỹ_n − uᵀg;  q = V − p;  w = q / D;  logL = −½ Σ log|D| − ½ Σ z²/D − ½ N log 2π.
Backward step n, with the state adjoint T̄ kept SYMMETRIC (T and Tin are symmetric functions of the inputs, so only the symmetric
part of an adjoint reaches them; it lets every contraction be a row sum, as in the forward tile):
    z̄ = Σ ḡin₊∘w − z/D                         D̄ = −½/D + ½ z²/D² − (w̄·w)/D          q̄ ← q̄ + w̄/D  (= V̄)
    p̄ = −q̄ − D̄ u;   ḡ ← ḡ − z̄ u;   ū = −z̄ g − D̄ p + T p̄;   T̄ ← T̄ + ½(p̄ uᵀ + u p̄ᵀ)
    φ̄ = 2 Σ_c (T̄∘Tin)_rc φ_c + ḡ∘gin;   T̄ ← (φφᵀ)∘T̄;   q̄₋ = T̄ w₋;   ḡin = φ∘ḡ;   w̄₋ = T̄ q₋ + ḡin z₋;   ḡ₋ = ḡin
and the row tables map back to the terms (U_cos = a cos + b sin, U_sin = a sin − b cos, V = (cos, sin), φ = e^{−cΔ}, θ = d t):
    ā += Ū_c cos + Ū_s sin;  b̄ += Ū_c sin − Ū_s cos;  d̄ += t (Ū_s U_c − Ū_c U_s − V̄_c sin + V̄_s cos);  c̄ += −Δ φ φ̄.
A real term takes one row (U = a, V = 1) and reports b̄ = d̄ = 0 exactly.  ȳ_n = z̄_n, μ̄ = −Σ z̄, s̄2_n = ν D̄_n, ν̄ = Σ s2 D̄.
tests/test_vjp_proto.py checks this by duality against the dual-number oracle tests/tools/oracle_jvp.c: ⟨∇, v⟩ = JVP(v)."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from jvp_math import LOG_2PI, term_rows  # noqa: E402


def logl_vjp(a, b, c, d, t, y, s2, mu=0.0, nu=1.0, rows=None):
    """One coefficient set → (logL, {"a", "b", "c", "d" [Jt], "mu", "nu" (float), "y", "s2" [N]})."""
    a, b, c, d = (np.asarray(x, dtype=np.float64) for x in (a, b, c, d))
    t, y, s2 = (np.asarray(x, dtype=np.float64) for x in (t, y, s2))
    Jt, N = a.shape[0], t.shape[0]
    if rows is None:
        rows, R = term_rows(b, d)
    else:
        R = sum(1 if r < 0 else 2 for r in rows)
    U, V, PH = np.zeros((N, R)), np.zeros((N, R)), np.zeros((N, R))
    dt = np.concatenate([[0.0], np.diff(t)])
    for m in range(Jt):
        ph = np.exp(-c[m] * dt)
        ph[0] = 0.0
        tr = rows[m]
        if tr < 0:
            U[:, -tr - 1], V[:, -tr - 1], PH[:, -tr - 1] = a[m], 1.0, ph
        else:
            co, si = np.cos(d[m] * t), np.sin(d[m] * t)
            U[:, tr], U[:, tr + 1] = a[m] * co + b[m] * si, a[m] * si - b[m] * co
            V[:, tr], V[:, tr + 1] = co, si
            PH[:, tr] = PH[:, tr + 1] = ph
    # ---- forward: keep Tin, q, g, D, z per step (the kernel keeps q, g, D, z and recomputes Tin from checkpoints)
    suma = a.sum()
    T, g, q, w, zprev = np.zeros((R, R)), np.zeros(R), np.zeros(R), np.zeros(R), 0.0
    Tins, qs, gs, Ds, zs = [], np.zeros((N, R)), np.zeros((N, R)), np.zeros(N), np.zeros(N)
    chi2 = logdet = 0.0
    for n in range(N):
        ph, u = PH[n], U[n]
        g = ph * (g + w * zprev)
        Tin = T + np.outer(q, w)
        Tins.append(Tin)
        T = np.outer(ph, ph) * Tin
        p = T @ u
        D = suma + nu * s2[n] - u @ p
        z = (y[n] - mu) - u @ g
        q = V[n] - p
        w = q / D
        zprev = z
        qs[n], gs[n], Ds[n], zs[n] = q, g, D, z
        chi2 += z * z / D
        logdet += np.log(D) if n == 0 else np.log(abs(D))
    L = -logdet / 2 - N * LOG_2PI / 2 - chi2 / 2
    # ---- backward
    Tb, qb, wb, gb = np.zeros((R, R)), np.zeros(R), np.zeros(R), np.zeros(R)
    Ub, Vb, PHb = np.zeros((N, R)), np.zeros((N, R)), np.zeros((N, R))
    yb, Db = np.zeros(N), np.zeros(N)
    for n in range(N - 1, -1, -1):
        ph, u, D, z, qn, gn = PH[n], U[n], Ds[n], zs[n], qs[n], gs[n]
        wn = qn / D
        qm, gm, zm = (qs[n - 1], gs[n - 1], zs[n - 1]) if n else (np.zeros(R), np.zeros(R), 0.0)
        wm = qm / Ds[n - 1] if n else np.zeros(R)
        zbar = gb @ wn - z / D                       # gb is ḡin of step n + 1 here
        Dbar = -0.5 / D + 0.5 * z * z / (D * D) - (wb @ wn) / D
        qbn = qb + wb / D
        pb = -qbn - Dbar * u
        gbn = gb - zbar * u
        Tn = np.outer(ph, ph) * Tins[n]
        ub = -zbar * gn - Dbar * (V[n] - qn) + Tn @ pb
        Tb = Tb + 0.5 * (np.outer(pb, u) + np.outer(u, pb))
        gin = gm + wm * zm
        PHb[n] = 2.0 * (Tb * Tins[n]) @ ph + gbn * gin
        Tb = np.outer(ph, ph) * Tb
        ginb = ph * gbn
        qb, wb, gb = Tb @ wm, Tb @ qm + ginb * zm, ginb
        Ub[n], Vb[n], yb[n], Db[n] = ub, qbn, zbar, Dbar
    grad = {"a": np.full(Jt, Db.sum()), "b": np.zeros(Jt), "c": np.zeros(Jt), "d": np.zeros(Jt),
            "mu": -yb.sum(), "nu": float(s2 @ Db), "y": yb, "s2": nu * Db}
    for m in range(Jt):
        tr = rows[m]
        if tr < 0:
            r = -tr - 1
            grad["a"][m] += Ub[:, r].sum()
            grad["c"][m] = np.sum(-dt * PH[:, r] * PHb[:, r])
        else:
            co, si = V[:, tr], V[:, tr + 1]
            uc, us = U[:, tr], U[:, tr + 1]
            grad["a"][m] += np.sum(Ub[:, tr] * co + Ub[:, tr + 1] * si)
            grad["b"][m] = np.sum(Ub[:, tr] * si - Ub[:, tr + 1] * co)
            grad["d"][m] = np.sum(t * (Ub[:, tr + 1] * uc - Ub[:, tr] * us - Vb[:, tr] * si + Vb[:, tr + 1] * co))
            grad["c"][m] = np.sum(-dt * PH[:, tr] * (PHb[:, tr] + PHb[:, tr + 1]))
    return L, grad


def logl_vjp_batch(a, b, c, d, t, y, s2, mu=None, nu=None, y_batch=None, s2_batch=None):
    """Batched form with the shapes of Context.celerite_logl_vjp; term rows over the whole batch."""
    a, b, c, d = (np.atleast_2d(np.asarray(x, dtype=np.float64)) for x in (a, b, c, d))
    B = a.shape[0]
    rows, _ = term_rows(b, d)
    L, G = np.empty(B), []
    for i in range(B):
        L[i], gi = logl_vjp(a[i], b[i], c[i], d[i], t, y_batch[i] if y_batch is not None else y,
                            s2_batch[i] if s2_batch is not None else s2, 0.0 if mu is None else mu[i], 1.0 if nu is None else nu[i],
                            rows=rows)
        G.append(gi)
    return L, {k: np.array([g[k] for g in G]) for k in G[0]}
