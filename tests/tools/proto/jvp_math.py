"""Math-level prototype of the K5g step rule (csrc/jvp.cuh): the forward-mode tangent of the explicit-coefficient celerite sweep,
in the full-square state form of the register-file kernels, with tangents on a, b, c, d, μ, ν, y and σ².  P directions are carried
at once (ForwardDiff's chunk).  Checked against central differences of the oracle's logl (oracle/pioran_oracle.c) when run as a
script; tests/test_jvp_proto.py runs the same checks.  The GPU tests compare against the independent dual-number oracle
tests/tools/oracle_jvp.c instead (the reference's own sweep, not this full-square form)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
LOG_2PI = 1.8378770664093453


def term_rows(b, d):
    """make_term_rows (csrc/api.cu) over a batch [B × Jt] or one set [Jt]: a term real for every set takes one row."""
    b, d = np.atleast_2d(b), np.atleast_2d(d)
    real = np.all((b == 0.0) & (d == 0.0), axis=0)
    rows, R = [], 0
    for m in range(b.shape[1]):
        rows.append(-(R + 1) if real[m] else R)
        R += 1 if real[m] else 2
    return rows, R


def logl_jvp(a, b, c, d, t, y, s2, mu=0.0, nu=1.0, da=None, db=None, dc=None, dd=None, dmu=None, dnu=None, dy=None, ds2=None,
             rows=None):
    """One coefficient set: a, b, c, d [Jt]; tangents da … dd [P × Jt], dmu, dnu [P], dy, ds2 [P × N] (None = zero).
    Returns (logL, dlogL [P])."""
    a, b, c, d = (np.asarray(x, dtype=np.float64) for x in (a, b, c, d))
    t, y, s2 = (np.asarray(x, dtype=np.float64) for x in (t, y, s2))
    Jt, N = a.shape[0], t.shape[0]
    given = [x for x in (da, db, dc, dd, dmu, dnu, dy, ds2) if x is not None]
    P = np.shape(given[0])[0] if given else 1
    z2 = lambda n: np.zeros((P, n))
    da, db, dc, dd = (np.asarray(x, dtype=np.float64) if x is not None else z2(Jt) for x in (da, db, dc, dd))
    dmu = np.asarray(dmu, dtype=np.float64) if dmu is not None else np.zeros(P)
    dnu = np.asarray(dnu, dtype=np.float64) if dnu is not None else np.zeros(P)
    dy, ds2 = (np.asarray(x, dtype=np.float64) if x is not None else z2(N) for x in (dy, ds2))
    if rows is None:
        rows, R = term_rows(b, d)
    else:
        R = sum(1 if r < 0 else 2 for r in rows)
    # row tables and their tangents [N × R], [P × N × R]
    U, V, PH = np.zeros((N, R)), np.zeros((N, R)), np.zeros((N, R))
    dU, dV, dPH = np.zeros((P, N, R)), np.zeros((P, N, R)), np.zeros((P, N, R))
    dt = np.concatenate([[0.0], np.diff(t)])
    for m in range(Jt):
        ph = np.exp(-c[m] * dt)
        ph[0] = 0.0
        dph = -dc[:, m, None] * dt[None, :] * ph[None, :]
        tr = rows[m]
        if tr < 0:
            r0 = -tr - 1
            U[:, r0], V[:, r0], PH[:, r0] = a[m], 1.0, ph
            dU[:, :, r0], dPH[:, :, r0] = da[:, m, None], dph
        else:
            co, si = np.cos(d[m] * t), np.sin(d[m] * t)
            uc, us = a[m] * co + b[m] * si, a[m] * si - b[m] * co
            U[:, tr], U[:, tr + 1] = uc, us
            V[:, tr], V[:, tr + 1] = co, si
            PH[:, tr] = PH[:, tr + 1] = ph
            dtd = dd[:, m, None] * t[None, :]
            dU[:, :, tr] = da[:, m, None] * co + db[:, m, None] * si - dtd * us
            dU[:, :, tr + 1] = da[:, m, None] * si - db[:, m, None] * co + dtd * uc
            dV[:, :, tr], dV[:, :, tr + 1] = -dtd * si, dtd * co
            dPH[:, :, tr] = dPH[:, :, tr + 1] = dph
    suma, dsuma = a.sum(), da.sum(axis=1)
    T, dT = np.zeros((R, R)), np.zeros((P, R, R))
    g, dg = np.zeros(R), np.zeros((P, R))
    q, dq, w, dw = np.zeros(R), np.zeros((P, R)), np.zeros(R), np.zeros((P, R))
    zprev, dzprev = 0.0, np.zeros(P)
    chi2, dchi2, logdet, dlog = 0.0, np.zeros(P), 0.0, np.zeros(P)
    for n in range(N):
        ph, dph, u, du = PH[n], dPH[:, n], U[n], dU[:, n]
        gin, dgin = g + w * zprev, dg + dw * zprev + w[None] * dzprev[:, None]
        dg = dph * gin[None] + ph[None] * dgin
        g = ph * gin
        Tin = T + np.outer(q, w)
        dTin = dT + dq[:, :, None] * w[None, None, :] + q[None, :, None] * dw[:, None, :]
        PP = np.outer(ph, ph)
        dPP = dph[:, :, None] * ph[None, None, :] + ph[None, :, None] * dph[:, None, :]
        T, dT = PP * Tin, dPP * Tin[None] + PP[None] * dTin
        p = T @ u
        dp = np.einsum("prc,c->pr", dT, u) + du @ T.T
        D = suma + nu * s2[n] - u @ p
        dD = dsuma + dnu * s2[n] + nu * ds2[:, n] - (du @ p + dp @ u)
        z = (y[n] - mu) - u @ g
        dz = (dy[:, n] - dmu) - (du @ g + dg @ u)
        q, dq = V[n] - p, dV[:, n] - dp
        w = q / D
        dw = (dq - w[None] * dD[:, None]) / D
        zprev, dzprev = z, dz
        chi2 += z * z / D
        dchi2 += (2 * z * dz - z * z * dD / D) / D
        logdet += np.log(D) if n == 0 else np.log(abs(D))
        dlog += dD / D
    return -logdet / 2 - N * LOG_2PI / 2 - chi2 / 2, -dlog / 2 - dchi2 / 2


def logl_jvp_batch(a, b, c, d, t, y, s2, mu=None, nu=None, y_batch=None, s2_batch=None, **tan):
    """Batched form with the shapes of Context.celerite_logl_jvp (tangents [B × P × …]); term rows over the whole batch."""
    a, b, c, d = (np.atleast_2d(np.asarray(x, dtype=np.float64)) for x in (a, b, c, d))
    B = a.shape[0]
    rows, _ = term_rows(b, d)
    L, G = np.empty(B), []
    for i in range(B):
        ti = {k: (v[i] if v is not None else None) for k, v in tan.items()}
        L[i], gi = logl_jvp(a[i], b[i], c[i], d[i], t, y_batch[i] if y_batch is not None else y,
                            s2_batch[i] if s2_batch is not None else s2, 0.0 if mu is None else mu[i], 1.0 if nu is None else nu[i],
                            rows=rows, **ti)
        G.append(gi)
    return L, np.array(G)


def central_difference(a, b, c, d, t, y, s2, mu, nu, direction, h=1e-6):
    """(logl(x + h v) − logl(x − h v)) / 2h of the oracle, along one direction v = dict(da=[Jt], …, dy=[N], dmu=float, …)."""
    sys.path.insert(0, ROOT)
    from oracle import oracle as orc

    def at(e):
        g = lambda k, base: base + e * np.asarray(direction.get(k, 0.0))
        nu_e, s2_e = g("dnu", nu), g("ds2", s2)
        return orc.celerite_logl(g("da", a), g("db", b), g("dc", c), g("dd", d), t, g("dy", y) - g("dmu", mu), nu_e * s2_e)

    return (at(h) - at(-h)) / (2 * h)


def _demo():
    sys.path.insert(0, ROOT)
    from oracle import oracle as orc
    rng = np.random.default_rng(0)
    N = 60
    t = np.cumsum(rng.uniform(0.2, 1.5, N)); y = rng.normal(size=N); s2 = np.full(N, 0.3)
    a, b = np.array([1.2, 0.8, -0.3, 0.5]), np.array([0.0, 0.3, -0.1, 0.0])
    c, d = np.array([0.3, 0.2, 1.0, 2.0]), np.array([0.0, 1.5, -2.0, 0.0])
    mu, nu = 0.1, 1.3
    L, _ = logl_jvp(a, b, c, d, t, y, s2, mu, nu)
    print("value vs oracle", abs(L - orc.celerite_logl(a, b, c, d, t, y - mu, nu * s2)))
    for name, size in (("da", 4), ("db", 4), ("dc", 4), ("dd", 4), ("dmu", None), ("dnu", None), ("dy", N), ("ds2", N)):
        v = rng.normal(size=size) if size else 1.0
        _, g = logl_jvp(a, b, c, d, t, y, s2, mu, nu, **{name: np.array([v])})
        cd = central_difference(a, b, c, d, t, y, s2, mu, nu, {name: v})
        print(f"{name:4s} jvp {g[0]: .10e}  cd {cd: .10e}  rel {abs(g[0] - cd) / max(1.0, abs(cd)):.1e}")


if __name__ == "__main__":
    _demo()
