"""Hamiltonian Monte Carlo on the reference's simu_single run with the GPU value-and-gradient entry (K5): what the NUTS scripts of
examples/turing_distributed/single_pl.jl do with ForwardDiff, here with a plain leapfrog integrator, 16 chains evaluated per call.
The likelihood alone is sampled (flat prior inside the box the chains start in), with the posterior standard deviations of the
shipped ultranest chain as the mass matrix.  Prints the acceptance rate, the energy error of the trajectories and the time per
gradient call — an end-to-end check that the gradients are the gradients of the log-likelihood the library returns.

    python tools/hmc_demo.py [SHO|DRWCelerite] [qpo [feature_scale]]

`qpo` adds one QPO feature (S₀, f₀, Q) to the continuum (n_features = 1): the gradient then runs K1 on dual numbers with the
feature branch and the K5g sweep (csrc/jvp.cuh).  The feature columns start at a fixed narrow peak with a small spread;
`feature_scale` (default 1) multiplies their mass-matrix scales, i.e. their step size, which are guesses rather than posterior
widths."""
import sys
import time

import numpy as np

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import pioran_b200 as pb              # noqa: E402
from conftest import GoldenRun        # noqa: E402

g = GoldenRun("simu_single", "SingleBendingPowerLaw", 3, True)
basis = sys.argv[1] if len(sys.argv) > 1 else "SHO"
qpo = len(sys.argv) > 2 and sys.argv[2] == "qpo"
feature_scale = float(sys.argv[3]) if len(sys.argv) > 3 else 1.0
like = pb.BatchedLikelihood(g.t, g.y, g.s2, "SingleBendingPowerLaw", 20, basis, f_min=g.f_min, f_max=g.f_max, n_features=int(qpo))
post = g.theta[-4000:]                                  # high-weight end of the nested-sampling chain
scale = post.std(axis=0)
rng = np.random.default_rng(1)
C = 16
theta = post[rng.integers(0, len(post), C)].copy()
eps, L, iters = 0.08, 12, 40
lo = np.array([0.0, 1e-6, 0.0, 1e-8, 1e-3, -np.inf])    # stay where the model is defined (α ≥ 0, f₁, variance, ν > 0)
if qpo:
    f0 = np.sqrt(g.f_min * g.f_max)
    feat = np.array([0.05, f0, 5.0])
    theta = np.column_stack([theta, feat * (1 + 0.05 * rng.standard_normal((C, 3)))])
    scale = np.concatenate([scale, feature_scale * np.array([0.02, 0.1 * f0, 1.0])])
    lo = np.concatenate([lo, [0.0, 1e-6, 0.6]])        # S₀ ≥ 0, f₀ > 0, Q > 1/2 (the feature's d = c √(4Q² − 1))
logl, grad = like.value_and_gradient(theta)
acc, dH, calls, t_call = 0, [], 0, 0.0
for it in range(iters):
    p = rng.standard_normal(theta.shape)
    th, lg, gr = theta.copy(), logl.copy(), grad.copy()
    H0 = -lg + 0.5 * (p ** 2).sum(axis=1)
    for _ in range(L):
        p = p + 0.5 * eps * gr * scale
        th = th + eps * p * scale
        t0 = time.perf_counter()
        lg, gr = like.value_and_gradient(th)
        t_call += time.perf_counter() - t0
        calls += 1
        p = p + 0.5 * eps * gr * scale
    H1 = -lg + 0.5 * (p ** 2).sum(axis=1)
    ok = np.isfinite(H1) & np.all(th > lo, axis=1)
    a = ok & (np.log(rng.uniform(size=C)) < np.where(ok, H0 - H1, -np.inf))
    dH.extend((H1 - H0)[ok])
    theta[a], logl[a], grad[a] = th[a], lg[a], gr[a]
    acc += a.sum()
like.close()
dH = np.array(dH)
print(f"{basis}{f' + 1 QPO (feature scale {feature_scale:g})' if qpo else ''}: {C} chains x {iters} trajectories x {L} leapfrog steps: acceptance {acc / (C * iters):.2f}, "
      f"median |dH| {np.median(np.abs(dH)):.3f}, {t_call / calls * 1e3:.2f} ms per value-and-gradient call of {C} chains")
