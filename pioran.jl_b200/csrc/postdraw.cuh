// postdraw.cuh — K7: draws from the posterior of the celerite GP at new times (rand of fp(τ, σ²_τ) for a PosteriorGP,
// the reference's dense route being cov(fp, τ) through predict_cov, src/direct_solver.jl:28-119, and an M × M Cholesky),
// by Matheron's rule in O((N + M)·R) per draw on two factors computed once per parameter vector:
//
//   G: the data times t merged with τ (a data point first at a tie, the τ points in their order), noise ν σ²_n at data points
//      and σ²_τ at τ points;  (W^G, D^G): the STEP_STORE factor of K(G, G) + diag(noise);  (W, D): that of K̃ = K(t, t) + diag(ν σ²).
//   draw(τ_m) = μ + u(τ_m) + Σ_n k(|τ_m − t_n|) z_n,   u = L^G √D^G q (a prior draw on G, sim of celerite_solver.jl:536-546),
//                                                      z = K̃⁻¹ (ỹ − μ − u(t))            (solve_prec!, :115-158)
// The result is distributed as fp(τ, σ²_τ): the posterior of the latent f at τ plus independent noise of variance σ²_τ.  For
// the same q it is not the draw the dense route makes (that factors the posterior covariance itself).
//
// Three passes over G per draw, all decays taken per G step (φ_k: t_{k−1} → t_k):
//   pass 1 (forward)   f ← φ_k ∘ f, g ← φ_k ∘ g;  e = √D^G_k q_k;  u_k = U_kᵀ f + e;  f ← f + W^G_k e
//                      data point n: z_n = (ỹ_n − μ − u_k) − U_kᵀ g;  g ← g + W_n z_n        τ point m: out_m = μ + u_k
//   pass 2 (backward)  data point n: z_n ← z_n / D_n − W_nᵀ P;  P ← P + U_k z_n                τ point m: out_m += V_kᵀ P
//                      then P ← φ_k ∘ P  (the backward substitution and pred's backward sweep share the state P)
//   pass 3 (forward)   Q ← φ_k ∘ Q;  data point n: Q ← Q + V_k z_n                              τ point m: out_m += U_kᵀ Q
// A data point tied with τ_m precedes it in G, so pass 3 absorbs it and pass 2 does not: each z_n enters each draw once.
// The numpy restatement is tests/tools/proto/postdraw_math.py.
//
// Layout: one CTA per (parameter vector, group of up to PD_MAXW draws), one warp per draw; lane l owns rows l + 32·j, j < PT.
// U, V, φ (sincos_large at absolute times, one exp per term), W^G, √D^G, W, D and ỹ − μ of PD_CH steps are staged in shared
// memory by the whole CTA and read by all its draws; the O(R²) factorisations are not repeated per draw.  A parameter vector
// whose factors have a pivot ≤ 0 (or NaN) gets NaN in all of its S·M outputs.
#pragma once
#include "common.cuh"
#include "posterior.cuh"

namespace pioran {

constexpr int PD_CH = 8;      // steps staged at once
constexpr int PD_MAXW = 16;   // draws (warps) per CTA

struct PostDrawArgs {
    const double* gt;                      // merged times [NG]
    const int* gcode;                      // [NG]: n ≥ 0 data point n, −m − 1 prediction point m
    int64_t N, M, NG;
    int S, Jt, R, RPL;                     // draws per set, terms, rank, leading dimension of both stored factors
    const double* a; const double* b; const double* c; const double* d;   // [B × Jt]
    const int* term_row;                   // as in the generic K2 kernel
    const double* mu;                      // [B] or nullptr
    const double* y;                       // resident data [N], or per set [B × N] when y_batch
    bool y_batch;
    const double* WG; const double* DG;    // factor of the merged covariance [B × NG × RPL], [B × NG]
    const double* W; const double* D;      // factor of the data covariance [B × N × RPL], [B × N]
    const double* q;                       // [B × S × NG] standard normals in merged order
    double* z;                             // workspace [B × S × N]
    double* out;                           // [B × S × M]
};

// Noise on the merged grid for B parameter vectors: ν σ²_n at data points, σ²_τ at prediction points ([B × NG]).
__global__ void merged_noise_kernel(const int* __restrict__ gcode, const double* __restrict__ s2, const double* __restrict__ nu,
                                    double s2tau, int64_t NG, int B, double* __restrict__ out) {
    const int64_t total = (int64_t)B * NG;
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < total; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = k / NG, code = gcode[k - i * NG];
        out[k] = code >= 0 ? (nu ? nu[i] : 1.0) * s2[code] : s2tau;
    }
}

// grid = (⌈S / warps⌉, B), block = 32 · warps (warps ≤ PD_MAXW)
template <int PT>
__global__ void __launch_bounds__(32 * PD_MAXW) celerite_postdraw_kernel(const PostDrawArgs pa) {
    constexpr int LD = 32 * PT;
    __shared__ __align__(16) double tabU[PD_CH][LD], tabV[PD_CH][LD], tabP[PD_CH][LD], tabWG[PD_CH][LD], tabW[PD_CH][LD];
    __shared__ double tabS[PD_CH], tabD[PD_CH], tabY[PD_CH];
    __shared__ int tabC[PD_CH];

    const int th = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, nthr = blockDim.x;
    const int s = blockIdx.x * (nthr >> 5) + (tid >> 5);   // this warp's draw
    const bool active = s < pa.S;
    const int Jt = pa.Jt, R = pa.R, RPL = pa.RPL;
    const int64_t N = pa.N, M = pa.M, NG = pa.NG;
    const double* ca = pa.a + (size_t)th * Jt;
    const double* cb = pa.b + (size_t)th * Jt;
    const double* cc = pa.c + (size_t)th * Jt;
    const double* cd = pa.d + (size_t)th * Jt;
    const double* WGs = pa.WG + (size_t)th * NG * RPL;
    const double* DGs = pa.DG + (size_t)th * NG;
    const double* Ws = pa.W + (size_t)th * N * RPL;
    const double* Ds = pa.D + (size_t)th * N;
    const double* ys = pa.y_batch ? pa.y + (size_t)th * N : pa.y;
    const double mu = pa.mu ? pa.mu[th] : 0.0;
    const size_t row = (size_t)th * pa.S + (active ? s : 0);
    const double* qs = pa.q + row * NG;
    double* zs = pa.z + row * N;
    double* out = pa.out + row * M;

    // a non-positive (or NaN) pivot in either factor: no draw exists, every output of the set is NaN
    int bad = 0;
    for (int64_t k = tid; k < NG; k += nthr) bad |= !(DGs[k] > 0.0);
    for (int64_t n = tid; n < N; n += nthr) bad |= !(Ds[n] > 0.0);
    if (__syncthreads_or(bad)) {
        if (active)
            for (int64_t m = lane; m < M; m += 32) out[m] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    for (int k = tid; k < PD_CH * LD; k += nthr) {   // rows ≥ R stay zero
        (&tabU[0][0])[k] = 0.0; (&tabV[0][0])[k] = 0.0; (&tabP[0][0])[k] = 0.0; (&tabWG[0][0])[k] = 0.0; (&tabW[0][0])[k] = 0.0;
    }
    __syncthreads();

    // U, V, φ of steps [k0, k0 + ns) (celerite_solver.jl:51-64), and the factor rows a pass reads
    auto stage = [&](int64_t k0, int ns, bool merged, bool data) {
        for (int idx = tid; idx < ns * Jt; idx += nthr) {
            const int st = idx / Jt, m = idx - st * Jt;
            const int64_t k = k0 + st;
            const double x = pa.gt[k];
            const double ph = k >= 1 ? exp(-cc[m] * (x - pa.gt[k - 1])) : 0.0;
            const int tr = pa.term_row[m];
            if (tr < 0) {
                const int r0 = -tr - 1;
                tabU[st][r0] = ca[m]; tabV[st][r0] = 1.0; tabP[st][r0] = ph;
            } else {
                double si, co;
                sincos_large(cd[m] * x, &si, &co);
                tabU[st][tr] = ca[m] * co + cb[m] * si;       // celerite_solver.jl:60
                tabU[st][tr + 1] = ca[m] * si - cb[m] * co;   // celerite_solver.jl:59
                tabV[st][tr] = co; tabV[st][tr + 1] = si;
                tabP[st][tr] = ph; tabP[st][tr + 1] = ph;
            }
        }
        for (int idx = tid; idx < ns * R; idx += nthr) {
            const int st = idx / R, r = idx - st * R;
            const int64_t k = k0 + st;
            const int code = pa.gcode[k];
            if (merged) tabWG[st][r] = WGs[k * RPL + r];
            if (data) tabW[st][r] = code >= 0 ? Ws[(int64_t)code * RPL + r] : 0.0;
        }
        for (int st = tid; st < ns; st += nthr) {
            const int64_t k = k0 + st;
            const int code = pa.gcode[k];
            tabC[st] = code;
            if (merged) { tabS[st] = sqrt(DGs[k]); tabY[st] = code >= 0 ? ys[code] - mu : 0.0; }
            if (data) tabD[st] = code >= 0 ? Ds[code] : 1.0;
        }
    };

    // ================================================================ pass 1: prior draw on G, forward substitution of the residual
    double f[PT], g[PT];
#pragma unroll
    for (int j = 0; j < PT; j++) { f[j] = 0.0; g[j] = 0.0; }
    for (int64_t kb = 0; kb < NG; kb += PD_CH) {
        const int ns = (int)((NG - kb) < PD_CH ? (NG - kb) : PD_CH);
        stage(kb, ns, true, true);
        __syncthreads();
        if (active) {
            for (int st = 0; st < ns; st++) {
                const double e = tabS[st] * qs[kb + st];
                double pf = 0.0, pg = 0.0;
#pragma unroll
                for (int j = 0; j < PT; j++) {
                    const double ph = tabP[st][lane + 32 * j], u = tabU[st][lane + 32 * j];
                    f[j] *= ph; g[j] *= ph;
                    pf = fma(u, f[j], pf);
                    pg = fma(u, g[j], pg);
                }
#pragma unroll
                for (int sft = 16; sft >= 1; sft >>= 1) {
                    pf += __shfl_xor_sync(FULL, pf, sft);
                    pg += __shfl_xor_sync(FULL, pg, sft);
                }
                const double u = pf + e;
#pragma unroll
                for (int j = 0; j < PT; j++) f[j] = fma(tabWG[st][lane + 32 * j], e, f[j]);
                const int code = tabC[st];
                if (code >= 0) {
                    const double zf = (tabY[st] - u) - pg;
#pragma unroll
                    for (int j = 0; j < PT; j++) g[j] = fma(tabW[st][lane + 32 * j], zf, g[j]);
                    if (lane == 0) zs[code] = zf;
                } else if (lane == 0) {
                    out[-code - 1] = mu + u;
                }
            }
        }
        __syncthreads();   // the tables are rebuilt for the next PD_CH steps
    }

    // ================================================================ pass 2: backward substitution and pred's backward sweep
    double P[PT];
#pragma unroll
    for (int j = 0; j < PT; j++) P[j] = 0.0;
    for (int64_t hi = NG; hi > 0; hi -= PD_CH) {
        const int64_t lo = hi - PD_CH > 0 ? hi - PD_CH : 0;
        const int ns = (int)(hi - lo);
        stage(lo, ns, false, true);
        __syncthreads();
        if (active) {
            for (int st = ns - 1; st >= 0; st--) {
                const int code = tabC[st];
                double part = 0.0;
#pragma unroll
                for (int j = 0; j < PT; j++) part = fma(code >= 0 ? tabW[st][lane + 32 * j] : tabV[st][lane + 32 * j], P[j], part);
                part = warp_sum(part);
                if (code >= 0) {
                    const double zn = zs[code] / tabD[st] - part;
#pragma unroll
                    for (int j = 0; j < PT; j++) P[j] = fma(tabU[st][lane + 32 * j], zn, P[j]);
                    __syncwarp();
                    if (lane == 0) zs[code] = zn;
                } else if (lane == 0) {
                    out[-code - 1] += part;
                }
#pragma unroll
                for (int j = 0; j < PT; j++) P[j] *= tabP[st][lane + 32 * j];
            }
        }
        __syncthreads();
    }

    // ================================================================ pass 3: pred's forward sweep
    double Q[PT];
#pragma unroll
    for (int j = 0; j < PT; j++) Q[j] = 0.0;
    for (int64_t kb = 0; kb < NG; kb += PD_CH) {
        const int ns = (int)((NG - kb) < PD_CH ? (NG - kb) : PD_CH);
        stage(kb, ns, false, false);
        __syncthreads();
        if (active) {
            for (int st = 0; st < ns; st++) {
                const int code = tabC[st];
#pragma unroll
                for (int j = 0; j < PT; j++) Q[j] *= tabP[st][lane + 32 * j];
                if (code >= 0) {
                    const double zn = zs[code];
#pragma unroll
                    for (int j = 0; j < PT; j++) Q[j] = fma(tabV[st][lane + 32 * j], zn, Q[j]);
                } else {
                    double part = 0.0;
#pragma unroll
                    for (int j = 0; j < PT; j++) part = fma(tabU[st][lane + 32 * j], Q[j], part);
                    part = warp_sum(part);
                    if (lane == 0) out[-code - 1] += part;
                }
            }
        }
        __syncthreads();
    }
}

}  // namespace pioran
