// postcov.cuh — K8: the full posterior covariance of the celerite GP at new times (cov / mean_and_cov of a PosteriorGP, the
// reference's dense route being predict_cov, src/direct_solver.jl:28-119), one O((N + M)·R) walk per column on the factor
// (W_n, D_n) of the STEP_STORE sweep and the per-point vectors of K6 (postvar.cuh, COV = true).  No matrix inverse.
//
//   C(x, x′) = k(x, x′) − k(x, t)ᵀ K̃⁻¹ k(t, x′),  x ≤ x′
//
// G: the data times and τ merged, a τ point first at a tie (so that a data point at τ lies after it, as n₀ = #{t_n < τ}
// says).  Column x′ = τ_{m′} carries one R-vector w = v + h̃ from x′ down to the start of G:
//   v = Φ(· → x′) U(x′)                       the prior row of x′, decayed back (the data before both points)
//   h̃ = Φ(· → t_{n₀}) h_{n₀}, h_n = A_nᵀ (φ_{n+1} ∘ h_{n+1}) − U_n (W_nᵀ v_n), A_n = I − W_n U_nᵀ   (the data after x)
//   start at x′:      w = w₀(x′) = U(x′) + e_{x′→t_{n₀′}} ∘ (Ξ_{n₀′} g_{x′})   (K6)
//   each G step down: w ← φ^G ∘ w                                            (decay between the two G times, ≤ 1)
//   data point n:     w ← w − U_n (W_nᵀ w)
//   τ point x:        C(x, x′) = −r(x)ᵀ w,   r(x) = S_x U(x) − V(x)            (K6)
// The diagonal is K6's variance D_τ − g_τᵀ Ξ g_τ up to rounding.  The numpy restatement and its derivation are
// tests/tools/proto/postcov_math.py.
//
// Layout (that of K7): one CTA per (parameter vector, group of up to PC_MAXW consecutive columns), one warp per column;
// lane l owns rows l + 32·j, j < PT.  φ^G, U (data steps) and W_n or r(x) of PC_CH steps are staged in shared memory by the
// whole CTA and read by all its columns; a warp joins the walk at its own x′.  Each entry is written twice, at (x′, x) and
// at (x, x′), from one value: the output is exactly symmetric.  A column range [c0, c0 + w) writes rows c0 … c0 + w − 1
// into `out` (row m′ − c0, leading dimension ldo) and its mirror entries in rows m < c0 into `up` ([c0 × w]); with c0 = 0 and
// w = M the two are one M × M matrix.  A parameter vector with a pivot ≤ 0 has NaN r and w₀ from K6, so all its entries are NaN.
#pragma once
#include "common.cuh"
#include "posterior.cuh"

namespace pioran {

constexpr int PC_CH = 8;      // steps staged at once
constexpr int PC_MAXW = 16;   // columns (warps) per CTA

struct PostCovArgs {
    const double* gt;                      // merged times [NG], a τ point first at a tie
    const int* gcode;                      // [NG]: n ≥ 0 data point n, −m − 1 prediction point m
    const int* gpos;                       // [M] position of τ_m in G
    int64_t N, M, NG;
    int Jt, R, RPL;                        // terms, rank, leading dimension of the stored factor
    const double* a; const double* b; const double* c; const double* d;   // [B × Jt]
    const int* term_row;                   // as in the generic K2 kernel
    const double* W;                       // stored factor [B × N × RPL]
    const double* pt;                      // [B × M × 2R]: r(τ), w₀(τ) (K6, COV = true)
    int64_t c0, w;                         // the columns of this launch: [c0, c0 + w)
    double* out; int64_t ldo;              // rows c0 … c0 + w − 1: [B × w × ldo]
    double* up;                            // rows 0 … c0 − 1, columns c0 … c0 + w − 1: [B × c0 × w]
};

// grid = (⌈w / warps⌉, B), block = 32 · warps (warps ≤ PC_MAXW)
template <int PT>
__global__ void __launch_bounds__(32 * PC_MAXW) celerite_postcov_kernel(const PostCovArgs pa) {
    constexpr int LD = 32 * PT;
    __shared__ __align__(16) double tabP[PC_CH][LD], tabU[PC_CH][LD], tabX[PC_CH][LD];
    __shared__ int tabC[PC_CH];

    const int th = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, nthr = blockDim.x, nw = nthr >> 5;
    const int Jt = pa.Jt, R = pa.R, RPL = pa.RPL;
    const int64_t M = pa.M, NG = pa.NG, c0 = pa.c0, wcols = pa.w;
    const double* ca = pa.a + (size_t)th * Jt;
    const double* cb = pa.b + (size_t)th * Jt;
    const double* cc = pa.c + (size_t)th * Jt;
    const double* cd = pa.d + (size_t)th * Jt;
    const double* Ws = pa.W + (size_t)th * pa.N * RPL;
    const double* pts = pa.pt + (size_t)th * M * 2 * R;
    double* out = pa.out + (size_t)th * wcols * pa.ldo;
    double* up = pa.up ? pa.up + (size_t)th * c0 * wcols : nullptr;

    // this CTA's columns: the last group first, as the walk of column x′ is as long as the part of G up to x′.  Longest first,
    // a greedy schedule of the 625 CTAs of a one-set launch at N = M = 1e4 on 296 CTA slots ends at 1.05× the mean load per
    // slot; in column order at 1.5×.
    const int64_t cfirst = c0 + (int64_t)(gridDim.x - 1 - blockIdx.x) * nw;
    const int64_t clast = (cfirst + nw < c0 + wcols ? cfirst + nw : c0 + wcols) - 1;
    const int64_t col = cfirst + (tid >> 5);                               // this warp's column
    const bool active = col <= clast;
    const int64_t kstart = active ? pa.gpos[col] : -1;                     // where this warp joins the walk
    const int64_t ktop = pa.gpos[clast];

    for (int k = tid; k < PC_CH * LD; k += nthr) {   // rows ≥ R stay zero
        (&tabP[0][0])[k] = 0.0; (&tabU[0][0])[k] = 0.0; (&tabX[0][0])[k] = 0.0;
    }
    __syncthreads();

    double wv[PT];
#pragma unroll
    for (int j = 0; j < PT; j++) wv[j] = 0.0;
    for (int64_t hi = ktop + 1; hi > 0; hi -= PC_CH) {
        const int64_t lo = hi - PC_CH > 0 ? hi - PC_CH : 0;
        const int ns = (int)(hi - lo);
        // φ^G between G_k and G_{k+1} (one exp per term), U(t_n) at data steps (celerite_solver.jl:51-64)
        for (int idx = tid; idx < ns * Jt; idx += nthr) {
            const int st = idx / Jt, m = idx - st * Jt;
            const int64_t k = lo + st;
            const double x = pa.gt[k];
            const double ph = k + 1 < NG ? exp(-cc[m] * (pa.gt[k + 1] - x)) : 0.0;
            const bool data = pa.gcode[k] >= 0;
            const int tr = pa.term_row[m];
            if (tr < 0) {
                const int r0 = -tr - 1;
                tabU[st][r0] = data ? ca[m] : 0.0; tabP[st][r0] = ph;
            } else {
                double si = 0.0, co = 0.0;
                if (data) sincos_large(cd[m] * x, &si, &co);
                tabU[st][tr] = ca[m] * co + cb[m] * si;       // celerite_solver.jl:60
                tabU[st][tr + 1] = ca[m] * si - cb[m] * co;   // celerite_solver.jl:59
                tabP[st][tr] = ph; tabP[st][tr + 1] = ph;
            }
        }
        // W_n at a data step, r(τ_m) at a prediction step
        for (int idx = tid; idx < ns * R; idx += nthr) {
            const int st = idx / R, r = idx - st * R;
            const int code = pa.gcode[lo + st];
            tabX[st][r] = code >= 0 ? Ws[(int64_t)code * RPL + r] : pts[(int64_t)(-code - 1) * 2 * R + r];
        }
        for (int st = tid; st < ns; st += nthr) tabC[st] = pa.gcode[lo + st];
        __syncthreads();
        if (active) {
            for (int st = ns - 1; st >= 0; st--) {
                const int64_t k = lo + st;
                if (k > kstart) continue;
                if (k == kstart) {
                    const double* w0 = pts + col * 2 * R + R;
#pragma unroll
                    for (int j = 0; j < PT; j++) wv[j] = lane + 32 * j < R ? w0[lane + 32 * j] : 0.0;
                } else {
#pragma unroll
                    for (int j = 0; j < PT; j++) wv[j] *= tabP[st][lane + 32 * j];
                }
                const int code = tabC[st];
                double part = 0.0;
#pragma unroll
                for (int j = 0; j < PT; j++) part = fma(tabX[st][lane + 32 * j], wv[j], part);
                part = warp_sum(part);
                if (code >= 0) {
#pragma unroll
                    for (int j = 0; j < PT; j++) wv[j] = fma(-tabU[st][lane + 32 * j], part, wv[j]);
                } else if (lane == 0) {
                    const int64_t m = -code - 1;   // m ≤ col
                    out[(col - c0) * pa.ldo + m] = -part;
                    if (m >= c0) out[(m - c0) * pa.ldo + col] = -part;
                    else up[m * wcols + (col - c0)] = -part;
                }
            }
        }
        __syncthreads();   // the tables are rebuilt for the next PC_CH steps
    }
}

}  // namespace pioran
