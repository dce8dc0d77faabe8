// grad.cuh — K5: gradient of the fused approx + celerite log-likelihood (forward mode, FP64, sm_100a).
//
// The reference gets ∇θ logℒ for HMC/NUTS by pushing ForwardDiff dual numbers through approx → ScalableGP → logpdf
// (test/test_likelihood.jl:24-43,55; examples/turing_distributed/single_pl.jl).  Here the same forward-mode rule is
// applied to the two kernels of the likelihood path:
//   approx_grad_kernel     (K1 on duals)  θ → row amplitudes and Σa with their derivative along one θ-direction.  On the
//                          approx path c_j, d_j depend on the spectral grid only (src/psd.jl:250,266-267), so the series
//                          table (cos/sin/exp) carries no tangent: only amp, Σa, ν and μ do.
//   celerite_grad_kernel   (K2 on duals, block sizes ≤ 5)  one WARP per (parameter vector, θ-direction): the celerite_step
//                          recursion of celerite.cuh (non-pre-decayed form) with every θ-dependent quantity a (value, tangent) pair.
//                          Per stored entry 4 FP64 issues for the value + 5 for the tangent.  Same lane → block mapping,
//                          same TMA-staged shared series table, same reductions (on pairs).
// Directions k = 0 … n_psd_par−1: PSD parameters; k = n_psd_par: ν.  ∂/∂μ needs no block tangent (μ moves only the right-hand
// side): every warp carries it as two extra vector entries, the k = 0 warp reports it.  ∂/∂norm needs no sweep at all: K is
// homogeneous of degree 1 in (norm, ν), so norm ∂logL/∂norm + ν ∂logL/∂ν = ½ yᵀK⁻¹y − N/2, and the ν warp reports both.
#pragma once
#include "approx.cuh"
#include "celerite.cuh"

namespace pioran {

struct D2 { double v, d; };
__device__ __forceinline__ D2 mk2(double v, double d) { D2 r; r.v = v; r.d = d; return r; }
__device__ __forceinline__ D2 operator+(D2 a, D2 b) { return mk2(a.v + b.v, a.d + b.d); }
__device__ __forceinline__ D2 operator-(D2 a, D2 b) { return mk2(a.v - b.v, a.d - b.d); }
__device__ __forceinline__ D2 operator*(D2 a, D2 b) { return mk2(a.v * b.v, fma(a.d, b.v, a.v * b.d)); }
__device__ __forceinline__ D2 operator*(double c, D2 a) { return mk2(c * a.v, c * a.d); }
// c·x + y with a constant c
__device__ __forceinline__ D2 fmac(double c, D2 x, D2 y) { return mk2(fma(c, x.v, y.v), fma(c, x.d, y.d)); }
// a·b + c on pairs
__device__ __forceinline__ D2 fma2(D2 a, D2 b, D2 c) { return mk2(fma(a.v, b.v, c.v), fma(a.d, b.v, fma(a.v, b.d, c.d))); }
__device__ __forceinline__ D2 sel2(bool p, D2 a, D2 b) { return mk2(p ? a.v : b.v, p ? a.d : b.d); }
__device__ __forceinline__ D2 shfl2(D2 a, int src) { return mk2(__shfl_sync(FULL, a.v, src), __shfl_sync(FULL, a.d, src)); }
__device__ __forceinline__ D2 shflx2(D2 a, int m) { return mk2(__shfl_xor_sync(FULL, a.v, m), __shfl_xor_sync(FULL, a.d, m)); }
__device__ __forceinline__ D2 div2(D2 a, D2 b) { const double q = a.v / b.v; return mk2(q, (a.d - q * b.d) / b.v); }
// x^e, both pairs:  d = x^e (e' ln x + e x'/x)
__device__ __forceinline__ D2 pow2(D2 x, D2 e) {
    const double p = pow(x.v, e.v);
    return mk2(p, p * (e.d * log(x.v) + e.v * x.d / x.v));
}

// Tonari closed forms (test/test_psd.jl:6,12) on pairs; p: PSD parameters with the tangent of direction k.
__device__ __forceinline__ D2 psd_eval2(int model, const D2* p, double f) {
    const D2 one = mk2(1.0, 0.0);
    const D2 x = div2(mk2(f, 0.0), p[1]);
    D2 v = div2(pow2(x, mk2(-p[0].v, -p[0].d)), one + pow2(x, p[2] - p[0]));
    if (model == 1) v = div2(v, one + pow2(div2(mk2(f, 0.0), p[3]), p[4] - p[2]));
    return v;
}

// One thread per (parameter vector i, PSD-parameter direction k < n_psd_par).  theta: [B × tstride].
//   amp_rows [B × RP], suma [B]                     (written by the k = 0 thread; same values as approx_kernel)
//   damp_rows [B × ND × RP], dsuma [B × ND]         ND = n_psd_par
__global__ void approx_grad_kernel(const ApproxPlan* __restrict__ plan, int B, const double* __restrict__ theta,
                                   int tstride, double* __restrict__ amp_rows, double* __restrict__ damp_rows, int RP,
                                   double* __restrict__ suma, double* __restrict__ dsuma) {
    const ApproxPlan& P = *plan;
    const int ND = P.n_psd_par;         // the norm direction needs no sweep (celerite_grad_kernel uses the scaling identity)
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= B * ND) return;
    const int i = gid / ND, k = gid - i * ND;
    const int J = P.J;
    const double* th = theta + (size_t)i * tstride;
    D2 par[8];
    for (int q = 0; q < P.n_psd_par; q++) par[q] = mk2(th[q], q == k ? 1.0 : 0.0);
    const D2 norm = mk2(th[P.n_psd_par], 0.0);
    double x[MAXJ], dx[MAXJ];
    {   // get_normalised_psd (src/psd.jl:52-56)
        const D2 p0 = psd_eval2(P.model, par, P.fj[0]);
        for (int j = 0; j < J; j++) {
            const D2 r = div2(psd_eval2(P.model, par, P.fj[j]), p0);
            x[j] = r.v; dx[j] = r.d;
        }
    }
    // amplitudes = B \ p (src/psd.jl:109-112): the solve is linear, so the tangent goes through the same LU
    for (int kk = 0; kk < J; kk++) {
        const int pk = P.piv[kk];
        if (pk != kk) {
            double tmp = x[kk]; x[kk] = x[pk]; x[pk] = tmp;
            tmp = dx[kk]; dx[kk] = dx[pk]; dx[pk] = tmp;
        }
    }
    for (int kk = 0; kk < J; kk++) {
        const double xk = x[kk], dxk = dx[kk];
        for (int r = kk + 1; r < J; r++) { const double l = P.lu[r + kk * J]; x[r] -= l * xk; dx[r] -= l * dxk; }
    }
    for (int kk = J - 1; kk >= 0; kk--) {
        const double u = P.lu[kk + kk * J];
        x[kk] /= u; dx[kk] /= u;
        const double xk = x[kk], dxk = dx[kk];
        for (int r = 0; r < kk; r++) { const double l = P.lu[r + kk * J]; x[r] -= l * xk; dx[r] -= l * dxk; }
    }
    // normalisation (src/psd.jl:236-238, 375-395): linear in the amplitudes
    D2 integ;
    if (P.is_integrated_power) {
        integ.v = basis_integral(P.basis, J, x, P.fj, P.f_max) - basis_integral(P.basis, J, x, P.fj, P.f_min);
        integ.d = basis_integral(P.basis, J, dx, P.fj, P.f_max) - basis_integral(P.basis, J, dx, P.fj, P.f_min);
    } else {
        double s = 0.0, ds = 0.0;
        for (int j = 0; j < J; j++) { s += x[j] * P.fj[j]; ds += dx[j] * P.fj[j]; }
        const double cst = (P.basis == 0) ? 3.141592653589793 / 1.4142135623730951 : 2.0 * 3.141592653589793 / 3.0;
        integ = mk2(s * cst, ds * cst);
    }
    const D2 scale = div2(norm, integ);
    const double PI = 3.141592653589793, S2 = 1.4142135623730951;
    const double cst = (P.basis == 0) ? PI / S2 : PI / 3.0;
    double sa = 0.0, dsa = 0.0;
    double* ar = amp_rows + (size_t)i * RP;
    double* dr = damp_rows + ((size_t)i * ND + k) * RP;
    for (int j = 0; j < J; j++) {
        const D2 aj = cst * (P.fj[j] * (mk2(x[j], dx[j]) * scale));
        sa += aj.v; dsa += aj.d;
        dr[2 * j] = aj.d; dr[2 * j + 1] = aj.d;
        if (P.basis != 0) dr[2 * J + j] = aj.d;
        if (k == 0) {
            ar[2 * j] = aj.v; ar[2 * j + 1] = aj.v;
            if (P.basis != 0) ar[2 * J + j] = aj.v;
        }
    }
    const int Rl = (P.basis == 0) ? 2 * J : 3 * J;
    for (int r = Rl; r < RP; r++) { dr[r] = 0.0; if (k == 0) ar[r] = 0.0; }
    if (P.basis != 0) { sa += sa; dsa += dsa; }        // 2J terms: the celerite parts and the DRW parts (src/psd.jl:264-275)
    dsuma[(size_t)i * ND + k] = dsa;
    if (k == 0) suma[i] = sa;
}

// ------------------------------------------------------------------------------------------------ K2 on pairs
// Block sizes ≤ 5 only: 2·BS² doubles per lane fit the register file next to the step's operands.  Larger blocks go through
// grad_pipe.cuh (the value recursion once per parameter vector, tangent-only warps).
template <int BS>
struct LaneStateD {
    double Mv[BS][BS];
    double Md[BS][BS];
    D2 sjj[2], g[2], amp[2];
    D2 chi2;
    double logacc, dkeep, dfirst, dlog;     // Σ log|D_n| (ring as in LaneState) and its tangent Σ D'_n / D_n
    double gmu[2], chimu;                   // ∂/∂μ of g and of Σ z²/D: μ moves only the right-hand side (no block tangent), so
                                            // every warp carries it as two vector entries and the k = 0 warp reports it
};

template <int BS>
__device__ __forceinline__ void load_slice2(D2 (&dst)[BS], const double* __restrict__ pv, const double* __restrict__ pd) {
    double a[BS], b[BS];
    load_slice<BS>(a, pv);
    load_slice<BS>(b, pd);
#pragma unroll
    for (int r = 0; r < BS; r++) dst[r] = mk2(a[r], b[r]);
}

// One step on pairs — the structure of celerite_step<BS, ODD, /*PRE=*/false> (celerite.cuh), line by line.
//   sv, sd : per-warp scratch, values and tangents: q at [0, RPS), w at [RPS, 2·RPS)
template <int BS, bool ODD>
__device__ __forceinline__ void celerite_step_dual(LaneStateD<BS>& st, const double* __restrict__ T, double* __restrict__ sv,
                                                   double* __restrict__ sd, const LaneMap& lm, const double yn,
                                                   const double s2n, const D2 suma, const D2 mu, const D2 nu,
                                                   const int64_t n, const int lane) {
    constexpr int RP = rps_of(BS);
    const int o = lm.o;
    const D2 zero = mk2(0.0, 0.0);
    D2 qrow[BS];
    double urow[BS], xrow[BS], prow[BS];
    load_slice2<BS>(qrow, sv + lm.rowI, sd + lm.rowI);
    load_slice<BS>(urow, T + (ODD ? F_UH : F_UT) * RP + lm.rowI);
    load_slice<BS>(xrow, T + (ODD ? F_PHI : F_KAP) * RP + lm.rowI);
    if (!ODD) load_slice<BS>(prow, T + F_PHI * RP + lm.rowI);
    D2 rowpart[BS], acc[BS];
#pragma unroll
    for (int r = 0; r < BS; r++) rowpart[r] = zero;

    const double* wv = sv + RP;
    const double* wd = sd + RP;
    const double* uAp = T + (ODD ? F_UT : F_UH) * RP + lm.colA;
    const double* uBp = T + (ODD ? F_UT : F_UH) * RP + lm.colB;
    const double* zAp = T + F_KAP * RP + lm.colA;
    const double* zBp = T + F_KAP * RP + lm.colB;
#pragma unroll
    for (int c = 0; c < BS; c++) {
        const D2 wA = mk2(wv[lm.colA + c], wd[lm.colA + c]), wB = mk2(wv[lm.colB + c], wd[lm.colB + c]);
        const double uA = uAp[c], uB = uBp[c];
        const double zA = ODD ? zAp[c] : 0.0, zB = ODD ? zBp[c] : 0.0;
        D2 cA = zero, cB = zero;
#pragma unroll
        for (int r = 0; r < BS; r++) {
            const bool useA = r > c;  // compile-time after unrolling
            const D2 w = useA ? wA : wB;
            const double u = useA ? uA : uB;
            const D2 qr = (r == c) ? sel2(lm.dzero, zero, qrow[r]) : qrow[r];
            const D2 m = fmac(ODD ? (useA ? zA : zB) : xrow[r], mk2(st.Mv[r][c], st.Md[r][c]), qr * w);
            st.Mv[r][c] = m.v;
            st.Md[r][c] = m.d;
            rowpart[r] = fmac(u, m, rowpart[r]);
            if (useA) cA = fmac(urow[r], m, cA);
            else      cB = fmac(urow[r], m, cB);
        }
        const D2 yv = shfl2(cB + sel2(o != 0, cA, zero), lm.src_lane);
        acc[c] = yv + sel2(o != 0, zero, cA);
    }

    const double ut0 = T[F_UT * RP + lm.j0], ut1 = T[F_UT * RP + lm.j1];
    D2 sblk = zero;
#pragma unroll
    for (int r = 0; r < BS; r++) sblk = fmac(urow[r], rowpart[r], sblk);
    D2 spart = fmac(ut1 * ut1, st.sjj[1], fmac(ut0 * ut0, st.sjj[0], sblk + sblk));
    D2 upart = fmac(ut1, st.g[1], ut0 * st.g[0]);
    double umu = fma(ut1, st.gmu[1], ut0 * st.gmu[0]);
#pragma unroll
    for (int sft = 16; sft >= 1; sft >>= 1) {
        spart = spart + shflx2(spart, sft);
        upart = upart + shflx2(upart, sft);
        umu += __shfl_xor_sync(FULL, umu, sft);
    }

    // matvec reduction: reduce-scatter of the BS row sums over the 4 lanes of the block-row
    D2 tot[BS];
#pragma unroll
    for (int c = 0; c < BS; c++) {
        if (ODD) tot[c] = fmac(xrow[c], rowpart[c], acc[c]);
        else     tot[c] = fmac(prow[c], acc[c], rowpart[c]);
    }
    const bool bit0 = (o & 1) != 0, bit1 = (o & 2) != 0;
    D2 e[4];
#pragma unroll
    for (int m = 0; m < 4; m++) {
        if (2 * m < BS) {
            const D2 lo = tot[(2 * m < BS) ? 2 * m : 0];
            const D2 hi = (2 * m + 1 < BS) ? tot[(2 * m + 1 < BS) ? 2 * m + 1 : 0] : zero;
            const D2 recv = shflx2(sel2(bit0, lo, hi), 1);
            e[m] = sel2(bit0, hi, lo) + recv;
        } else {
            e[m] = zero;
        }
    }
    D2 f0, f1 = zero;
    {
        const D2 recv = shflx2(sel2(bit1, e[0], e[1]), 2);
        f0 = sel2(bit1, e[1], e[0]) + recv;
    }
    if (BS > 4) {
        const D2 recv = shflx2(sel2(bit1, e[2], e[3]), 2);
        f1 = sel2(bit1, e[3], e[2]) + recv;
    }

    // owner phase: rows j0 (and j1)
    const double v0 = T[F_V * RP + lm.j0], v1 = T[F_V * RP + lm.j1];
    const double pn0 = T[F_PHN * RP + lm.j0], pn1 = T[F_PHN * RP + lm.j1];
    const D2 p0 = fmac(ut0, st.sjj[0], f0);
    const D2 p1 = fmac(ut1, st.sjj[1], f1);
    const D2 An = fmac(s2n, nu, suma);
    const D2 D = An - spart;                       // celerite_solver.jl:92
    D2 rD;
    rD.v = fast_rcp(D.v);
    rD.d = -D.d * rD.v * rD.v;
    const D2 z = mk2((yn - mu.v) - upart.v, -mu.d - upart.d);   // celerite_solver.jl:141
    st.chi2 = fma2(z * z, rD, st.chi2);
    const double dzmu = -1.0 - umu;                             // ∂z_n/∂μ
    st.chimu = fma(2.0 * z.v * dzmu, rD.v, st.chimu);
    if (n == 0) st.dfirst = D.v;
    else if ((int)(n & 31) == lane) st.dkeep = D.v;
    if ((n & 31) == 31) { st.logacc += log(fabs(st.dkeep)); st.dkeep = 1.0; }
    st.dlog = fma(D.d, rD.v, st.dlog);

    const D2 q0 = fmac(v0, st.amp[0], mk2(-p0.v, -p0.d)), q1 = fmac(v1, st.amp[1], mk2(-p1.v, -p1.d));
    const D2 w0 = q0 * rD, w1 = q1 * rD;
    st.g[0] = pn0 * fma2(w0, z, st.g[0]);
    st.g[1] = pn1 * fma2(w1, z, st.g[1]);
    st.gmu[0] = pn0 * fma(w0.v, dzmu, st.gmu[0]);
    st.gmu[1] = pn1 * fma(w1.v, dzmu, st.gmu[1]);
    st.sjj[0] = (pn0 * pn0) * fma2(q0, w0, st.sjj[0]);   // celerite_solver.jl:85
    st.sjj[1] = (pn1 * pn1) * fma2(q1, w1, st.sjj[1]);
    __syncwarp();
    // the NEXT step is odd iff this one is even: odd steps consume (q, φ∘w), even steps (φ∘q, w)
    const D2 qo0 = ODD ? pn0 * q0 : q0, wo0 = ODD ? w0 : pn0 * w0;
    const D2 qo1 = ODD ? pn1 * q1 : q1, wo1 = ODD ? w1 : pn1 * w1;
    sv[lm.j0] = qo0.v; sd[lm.j0] = qo0.d; sv[RP + lm.j0] = wo0.v; sd[RP + lm.j0] = wo0.d;
    if (lm.valid1) { sv[lm.j1] = qo1.v; sd[lm.j1] = qo1.d; sv[RP + lm.j1] = wo1.v; sd[RP + lm.j1] = wo1.d; }
    __syncwarp();
}

struct GradArgs {
    const WorkItem* work;       // items over the virtual batch e = θ·(ND+1) + k (theta_begin, count, out_begin in that index space)
    const double* amp;          // [nθ × RP] (logical rows)
    const double* damp;         // [nθ × ND × RP]
    const double* suma;         // [nθ]
    const double* dsuma;        // [nθ × ND]
    const double* theta;        // [nθ × pstride]; norm at column ND, ν at ND + 1, μ at ND + 2
    int pstride;
    int ND;                     // n_psd_par; ND + 1 warps (directions psd…, ν) and ND + 3 outputs per θ
    double* logl;               // [nθ] or nullptr
    double* grad;               // [nθ × P]
    // blocked_grad.cuh only — log-normal series (docs/src/ultranest.md:197-217): per-θ data yn = log(y − c), σ² = σ²/(y − c)² and one
    // more direction, c, after ν (its tangents ∂yn/∂c = −e^{−yn}, ∂σ²/∂c = 2 σ² e^{−yn} are formed from the transformed data)
    const double* y_batch;      // [nθ × ystride] or nullptr
    const double* s2_batch;
    int64_t ystride;
    int cdir;                   // 1: directions psd…, ν, c and ND + 4 outputs per θ (…, norm, ν, μ, c)
};

// grid = work items; block = NW warps; each warp one (θ, direction).  Shared memory: 2 TMA stages of the series table |
// NW × 4·RPS scratch | 2 mbarriers | 2 stage counters (as celerite_shared_kernel).
template <int BS, int NW>
constexpr size_t grad_smem_bytes() {
    return sizeof(double) * (2 * (size_t)CHUNK_STEPS * table_step_doubles(rps_of(BS)) + (size_t)NW * 4 * rps_of(BS)) +
           2 * sizeof(uint64_t) + 16;
}
template <int BS, int NW>
__global__ void __launch_bounds__(NW * 32, 1) celerite_grad_kernel(const GradArgs args) {
    static_assert(BS <= 5, "block sizes >= 6: grad_pipe.cuh");
    constexpr int CS = CHUNK_STEPS;
    constexpr int RP = G * BS, RPS = rps_of(BS), SD = table_step_doubles(RPS), STAGE = CS * SD;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* stages = reinterpret_cast<double*>(smem_raw);
    double* scratch = stages + 2 * STAGE;
    uint64_t* bars = reinterpret_cast<uint64_t*>(scratch + NW * 4 * RPS);
    int* done = reinterpret_cast<int*>(bars + 2);

    const WorkItem wk = args.work[blockIdx.x];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t N = wk.N;
    const int64_t nchunks = (N + CS - 1) / CS;
    constexpr uint32_t STAGE_BYTES = STAGE * sizeof(double);

    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        done[0] = done[1] = 0;
        fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 0; k < 2 && k < nchunks; k++) {
            mbar_arrive_expect_tx(&bars[k], STAGE_BYTES);
            tma_load_1d(stages + k * STAGE, wk.table + (size_t)k * STAGE, STAGE_BYTES, &bars[k]);
        }
    }

    const bool active = warp < wk.count;
    const int e = wk.theta_begin + (active ? warp : wk.count - 1);
    const int P = args.ND + 3;          // outputs per parameter vector: psd parameters…, norm, ν, μ
    const int PW = args.ND + 1;         // warps per parameter vector: psd parameters…, ν.  ∂/∂μ rides along (LaneStateD::gmu) and
                                        // ∂/∂norm follows from ∂/∂ν: K = norm·K̂ + ν·Σ is homogeneous of degree 1 in (norm, ν), so
                                        // norm ∂logL/∂norm + ν ∂logL/∂ν = ½ yᵀK⁻¹y − N/2 (Euler)
    const int th = e / PW, k = e - th * PW;
    const LaneMap lm = make_lane_map<BS>(lane);
    const int i = lane >> 2, o = lane & 3;

    LaneStateD<BS> st;
    const D2 zero = mk2(0.0, 0.0);
#pragma unroll
    for (int r = 0; r < BS; r++)
#pragma unroll
        for (int c = 0; c < BS; c++) { st.Mv[r][c] = 0.0; st.Md[r][c] = 0.0; }
    st.sjj[0] = st.sjj[1] = st.g[0] = st.g[1] = zero;
    st.chi2 = zero; st.logacc = 0.0; st.dkeep = 1.0; st.dfirst = 1.0; st.dlog = 0.0;
    st.gmu[0] = st.gmu[1] = 0.0; st.chimu = 0.0;
    const bool amp_dir = k < args.ND;
    const double* av = args.amp + (size_t)th * RP;
    const double* ad = args.damp + ((size_t)th * args.ND + (amp_dir ? k : 0)) * RP;
    st.amp[0] = mk2(av[i * BS + o], amp_dir ? ad[i * BS + o] : 0.0);
    st.amp[1] = lm.valid1 ? mk2(av[i * BS + o + 4], amp_dir ? ad[i * BS + o + 4] : 0.0) : zero;
    const D2 suma = mk2(args.suma[th], amp_dir ? args.dsuma[(size_t)th * args.ND + k] : 0.0);
    const double* trow = args.theta + (size_t)th * args.pstride;
    const D2 nu = mk2(trow[args.ND + 1], k == args.ND ? 1.0 : 0.0);
    const D2 mu = mk2(trow[args.ND + 2], 0.0);

    double* sv = scratch + warp * 4 * RPS;
    double* sd = sv + 2 * RPS;
    for (int q = lane; q < 4 * RPS; q += 32) sv[q] = 0.0;
    __syncwarp();

    for (int64_t kc = 0; kc < nchunks; kc++) {
        const int sidx = (int)(kc & 1);
        mbar_wait(&bars[sidx], (uint32_t)((kc >> 1) & 1));
        const double* stage = stages + sidx * STAGE;
        const int64_t nbeg = kc * CS;
        const int nsteps = (int)((N - nbeg) < CS ? (N - nbeg) : CS);
        for (int s = 0; s < nsteps; s += 2) {
            const double* T0 = stage + s * SD;
            const double* T1 = T0 + SD;
            const int64_t n = nbeg + s;
            celerite_step_dual<BS, false>(st, T0, sv, sd, lm, T0[6 * RPS + 0], T0[6 * RPS + 1], suma, mu, nu, n, lane);
            if (s + 1 < nsteps)
                celerite_step_dual<BS, true>(st, T1, sv, sd, lm, T1[6 * RPS + 0], T1[6 * RPS + 1], suma, mu, nu, n + 1, lane);
        }
        __syncwarp();
        if (lane == 0 && kc + 2 < nchunks) {
            __threadfence_block();
            if (atomicAdd(&done[sidx], 1) == NW - 1) {
                done[sidx] = 0;
                fence_proxy_async();
                mbar_arrive_expect_tx(&bars[sidx], STAGE_BYTES);
                tma_load_1d(stages + sidx * STAGE, wk.table + (size_t)(kc + 2) * STAGE, STAGE_BYTES, &bars[sidx]);
            }
        }
    }
    // Σ log|D_n| (log D_1 without abs, celerite_solver.jl:126) and logL (celerite_solver.jl:333) with their tangents
    double la = st.logacc + log(fabs(st.dkeep));
#pragma unroll
    for (int sft = 16; sft >= 1; sft >>= 1) la += __shfl_xor_sync(FULL, la, sft);
    const double logdet = log(st.dfirst) + la;
    if (active && lane == 0) {
        if (k == 0 && args.logl) args.logl[th] = -logdet / 2 - (double)N * 1.8378770664093453 / 2 - st.chi2.v / 2;
        const double gk = -st.dlog / 2 - st.chi2.d / 2;
        if (k < args.ND) {
            args.grad[(size_t)th * P + k] = gk;
        } else {      // the ν warp also reports ∂/∂norm
            args.grad[(size_t)th * P + args.ND + 1] = gk;
            args.grad[(size_t)th * P + args.ND] = (0.5 * st.chi2.v - 0.5 * (double)N - nu.v * gk) / trow[args.ND];
        }
        if (k == 0) args.grad[(size_t)th * P + args.ND + 2] = -st.chimu / 2;
    }
}

// ------------------------------------------------------------------------------------------------ K1 on pairs with PSD features
// Gradient of pioran_approx_features_logl: the feature branch of approx_kernel (src/psd.jl:15-44, 229-243) on pairs, one thread
// per (parameter vector i, θ-direction k), k over every column of the θ row [psd parameters…, norm, ν, μ, (S₀, f₀, Q)…].  Unlike
// approx_grad_kernel, c and d of the feature terms depend on θ (f₀, Q), so the output is the full coefficient set (a, b, c, d)
// with its tangent, written straight into the layout of celerite_jvp_kernel (jvp.cuh): the sweep that follows is the JVP with
// P = tstride directions.  The coupling runs both ways: the continuum parameters move the feature amplitudes (division by the
// PSD at the first grid point, and the normalisation integral), the feature parameters move the continuum amplitudes through
// the normalisation when it is the integrated power.  norm is one more direction (every amplitude is ∝ norm, so da = a/norm);
// ν and μ carry no coefficient tangent and enter as dν = 1, dμ = 1.
__device__ __forceinline__ D2 sqrt2d(D2 x) { const double r = sqrt(x.v); return mk2(r, 0.5 * x.d / r); }
__device__ __forceinline__ D2 atan2d(D2 y, D2 x) {
    return mk2(atan2(y.v, x.v), (x.v * y.d - y.v * x.d) / (x.v * x.v + y.v * y.v));
}
// integral_celerite (approx.cuh) on pairs
__device__ __forceinline__ D2 integral_celerite2(D2 a, D2 b, D2 c, D2 d, double x) {
    const double TWO_PI = 6.283185307179586;
    const D2 dp = d + mk2(TWO_PI * x, 0.0), dm = d - mk2(TWO_PI * x, 0.0);
    const D2 num = c * c + dp * dp, den = c * c + dm * dm;
    const D2 r = div2(num, den);
    const D2 lg = mk2(log(r.v), r.d / r.v);
    return (1.0 / TWO_PI) * (2.0 * (a * (atan2d(c, dm) - atan2d(c, dp))) + b * lg);
}

// theta [B × tstride]; nfeat features at columns feat_off + 3f (S₀, f₀, Q); norm at n_psd_par, ν, μ at n_psd_par + 1, + 2.
// Outputs (P = tstride directions, Jt = continuum terms + nfeat):
//   a, b, c, d [B × Jt], mu, nu [B]                      written by the k = 0 thread
//   da, db, dc, dd [B × P × Jt], dmu, dnu [B × P]
__global__ void approx_features_grad_kernel(const ApproxPlan* __restrict__ plan, int B, const double* __restrict__ theta,
                                            int tstride, int nfeat, int feat_off, double* __restrict__ a, double* __restrict__ b,
                                            double* __restrict__ c, double* __restrict__ d, double* __restrict__ mu,
                                            double* __restrict__ nu, double* __restrict__ da, double* __restrict__ db,
                                            double* __restrict__ dc, double* __restrict__ dd, double* __restrict__ dmu,
                                            double* __restrict__ dnu) {
    const ApproxPlan& P = *plan;
    const int ND = tstride, npar = P.n_psd_par;
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= B * ND) return;
    const int i = gid / ND, k = gid - i * ND;
    const int J = P.J;
    const double* th = theta + (size_t)i * tstride;
    D2 par[8];
    for (int q = 0; q < npar; q++) par[q] = mk2(th[q], q == k ? 1.0 : 0.0);
    const D2 norm = mk2(th[npar], k == npar ? 1.0 : 0.0);
    double x[MAXJ], dx[MAXJ];
    // get_normalised_psd (src/psd.jl:52-56)
    const D2 p0 = psd_eval2(P.model, par, P.fj[0]);
    for (int j = 0; j < J; j++) {
        const D2 r = div2(psd_eval2(P.model, par, P.fj[j]), p0);
        x[j] = r.v; dx[j] = r.d;
    }
    // amplitudes = B \ p (src/psd.jl:109-112), value and tangent through the same LU
    for (int kk = 0; kk < J; kk++) {
        const int pk = P.piv[kk];
        if (pk != kk) {
            double tmp = x[kk]; x[kk] = x[pk]; x[pk] = tmp;
            tmp = dx[kk]; dx[kk] = dx[pk]; dx[pk] = tmp;
        }
    }
    for (int kk = 0; kk < J; kk++) {
        const double xk = x[kk], dxk = dx[kk];
        for (int r = kk + 1; r < J; r++) { const double l = P.lu[r + kk * J]; x[r] -= l * xk; dx[r] -= l * dxk; }
    }
    for (int kk = J - 1; kk >= 0; kk--) {
        const double u = P.lu[kk + kk * J];
        x[kk] /= u; dx[kk] /= u;
        const double xk = x[kk], dxk = dx[kk];
        for (int r = 0; r < kk; r++) { const double l = P.lu[r + kk * J]; x[r] -= l * xk; dx[r] -= l * dxk; }
    }
    // normalisation (src/psd.jl:236-238, 375-395): linear in the amplitudes
    D2 integ;
    if (P.is_integrated_power) {
        integ.v = basis_integral(P.basis, J, x, P.fj, P.f_max) - basis_integral(P.basis, J, x, P.fj, P.f_min);
        integ.d = basis_integral(P.basis, J, dx, P.fj, P.f_max) - basis_integral(P.basis, J, dx, P.fj, P.f_min);
    } else {
        double s = 0.0, ds = 0.0;
        for (int j = 0; j < J; j++) { s += x[j] * P.fj[j]; ds += dx[j] * P.fj[j]; }
        const double cst = (P.basis == 0) ? 3.141592653589793 / 1.4142135623730951 : 2.0 * 3.141592653589793 / 3.0;
        integ = mk2(s * cst, ds * cst);
    }
    // features: convert_feature (src/psd.jl:15-28), amplitudes divided by the continuum's PSD at the first grid point
    D2 fa[MAXFEAT], fb[MAXFEAT], fc[MAXFEAT], fd[MAXFEAT];
    for (int f = 0; f < nfeat; f++) {
        const int col = feat_off + 3 * f;
        const D2 S0 = mk2(th[col], k == col ? 1.0 : 0.0);
        const D2 f0q = mk2(th[col + 1], k == col + 1 ? 1.0 : 0.0);
        const D2 Q = mk2(th[col + 2], k == col + 2 ? 1.0 : 0.0);
        const D2 dl = sqrt2d(4.0 * (Q * Q) - mk2(1.0, 0.0));
        const D2 w0 = 6.283185307179586 * f0q;
        const D2 ak = 0.25 * (S0 * w0 * Q);
        fa[f] = div2(ak, p0); fb[f] = div2(div2(ak, dl), p0);
        fc[f] = 0.5 * div2(w0, Q); fd[f] = fc[f] * dl;
        if (P.is_integrated_power)
            integ = integ + (integral_celerite2(fa[f], fb[f], fc[f], fd[f], P.f_max) - integral_celerite2(fa[f], fb[f], fc[f], fd[f], P.f_min));
    }
    const D2 scale = div2(norm, integ);
    const int Jc = P.basis == 0 ? J : 2 * J, Jt = Jc + nfeat;
    const size_t ro = (size_t)i * Jt, to = ((size_t)i * ND + k) * Jt;
    const bool v = k == 0;
    const double PI = 3.141592653589793, S2 = 1.4142135623730951, S3 = 1.7320508075688772;
    for (int j = 0; j < J; j++) {
        if (P.basis == 0) {   // SHO: a = b = A f π/√2, c = d = √2 π f   (src/psd.jl:249-252)
            const D2 aj = (PI / S2) * (P.fj[j] * (mk2(x[j], dx[j]) * scale));
            const double cj = S2 * PI * P.fj[j];
            if (v) { a[ro + j] = aj.v; b[ro + j] = aj.v; c[ro + j] = cj; d[ro + j] = cj; }
            da[to + j] = aj.d; db[to + j] = aj.d; dc[to + j] = 0.0; dd[to + j] = 0.0;
        } else {              // DRWCelerite: (a, √3a, πf, √3πf) ++ (a, 0, 2πf, 0)   (src/psd.jl:264-275)
            const D2 aj = (PI / 3.0) * (P.fj[j] * (mk2(x[j], dx[j]) * scale));
            const double cj = PI * P.fj[j];
            if (v) {
                a[ro + j] = aj.v; b[ro + j] = S3 * aj.v; c[ro + j] = cj; d[ro + j] = S3 * cj;
                a[ro + J + j] = aj.v; b[ro + J + j] = 0.0; c[ro + J + j] = 2.0 * cj; d[ro + J + j] = 0.0;
            }
            da[to + j] = aj.d; db[to + j] = S3 * aj.d; dc[to + j] = 0.0; dd[to + j] = 0.0;
            da[to + J + j] = aj.d; db[to + J + j] = 0.0; dc[to + J + j] = 0.0; dd[to + J + j] = 0.0;
        }
    }
    for (int f = 0; f < nfeat; f++) {                           // src/psd.jl:254-259, 277-282
        const D2 af = 2.0 * (fa[f] * scale), bf = 2.0 * (fb[f] * scale);
        if (v) { a[ro + Jc + f] = af.v; b[ro + Jc + f] = bf.v; c[ro + Jc + f] = fc[f].v; d[ro + Jc + f] = fd[f].v; }
        da[to + Jc + f] = af.d; db[to + Jc + f] = bf.d; dc[to + Jc + f] = fc[f].d; dd[to + Jc + f] = fd[f].d;
    }
    if (v) { nu[i] = th[npar + 1]; mu[i] = th[npar + 2]; }
    dnu[(size_t)i * ND + k] = k == npar + 1 ? 1.0 : 0.0;
    dmu[(size_t)i * ND + k] = k == npar + 2 ? 1.0 : 0.0;
}

}  // namespace pioran
