// blocked_grad.cuh — K5t: gradient of the fused approx + celerite log-likelihood on the FP64 tensor pipe (sm_100a).
//
// Forward mode, like the reference's ForwardDiff.gradient over logpdf (test/test_likelihood.jl:24-43, 55; the NUTS runs of
// examples/turing_distributed/single_pl.jl) and like K5 (grad.cuh), but pushed through the BLOCKED recursion of blocked.cuh, so
// that the tangent's O(R²) work is DMMA as well.  On the approx path the table (Û, V̂, ψ8, H) carries no tangent: only the row
// amplitudes, Σa and ν do.  With a dot for the derivative along one direction, E = L⁻¹ and rd = 1/D of the value sweep:
//     Ṗ0 = Ẋ·Û                       Ċ = K̇_blk − Ûᵀ·Ṗ0                      K̇_blk = Σ_j ȧmp_j H_j,  diagonal Σȧ + ν̇ σ²_s
//     M  = E Ċ Eᵀ                    Ḋ = diag M,   N = strictly-lower(M)·D⁻¹   (C = L D Lᵀ  ⇒  E Ċ Eᵀ = N D + Ḋ + D Nᵀ, N = E L̇)
//     Ė  = −N E                      Q̂̇ = Ḃm·Eᵀ + Bm·Ėᵀ,   Ḃm = ȧmp∘V̂ − ψ8∘Ṗ0   Ŵ̇ = Q̂̇ D⁻¹ − Q̂ Ḋ D⁻²
//     Ẋ  ← (ψ8ψ8ᵀ)∘Ẋ + Q̂̇·Ŵᵀ + Q̂·Ŵ̇ᵀ
//     ∂Σlog D = Σ_s Ḋ_s/D_s          ∂(yᵀK⁻¹y) = Σ_s (2 z_s ż_s/D_s − z_s² Ḋ_s/D_s²),   z = Q̂[RG], ż = Q̂̇[RG]
// (tests/tools/proto/blocked_grad_math.py is the numpy form of exactly this, checked against central differences.)
//
// Mapping.  One CTA per parameter vector: warp 0 runs the value sweep (blocked_step, PUB) and publishes E, 1/D, Bm, Q̂ of every
// block to a 2-slot ring in shared memory, lane for lane in the accumulator layout; warps 1 … n_psd_par + 1 carry one tangent
// state Ẋ each (directions: PSD parameters, ν) one block behind, one __syncthreads per block.  ∂/∂μ moves only the right-hand
// side: it is a SECOND data row of the value state (row RM, right-hand side −1), whose innovations are ż, at no extra product.
// ∂/∂norm follows from ∂/∂ν by the homogeneity of K in (norm, ν) (grad.cuh).  A sinusoidal mean (celerite_blocked_grad_sine_kernel)
// adds one MEAN WARP: A, ϕ and T₀ move only the right-hand side too, but by a different amount at every step and for every θ, so
// their three data rows get a row tile of their own instead of slots in the value state (blocked_mean_step).
#pragma once
#include "blocked.cuh"
#include "grad.cuh"

namespace pioran {

#ifndef PIORAN_BLKG_TWO_CTA_MAX_NT
#define PIORAN_BLKG_TWO_CTA_MAX_NT 5
#endif
__host__ __device__ constexpr int blk_slot_doubles(int NTR) { return (4 + 4 * NTR) * 32; }

// One block of the tangent recursion.  xd: tangent state tiles (I ≥ K); slot: what the value warp published for this block.
template <int NT, int NTR, bool HALF>
__device__ __forceinline__ void blocked_tangent_step(double (&xd)[NTR][NT][2], const double* __restrict__ tab,
                                                     const double* __restrict__ slot, const double* __restrict__ damp_s,
                                                     const double* __restrict__ damp_l, const BlkLane& L, const int lane,
                                                     const double dsuma, const double dnu, const int64_t n0, const int64_t N,
                                                     const int RG, double& dlog, double& dchi,
                                                     const double* __restrict__ yb = nullptr, const double* __restrict__ sb = nullptr,
                                                     const bool cdir = false, const double nu = 1.0) {
    constexpr int O_VH = blk_off_vh(NT, NTR), O_PSI = blk_off_psi(NT, NTR);
    const int g = L.g, t = L.t;

    // ---- K̇_blk.  Log-shift direction c: the diagonal moves with the data, ∂(ν σ²_n)/∂c = 2 ν σ²_n e^{−yn_n}, σ² the transformed one
    double cd0, cd1;
    {
        double dgc = 0.0;
        if (cdir) {
            const int64_t n = n0 + g;
            dgc = (n < N) ? 2.0 * nu * sb[n] * exp(-yb[n]) : 0.0;
        }
        blk_kblk<NT, NTR, true>(tab, damp_l, L, lane, dsuma, dnu, n0, N, sb, cd0, cd1, cdir, dgc);
    }

    // ---- Ṗ0 = Ẋ·Û
    double P0[NTR][2];
#pragma unroll
    for (int I = 0; I < NTR; I++) P0[I][0] = P0[I][1] = 0.0;
#pragma unroll
    for (int K = 0; K < NT; K++) {
        const double2 u = *reinterpret_cast<const double2*>(tab + K * 64 + g * 8 + 2 * t);
#pragma unroll
        for (int I = 0; I < NTR; I++) {
            double a0, a1;
            if (I >= K) { a0 = xd[I][K][0]; a1 = xd[I][K][1]; }
            else tile_transpose(L, xd[K][I][0], xd[K][I][1], a0, a1);
            dmma(P0[I][0], P0[I][1], a0, u.x);
            if (!(HALF && K == NT - 1)) dmma(P0[I][0], P0[I][1], a1, u.y);
        }
    }
    // ---- Ċ = K̇_blk − Ûᵀ·Ṗ0
    {
        double ca0 = 0.0, ca1 = 0.0, cb0 = 0.0, cb1 = 0.0;
#pragma unroll
        for (int J = 0; J < NT; J++) {
            const double2 u = *reinterpret_cast<const double2*>(tab + J * 64 + g * 8 + 2 * t);
            double p0, p1;
            tile_transpose(L, P0[J][0], P0[J][1], p0, p1);
            const bool both = !(HALF && J == NT - 1);
            if (J & 1) { dmma(cb0, cb1, u.x, p0); if (both) dmma(cb0, cb1, u.y, p1); }
            else       { dmma(ca0, ca1, u.x, p0); if (both) dmma(ca0, ca1, u.y, p1); }
        }
        cd0 -= ca0 + cb0;
        cd1 -= ca1 + cb1;
    }
    // ---- Ẋ ← (ψ8ψ8ᵀ)∘Ẋ
    double psr[NTR];
#pragma unroll
    for (int I = 0; I < NTR; I++) psr[I] = tab[O_PSI + 8 * I + g];
#pragma unroll
    for (int K = 0; K < NT; K++) {
        const double2 pc = *reinterpret_cast<const double2*>(tab + O_PSI + 8 * K + 2 * t);
#pragma unroll
        for (int I = K; I < NTR; I++) {
            xd[I][K][0] *= psr[I] * pc.x;
            xd[I][K][1] *= psr[I] * pc.y;
        }
    }
    // ---- Ḃm = ȧmp∘V̂ − ψ8∘Ṗ0 (the data rows have no amplitude tangent: their entries are −Ṗ0)
#pragma unroll
    for (int I = 0; I < NTR; I++) {
        const int row = 8 * I + g;
        double2 vh = *reinterpret_cast<const double2*>(tab + O_VH + row * 8 + 2 * t);
        double am = damp_s[row];
        if (I == NTR - 1 && cdir && row == RG) {      // ∂yn/∂c = −1/(y − c) = −e^{−yn}: the data row's right-hand side moves
            const int64_t n = n0 + 2 * t;
            vh.x = (n < N) ? -exp(-yb[n]) : 0.0;
            vh.y = (n + 1 < N) ? -exp(-yb[n + 1]) : 0.0;
            am = 1.0;
        }
        P0[I][0] = fma(-psr[I], P0[I][0], am * vh.x);
        P0[I][1] = fma(-psr[I], P0[I][1], am * vh.y);
    }

    // ---- the value sweep's factor of this block
    const double* sl = slot + lane;
    const double e0 = sl[0], e1 = sl[32], rd0 = sl[64], rd1 = sl[96];
    // M = E Ċ Eᵀ (Ċ symmetric: its accumulator registers serve as the B operand)
    double t0 = 0.0, t1 = 0.0, m0 = 0.0, m1 = 0.0;
    dmma(t0, t1, e0, cd0); dmma(t0, t1, e1, cd1);
    dmma(m0, m1, t0, e0);  dmma(m0, m1, t1, e1);
    // Ḋ of this lane's two steps (diagonal entry (s, s) sits on lane (s, s>>1), register s&1)
    const double dd0 = __shfl_sync(FULL, m0, 4 * (2 * t) + t), dd1 = __shfl_sync(FULL, m1, 4 * (2 * t + 1) + t);
    dlog += (L.cdiag0 ? m0 * rd0 : 0.0) + (L.cdiag1 ? m1 * rd1 : 0.0);
    // N = strictly-lower(M)·D⁻¹,  Ė = −N E  (E as the B operand: its transpose in the accumulator layout)
    const double n0v = (g > 2 * t) ? m0 * rd0 : 0.0, n1v = (g > 2 * t + 1) ? m1 * rd1 : 0.0;
    double et0, et1;
    tile_transpose(L, e0, e1, et0, et1);
    double ed0 = 0.0, ed1 = 0.0;
    dmma(ed0, ed1, n0v, et0); dmma(ed0, ed1, n1v, et1);
    ed0 = -ed0; ed1 = -ed1;

    // ---- Q̂̇ = Ḃm·Eᵀ + Bm·Ėᵀ
    double Qd[NTR][2];
#pragma unroll
    for (int I = 0; I < NTR; I++) {
        const double bm0 = sl[(4 + 2 * I) * 32], bm1 = sl[(5 + 2 * I) * 32];
        Qd[I][0] = Qd[I][1] = 0.0;
        dmma(Qd[I][0], Qd[I][1], P0[I][0], e0);
        dmma(Qd[I][0], Qd[I][1], P0[I][1], e1);
        dmma(Qd[I][0], Qd[I][1], bm0, ed0);
        dmma(Qd[I][0], Qd[I][1], bm1, ed1);
    }
    // Ŵ̇ = Q̂̇ D⁻¹ − Q̂ Ḋ D⁻² : factors of this lane's two steps
    const double f0 = dd0 * rd0 * rd0, f1 = dd1 * rd1 * rd1;
    // ---- ∂(yᵀK⁻¹y): z = Q̂[RG], ż = Q̂̇[RG]
    {
        const double z0 = sl[(4 + 2 * NTR + 2 * (NTR - 1)) * 32], z1 = sl[(5 + 2 * NTR + 2 * (NTR - 1)) * 32];
        const bool isrg = (8 * (NTR - 1) + g == RG);
        const double v = fma(z0, fma(2.0 * rd0, Qd[NTR - 1][0], -(z0 * f0)), z1 * fma(2.0 * rd1, Qd[NTR - 1][1], -(z1 * f1)));
        dchi += isrg ? v : 0.0;
    }
    // ---- Ẋ += Q̂̇·Ŵᵀ + Q̂·Ŵ̇ᵀ
#pragma unroll
    for (int K = 0; K < NT; K++) {
        const double qk0 = sl[(4 + 2 * NTR + 2 * K) * 32], qk1 = sl[(5 + 2 * NTR + 2 * K) * 32];
        const double w0 = qk0 * rd0, w1 = qk1 * rd1;
        const double wd0 = fma(Qd[K][0], rd0, -(qk0 * f0)), wd1 = fma(Qd[K][1], rd1, -(qk1 * f1));
#pragma unroll
        for (int I = K; I < NTR; I++) {
            const double qi0 = sl[(4 + 2 * NTR + 2 * I) * 32], qi1 = sl[(5 + 2 * NTR + 2 * I) * 32];
            double x0 = xd[I][K][0], x1 = xd[I][K][1];
            dmma(x0, x1, Qd[I][0], w0);
            dmma(x0, x1, Qd[I][1], w1);
            dmma(x0, x1, qi0, wd0);
            dmma(x0, x1, qi1, wd1);
            xd[I][K][0] = x0; xd[I][K][1] = x1;
        }
    }
}

// Sinusoidal mean m(t) = μ + A·sin(2πt/T₀ + ϕ) (the reference's periodicity run, examples/ultranest/single_pl_periodicity.jl):
// the right-hand sides ∂ỹ/∂θ_k of its three parameters (A, ϕ, T₀) at the steps n0 + 2t, n0 + 2t + 1 of lane (g, t), row g = k.
// They are formed here from the times rather than read from rows the transform writes: 8 sines per block on the mean warp cost
// less than 24 N bytes per parameter vector of extra rows, written and read once.
__device__ __forceinline__ void sine_mean_rhs(const double* __restrict__ tt, const int64_t n0, const int64_t N, const int g,
                                              const int t, const double A, const double phi, const double T0, double& r0,
                                              double& r1) {
    double r[2];
#pragma unroll
    for (int c = 0; c < 2; c++) {
        const int64_t n = n0 + 2 * t + c;
        r[c] = 0.0;
        if (n < N && g < 3) {
            const double w = 6.283185307179586 * tt[n] / T0;      // 2π·t/T₀, as the reference forms the argument
            double si, co;
            sincos(w + phi, &si, &co);
            r[c] = g == 0 ? -si : g == 1 ? -A * co : A * co * (w / T0);
        }
    }
    r0 = r[0]; r1 = r[1];
}

// One block of the mean warp: the three data rows whose right-hand sides are ∂ỹ/∂(A, ϕ, T₀), one row tile of the state (row g =
// direction g, columns the celerite rows), following the value warp's published factor like a tangent warp; mpar = (A, ϕ, T₀),
// read per block rather than held in registers across the sweep.  With xm that tile:
//     P0 = xm·Û,   Bm = r − P0 (a data row: ψ8 = 1, amplitude 1),   ż = Bm·Eᵀ,   xm ← ψ8ᵀ∘xm + ż·Ŵᵀ
// and ∂χ²/∂θ_k = Σ_s 2 z_s ż_{k,s}/D_s.  2·NT + 2 + 2·NT DMMAs (fewer in HALF mode).
template <int NT, int NTR, bool HALF>
__device__ __forceinline__ void blocked_mean_step(double (&xm)[NT][2], const double* __restrict__ tab, const double* __restrict__ slot,
                                                  const BlkLane& L, const int lane, const double* __restrict__ tt,
                                                  const double* __restrict__ mpar, const int64_t n0, const int64_t N, const int RG,
                                                  double& dchi) {
    constexpr int O_PSI = blk_off_psi(NT, NTR);
    const int g = L.g, t = L.t;
    double b0 = 0.0, b1 = 0.0;
#pragma unroll
    for (int K = 0; K < NT; K++) {
        const double2 u = *reinterpret_cast<const double2*>(tab + K * 64 + g * 8 + 2 * t);
        dmma(b0, b1, xm[K][0], u.x);
        if (!(HALF && K == NT - 1)) dmma(b0, b1, xm[K][1], u.y);
    }
#pragma unroll
    for (int K = 0; K < NT; K++) {
        const double2 pc = *reinterpret_cast<const double2*>(tab + O_PSI + 8 * K + 2 * t);
        xm[K][0] *= pc.x;
        xm[K][1] *= pc.y;
    }
    double r0, r1;
    sine_mean_rhs(tt, n0, N, g, t, mpar[0], mpar[1], mpar[2], r0, r1);
    b0 = r0 - b0;
    b1 = r1 - b1;
    const double* sl = slot + lane;
    const double e0 = sl[0], e1 = sl[32], rd0 = sl[64], rd1 = sl[96];
    double q0 = 0.0, q1 = 0.0;
    dmma(q0, q1, b0, e0);
    dmma(q0, q1, b1, e1);
    // z of steps 2t, 2t + 1: the value warp's innovations, published by the lane that holds row RG
    const int zl = ((RG & 7) << 2) | t;
    const double z0 = slot[(4 + 2 * NTR + 2 * (NTR - 1)) * 32 + zl], z1 = slot[(5 + 2 * NTR + 2 * (NTR - 1)) * 32 + zl];
    dchi = fma(z0 * rd0, q0, fma(z1 * rd1, q1, dchi));
#pragma unroll
    for (int K = 0; K < NT; K++) {
        const double w0 = sl[(4 + 2 * NTR + 2 * K) * 32] * rd0, w1 = sl[(5 + 2 * NTR + 2 * K) * 32] * rd1;
        dmma(xm[K][0], xm[K][1], q0, w0);
        dmma(xm[K][0], xm[K][1], q1, w1);
    }
}

// grid = work items (one parameter vector each); block = 1 + NTAN warps (NTAN = n_psd_par + 1).
// dynamic smem: BLK_NSTAGE block records | 2 ring slots | (1 + NTAN) × (8·NTR + 8·NT) amplitudes | mbarriers | 2 result doubles
// Up to 5 row tiles two CTAs share an SM (≤ 200 registers per thread): the value warp of one overlaps the tangent warps of the other.
template <int NT, int NTR, bool HALF, int NTAN>
__global__ void __launch_bounds__((1 + NTAN) * 32, (NT <= PIORAN_BLKG_TWO_CTA_MAX_NT && NTAN <= 4) ? 2 : 1) celerite_blocked_grad_kernel(const GradArgs args, const int R, const int amp_stride, const int RG, const int RM) {
    constexpr int BD = blk_doubles(NT, NTR), RPT = 8 * NTR, APW = RPT + 8 * NT, SLOT = blk_slot_doubles(NTR);
    constexpr uint32_t STAGE_BYTES = BD * sizeof(double);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* stages = reinterpret_cast<double*>(smem_raw);
    double* ring = stages + BLK_NSTAGE * BD;
    double* amps = ring + 2 * SLOT;
    double* res = amps + (1 + NTAN) * APW;
    uint64_t* bars = reinterpret_cast<uint64_t*>(res + 2);

    const WorkItem wk = args.work[blockIdx.x];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int th = wk.theta_begin;
    const int64_t N = wk.N;
    const int64_t nblocks = (N + BLK - 1) / BLK;
    const int P = args.ND + 3 + args.cdir;

    if (threadIdx.x == 0) {
        for (int k = 0; k < BLK_NSTAGE; k++) mbar_init(&bars[k], 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 0; k < BLK_NSTAGE && k < nblocks; k++) {
            mbar_arrive_expect_tx(&bars[k], STAGE_BYTES);
            tma_load_1d(stages + k * BD, wk.table + (size_t)k * BD, STAGE_BYTES, &bars[k]);
        }
    }
    const BlkLane L = make_blk_lane(lane);
    const double* trow = args.theta + (size_t)th * args.pstride;
    const double nu = trow[args.ND + 1], mu = trow[args.ND + 2];
    const double* yb = args.y_batch ? args.y_batch + (size_t)th * args.ystride : nullptr;
    const double* sb = args.s2_batch ? args.s2_batch + (size_t)th * args.ystride : nullptr;

    // amplitudes of this warp: the values (warp 0, data rows = 1) or the tangent of direction warp − 1 (zero for ν)
    double* amp_s = amps + warp * APW;
    double* amp_l = amp_s + RPT;
    for (int k = lane; k < APW; k += 32) amp_s[k] = 0.0;
    __syncwarp();
    const int dir = warp - 1;
    const bool amp_dir = warp >= 1 && dir < args.ND;
    if (warp == 0 || amp_dir) {
        const double* src = warp == 0 ? args.amp + (size_t)th * amp_stride : args.damp + ((size_t)th * args.ND + dir) * amp_stride;
        for (int k = lane; k < R; k += 32) {
            const double av = src[k];
            amp_s[blk_phys_row(k, R)] = av;
            amp_l[k] = av;
        }
    }
    if (warp == 0 && lane == 0) { amp_s[RG] = 1.0; amp_s[RM] = 1.0; }
    __syncwarp();
    const double suma = args.suma[th];
    const double dsuma = amp_dir ? args.dsuma[(size_t)th * args.ND + dir] : 0.0;
    const bool c_dir = args.cdir && dir == args.ND + 1;          // directions: psd parameters…, ν, (c)
    const double dnu = (warp >= 1 && dir == args.ND) ? 1.0 : 0.0;

    BlkState<NT, NTR> st;      // warp 0: X;  tangent warps: Ẋ in st.x
#pragma unroll
    for (int I = 0; I < NTR; I++)
#pragma unroll
        for (int K = 0; K < NT; K++) st.x[I][K][0] = st.x[I][K][1] = 0.0;
    st.chi2 = 0.0; st.logacc = 0.0; st.dkeep = 1.0; st.dfirst = 1.0;
    double chimu = 0.0, dlog = 0.0, dchi = 0.0, cm0 = 0.0, cm1 = 0.0;

    // tick τ: the value warp sweeps block τ, the tangent warps block τ − 1; block b sits in stage b mod BLK_NSTAGE and its
    // published factor in ring slot b & 1
    for (int64_t tau = 0; tau <= nblocks; tau++) {
        if (warp == 0) {
            if (tau < nblocks) {
                const int sidx = (int)(tau % BLK_NSTAGE);
                mbar_wait(&bars[sidx], (uint32_t)((tau / BLK_NSTAGE) & 1));
                blocked_step<NT, NTR, HALF, true>(st, stages + sidx * BD, stages + sidx * BD, amp_s, amp_l, L, lane, suma, mu, nu,
                                                  tau * BLK, N, yb, sb, RG, cm0, cm1, ring + (tau & 1) * SLOT, RM, &chimu);
            }
        } else if (tau >= 1) {
            const int64_t b = tau - 1;
            const int sidx = (int)(b % BLK_NSTAGE);
            mbar_wait(&bars[sidx], (uint32_t)((b / BLK_NSTAGE) & 1));
            blocked_tangent_step<NT, NTR, HALF>(st.x, stages + sidx * BD, ring + (b & 1) * SLOT, amp_s, amp_l, L, lane, dsuma, dnu,
                                                b * BLK, N, RG, dlog, dchi, yb, sb, c_dir, nu);
        }
        __syncthreads();
        // every warp has left block τ − 1: its stage takes block τ − 1 + BLK_NSTAGE
        if (threadIdx.x == 0 && tau >= 1 && tau - 1 + BLK_NSTAGE < nblocks) {
            const int sidx = (int)((tau - 1) % BLK_NSTAGE);
            fence_proxy_async();
            mbar_arrive_expect_tx(&bars[sidx], STAGE_BYTES);
            tma_load_1d(stages + sidx * BD, wk.table + (size_t)(tau - 1 + BLK_NSTAGE) * BD, STAGE_BYTES, &bars[sidx]);
        }
    }

    if (warp == 0) {
        double la = st.logacc + log(fabs(st.dkeep)), ch = st.chi2, cmu = chimu;
#pragma unroll
        for (int sft = 16; sft >= 1; sft >>= 1) {
            la += __shfl_xor_sync(FULL, la, sft);
            ch += __shfl_xor_sync(FULL, ch, sft);
            cmu += __shfl_xor_sync(FULL, cmu, sft);
        }
        const double logdet = log(__shfl_sync(FULL, st.dfirst, 0)) + la;
        if (lane == 0) {
            if (args.logl) args.logl[th] = -logdet / 2 - (double)N * 1.8378770664093453 / 2 - ch / 2;
            args.grad[(size_t)th * P + args.ND + 2] = -cmu / 2;
            res[0] = ch;
        }
    }
    __syncthreads();
    if (warp >= 1) {
        double dl = dlog, dc = dchi;
#pragma unroll
        for (int sft = 16; sft >= 1; sft >>= 1) {
            dl += __shfl_xor_sync(FULL, dl, sft);
            dc += __shfl_xor_sync(FULL, dc, sft);
        }
        if (lane == 0) {
            const double gk = -dl / 2 - dc / 2;
            if (dir < args.ND) {
                args.grad[(size_t)th * P + dir] = gk;
            } else if (c_dir) {
                args.grad[(size_t)th * P + args.ND + 3] = gk;
            } else {      // the ν warp also reports ∂/∂norm (homogeneity of K in (norm, ν), grad.cuh)
                args.grad[(size_t)th * P + args.ND + 1] = gk;
                args.grad[(size_t)th * P + args.ND] = (0.5 * res[0] - 0.5 * (double)N - nu * gk) / trow[args.ND];
            }
        }
    }
}

// Sinusoidal mean: θ rows [psd parameters…, norm, ν, μ, A, ϕ, T₀] and args.y_batch = y − A·sin(2πt/T₀ + ϕ) per θ.  The CTA of
// celerite_blocked_grad_kernel plus the mean warp (warp 1 + NTAN); dynamic smem as there, with 2 + NTAN amplitude slots (the mean
// warp's is zeroed and never read).  A kernel of its own rather than a flag of celerite_blocked_grad_kernel: the existing
// instantiations then compile to the same code as before.
template <int NT, int NTR, bool HALF, int NTAN>
__global__ void __launch_bounds__((2 + NTAN) * 32, (NT <= PIORAN_BLKG_TWO_CTA_MAX_NT && NTAN + 1 <= 4) ? 2 : 1) celerite_blocked_grad_sine_kernel(const GradArgs args, const int R, const int amp_stride, const int RG, const int RM) {
    constexpr int BD = blk_doubles(NT, NTR), RPT = 8 * NTR, APW = RPT + 8 * NT, SLOT = blk_slot_doubles(NTR);
    constexpr uint32_t STAGE_BYTES = BD * sizeof(double);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* stages = reinterpret_cast<double*>(smem_raw);
    double* ring = stages + BLK_NSTAGE * BD;
    double* amps = ring + 2 * SLOT;
    double* res = amps + (2 + NTAN) * APW;
    uint64_t* bars = reinterpret_cast<uint64_t*>(res + 2);

    const WorkItem wk = args.work[blockIdx.x];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int th = wk.theta_begin;
    const int64_t N = wk.N;
    const int64_t nblocks = (N + BLK - 1) / BLK;
    const int P = args.ND + 6;

    if (threadIdx.x == 0) {
        for (int k = 0; k < BLK_NSTAGE; k++) mbar_init(&bars[k], 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 0; k < BLK_NSTAGE && k < nblocks; k++) {
            mbar_arrive_expect_tx(&bars[k], STAGE_BYTES);
            tma_load_1d(stages + k * BD, wk.table + (size_t)k * BD, STAGE_BYTES, &bars[k]);
        }
    }
    const BlkLane L = make_blk_lane(lane);
    const double* trow = args.theta + (size_t)th * args.pstride;
    const double nu = trow[args.ND + 1], mu = trow[args.ND + 2];
    const double* yb = args.y_batch + (size_t)th * args.ystride;      // σ² is the resident one

    // amplitudes of this warp: the values (warp 0, data rows = 1) or the tangent of direction warp − 1 (zero for ν)
    double* amp_s = amps + warp * APW;
    double* amp_l = amp_s + RPT;
    for (int k = lane; k < APW; k += 32) amp_s[k] = 0.0;
    __syncwarp();
    const int dir = warp - 1;
    const bool amp_dir = warp >= 1 && dir < args.ND;
    if (warp == 0 || amp_dir) {
        const double* src = warp == 0 ? args.amp + (size_t)th * amp_stride : args.damp + ((size_t)th * args.ND + dir) * amp_stride;
        for (int k = lane; k < R; k += 32) {
            const double av = src[k];
            amp_s[blk_phys_row(k, R)] = av;
            amp_l[k] = av;
        }
    }
    if (warp == 0 && lane == 0) { amp_s[RG] = 1.0; amp_s[RM] = 1.0; }
    __syncwarp();
    const double suma = args.suma[th];
    const double dsuma = amp_dir ? args.dsuma[(size_t)th * args.ND + dir] : 0.0;
    const double dnu = (warp >= 1 && dir == args.ND) ? 1.0 : 0.0;

    BlkState<NT, NTR> st;      // warp 0: X;  tangent warps: Ẋ in st.x
#pragma unroll
    for (int I = 0; I < NTR; I++)
#pragma unroll
        for (int K = 0; K < NT; K++) st.x[I][K][0] = st.x[I][K][1] = 0.0;
    st.chi2 = 0.0; st.logacc = 0.0; st.dkeep = 1.0; st.dfirst = 1.0;
    double chimu = 0.0, dlog = 0.0, dchi = 0.0, cm0 = 0.0, cm1 = 0.0;

    // tick τ: the value warp sweeps block τ, the tangent warps block τ − 1; block b sits in stage b mod BLK_NSTAGE and its
    // published factor in ring slot b & 1
    for (int64_t tau = 0; tau <= nblocks; tau++) {
        if (warp == 0) {
            if (tau < nblocks) {
                const int sidx = (int)(tau % BLK_NSTAGE);
                mbar_wait(&bars[sidx], (uint32_t)((tau / BLK_NSTAGE) & 1));
                blocked_step<NT, NTR, HALF, true>(st, stages + sidx * BD, stages + sidx * BD, amp_s, amp_l, L, lane, suma, mu, nu,
                                                  tau * BLK, N, yb, nullptr, RG, cm0, cm1, ring + (tau & 1) * SLOT, RM, &chimu);
            }
        } else if (tau >= 1) {
            const int64_t b = tau - 1;
            const int sidx = (int)(b % BLK_NSTAGE);
            mbar_wait(&bars[sidx], (uint32_t)((b / BLK_NSTAGE) & 1));
            if (warp == 1 + NTAN)      // the mean warp; its row tile is the last of st.x
                blocked_mean_step<NT, NTR, HALF>(st.x[NTR - 1], stages + sidx * BD, ring + (b & 1) * SLOT, L, lane, wk.t,
                                                 trow + args.ND + 3, b * BLK, N, RG, dchi);
            else
                blocked_tangent_step<NT, NTR, HALF>(st.x, stages + sidx * BD, ring + (b & 1) * SLOT, amp_s, amp_l, L, lane, dsuma, dnu,
                                                    b * BLK, N, RG, dlog, dchi);
        }
        __syncthreads();
        // every warp has left block τ − 1: its stage takes block τ − 1 + BLK_NSTAGE
        if (threadIdx.x == 0 && tau >= 1 && tau - 1 + BLK_NSTAGE < nblocks) {
            const int sidx = (int)((tau - 1) % BLK_NSTAGE);
            fence_proxy_async();
            mbar_arrive_expect_tx(&bars[sidx], STAGE_BYTES);
            tma_load_1d(stages + sidx * BD, wk.table + (size_t)(tau - 1 + BLK_NSTAGE) * BD, STAGE_BYTES, &bars[sidx]);
        }
    }

    if (warp == 0) {
        double la = st.logacc + log(fabs(st.dkeep)), ch = st.chi2, cmu = chimu;
#pragma unroll
        for (int sft = 16; sft >= 1; sft >>= 1) {
            la += __shfl_xor_sync(FULL, la, sft);
            ch += __shfl_xor_sync(FULL, ch, sft);
            cmu += __shfl_xor_sync(FULL, cmu, sft);
        }
        const double logdet = log(__shfl_sync(FULL, st.dfirst, 0)) + la;
        if (lane == 0) {
            if (args.logl) args.logl[th] = -logdet / 2 - (double)N * 1.8378770664093453 / 2 - ch / 2;
            args.grad[(size_t)th * P + args.ND + 2] = -cmu / 2;
            res[0] = ch;
        }
    }
    __syncthreads();
    if (warp == 1 + NTAN) {      // ∂logℒ/∂θ_k = −½ Σ_s 2 z_s ż_{k,s}/D_s: row g = k sits on lanes (g, ·)
        double dc = dchi;
        dc += __shfl_xor_sync(FULL, dc, 1);
        dc += __shfl_xor_sync(FULL, dc, 2);
        if (lane < 12 && (lane & 3) == 0) args.grad[(size_t)th * P + args.ND + 3 + (lane >> 2)] = -dc;
    } else if (warp >= 1) {
        double dl = dlog, dc = dchi;
#pragma unroll
        for (int sft = 16; sft >= 1; sft >>= 1) {
            dl += __shfl_xor_sync(FULL, dl, sft);
            dc += __shfl_xor_sync(FULL, dc, sft);
        }
        if (lane == 0) {
            const double gk = -dl / 2 - dc / 2;
            if (dir < args.ND) {
                args.grad[(size_t)th * P + dir] = gk;
            } else {      // the ν warp also reports ∂/∂norm (homogeneity of K in (norm, ν), grad.cuh)
                args.grad[(size_t)th * P + args.ND + 1] = gk;
                args.grad[(size_t)th * P + args.ND] = (0.5 * res[0] - 0.5 * (double)N - nu * gk) / trow[args.ND];
            }
        }
    }
}

}  // namespace pioran
