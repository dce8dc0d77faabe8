// lsp.cuh — K9: generalised Lomb–Scargle periodograms (floating mean, Zechmeister & Kürster 2009) of many rows on the times
// of one series, FP64 throughout.  The definition is tests/tools/proto/lsp_math.py.  Everything that depends on the
// frequency only (the basis cos πx, sin πx and the normalisers C, S, CC, SS, CS) is built once per frequency chunk and shared
// by every row; the one part that depends on the row is the product  [w·ỹ] [rows × N] · [cos | sin] [N × 2F]  on DMMA.
//
//   lsp_table_kernel    one warp per frequency: the basis columns (interleaved: column 2j = cos of frequency j, 2j + 1 = sin)
//                       stored column-major over n, and the normalisers, reduced over n in a fixed order;
//   lsp_rows_kernel     one warp per row: Ȳ = Σ w y, YY = Σ w ỹ², and the centered, weighted row w·ỹ;
//   lsp_product_kernel  the product on the tensor pipe with p(f) formed in the epilogue.  A lane's accumulator pair holds two
//                       adjacent columns, i.e. (YC, YS) of one frequency.  Every (row, frequency) is summed over n in the same
//                       order whatever the batch, the chunking or the row's position: there is no split over n.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "dense.cuh"       // dmma_8x8x4, cp_async16
#include "posterior.cuh"   // warp_sum: an xor butterfly, so every lane ends with the same bits (addition commutes)

namespace pioran {

constexpr int LSP_BM = 64;    // rows per CTA tile
constexpr int LSP_BN = 64;    // interleaved basis columns per CTA tile (32 frequencies)
constexpr int LSP_BK = 32;    // steps n per shared-memory stage; N is padded to a multiple (zero weight, zero row)
constexpr int LSP_LDS = LSP_BK + 4;   // shared row stride (doubles): a fragment load falls on 32 distinct banks
constexpr size_t LSP_SMEM = sizeof(double) * 2 * (LSP_BM + LSP_BN) * LSP_LDS;   // two stages: 73 728 bytes

// Per-frequency normalisers: CC, SS, CS and the denominator factor CC·SS − CS².
struct LspNorm { double cc, ss, cs, den; };

// grid = nfpad / 8, block = 256.  Frequencies j ≥ nf (the padding of the last column tile) get zero columns.
__global__ void __launch_bounds__(256) lsp_table_kernel(const double* __restrict__ t, const double* __restrict__ w, int64_t N,
                                                        int64_t Npad, const double* __restrict__ freq, int nf, int nfpad,
                                                        double* __restrict__ tab, LspNorm* __restrict__ norm) {
    const int j = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (j >= nfpad) return;
    double* cs = tab + (size_t)(2 * j) * Npad;
    double* sn = cs + Npad;
    if (j >= nf) {
        for (int64_t n = lane; n < Npad; n += 32) cs[n] = sn[n] = 0.0;
        return;
    }
    const double f2 = 2.0 * freq[j], t0 = t[0];
    double sc = 0.0, ss = 0.0, scc = 0.0, sss = 0.0, scs = 0.0;
    for (int64_t n = lane; n < Npad; n += 32) {
        double s = 0.0, c = 0.0;
        if (n < N) {
            sincospi(f2 * (t[n] - t0), &s, &c);   // exact range reduction of the phase
            const double wn = w[n];
            sc += wn * c; ss += wn * s;
            scc += wn * c * c; sss += wn * s * s; scs += wn * c * s;
        }
        cs[n] = c; sn[n] = s;
    }
    sc = warp_sum(sc); ss = warp_sum(ss); scc = warp_sum(scc); sss = warp_sum(sss); scs = warp_sum(scs);
    if (lane == 0) {
        LspNorm q;
        q.cc = scc - sc * sc; q.ss = sss - ss * ss; q.cs = scs - sc * ss;
        q.den = q.cc * q.ss - q.cs * q.cs;
        norm[j] = q;
    }
}

// grid = nrpad / 8, block = 256.  Row r < nr reads y + r·ldy; rows r ≥ nr (the padding of the last row tile) are zero.
__global__ void __launch_bounds__(256) lsp_rows_kernel(const double* __restrict__ y, int64_t ldy, const double* __restrict__ w,
                                                       int64_t N, int64_t Npad, int nr, int nrpad, double* __restrict__ A,
                                                       double* __restrict__ YY) {
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (r >= nrpad) return;
    double* a = A + (size_t)r * Npad;
    if (r >= nr) {
        for (int64_t n = lane; n < Npad; n += 32) a[n] = 0.0;
        if (lane == 0) YY[r] = 0.0;
        return;
    }
    const double* yr = y + (size_t)r * ldy;
    double m = 0.0;
    for (int64_t n = lane; n < N; n += 32) m += w[n] * yr[n];
    m = warp_sum(m);
    double q = 0.0;
    for (int64_t n = lane; n < Npad; n += 32) {
        double v = 0.0;
        if (n < N) {
            const double yt = yr[n] - m, wn = w[n];
            q += wn * yt * yt;
            v = wn * yt;
        }
        a[n] = v;
    }
    q = warp_sum(q);
    if (lane == 0) YY[r] = q;
}

// grid = (2·nfpad / BN, nrpad / BM), block = 256 = 8 warps, dynamic shared memory LSP_SMEM.  Warp (wy, wx) owns rows
// 32·wy … and columns 16·wx … of the tile as 4 × 2 DMMA tiles; the k-loop over n is staged through shared memory in two
// cp.async stages of BK steps.  out[r·ldo + j] = p of row r and frequency j of the chunk.
template <int BM, int BN, int BK>
__global__ void __launch_bounds__(256) lsp_product_kernel(const double* __restrict__ A, const double* __restrict__ tab, int64_t Npad,
                                                          const double* __restrict__ YY, const LspNorm* __restrict__ norm, int nr,
                                                          int nf, double* __restrict__ out, int64_t ldo) {
    static_assert(BM == 64 && BN == 64 && BK % 16 == 0, "warp layout: 2 × 4 warps of 32 × 16");
    constexpr int LDS = BK + 4, CH = BK / 2;   // 16-byte chunks per tile row
    extern __shared__ __align__(16) double lsp_sm[];
    double (*As)[BM][LDS] = reinterpret_cast<double (*)[BM][LDS]>(lsp_sm);            // [stage][row][k]
    double (*Bs)[BN][LDS] = reinterpret_cast<double (*)[BN][LDS]>(lsp_sm + 2 * BM * LDS);   // [stage][column][k]
    const int r0 = blockIdx.y * BM, c0 = blockIdx.x * BN;
    const double* Ag = A + (size_t)r0 * Npad;
    const double* Bg = tab + (size_t)c0 * Npad;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wy = warp >> 2, wx = warp & 3, gr = lane >> 2, gc = lane & 3;
    auto stage = [&](int st, int64_t k0) {
#pragma unroll
        for (int q = 0; q < BM * CH / 256; q++) {
            const int e = threadIdx.x + q * 256, r = e / CH, k = 2 * (e - r * CH);
            cp_async16(&As[st][r][k], Ag + (size_t)r * Npad + k0 + k);
        }
#pragma unroll
        for (int q = 0; q < BN * CH / 256; q++) {
            const int e = threadIdx.x + q * 256, r = e / CH, k = 2 * (e - r * CH);
            cp_async16(&Bs[st][r][k], Bg + (size_t)r * Npad + k0 + k);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    double acc[4][2][2];
#pragma unroll
    for (int u = 0; u < 4; u++)
#pragma unroll
        for (int v = 0; v < 2; v++) acc[u][v][0] = acc[u][v][1] = 0.0;
    const int64_t nk = Npad / BK;
    stage(0, 0);
    for (int64_t kt = 0; kt < nk; kt++) {
        const int st = (int)(kt & 1);
        if (kt + 1 < nk) {
            stage(st ^ 1, (kt + 1) * BK);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
#pragma unroll
        for (int k4 = 0; k4 < BK / 4; k4++) {
            double a[4], b[2];
#pragma unroll
            for (int u = 0; u < 4; u++) a[u] = As[st][32 * wy + 8 * u + gr][4 * k4 + gc];
#pragma unroll
            for (int v = 0; v < 2; v++) b[v] = Bs[st][16 * wx + 8 * v + gr][4 * k4 + gc];
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
                for (int v = 0; v < 2; v++) dmma_8x8x4(acc[u][v][0], acc[u][v][1], a[u], b[v]);
        }
        __syncthreads();   // the next iteration's copy overwrites this stage
    }
    // acc[u][v] = (YC, YS) of row 32·wy + 8u + gr and frequency (c0 + 16·wx + 8v + 2·gc) / 2
#pragma unroll
    for (int u = 0; u < 4; u++) {
        const int r = r0 + 32 * wy + 8 * u + gr;
        if (r >= nr) continue;
        const double yy = YY[r];
#pragma unroll
        for (int v = 0; v < 2; v++) {
            const int j = c0 / 2 + 8 * wx + 4 * v + gc;
            if (j >= nf) continue;
            const LspNorm q = norm[j];
            const double yc = acc[u][v][0], ys = acc[u][v][1];
            out[(size_t)r * ldo + j] = (q.ss * yc * yc + q.cc * ys * ys - 2.0 * q.cs * yc * ys) / (yy * q.den);
        }
    }
}

}  // namespace pioran
