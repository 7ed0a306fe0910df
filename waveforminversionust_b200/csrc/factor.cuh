// factor.cuh -- two-sided block-tridiagonal factorisation with explicit block inverses.
//
//   down chain: S_i = D_i - L_i T_{i-1} U_{i-1}          T_i = S_i^{-1}
//   up   chain: S_i = D_i - U_i T_{i+1} L_{i+1}
//   middle    : S_m = D_m - L_m T_{m-1} U_{m-1} - U_m T_{m+1} L_{m+1}
// (SURVEY.md Appendix A.5; replaces the LU half of SuperLU gssv behind solve_helmholtz.py:15-18.)
//
// Each T_i is formed by an in-place-equivalent blocked Gauss-Jordan inversion (block GJ_NB=64, no
// inter-block pivoting: the Schur complements are well conditioned, cond ~ 9, first PML row ~ 7e2),
// ping-ponging between the T slot and a scratch block so that no kernel reads what it writes:
//   step k:  P  = inv(X_kk)
//            R  = P * Xtilde_k,:          (Xtilde = X with block column k replaced by e_k blocks)
//            X' = Xtilde - X_:,k * R      (rows i != k);    X'_k,: = R
// schur_kernel     : builds S_i from T_prev and the coefficient planes (O(n^2), 3x3 stencil on T_prev)
// gj_pivot_kernel   : pivot-block inverse in shared memory (one CTA per chain)
// gj_rowpanel_kernel: row panel R = P * Xtilde_k,:
// gj_update_kernel : rank-64 update of every other block row (the GEMM-shaped part)
#pragma once
#include "common.cuh"
#include "gemm_simt.cuh"
#include "gemm_tc2.cuh"
#include "gemm_tc2h.cuh"

namespace ust {

template <typename R>
struct FactorArgs {
    Geom g;
    int phase, step, nbatch;
    const cx<R>* planes;  // [nfreq][9][Ny][Nx]
    cx<R>* T;             // [nfreq][M][nP*nP]
    cx<R>* scratch;       // [2*nfreq][nP*nP]
    cx<R>* pbuf;          // [2*nfreq][64*64] pivot-block inverses (transposed)
    int* status;
    // TMA-fed tensor-core update (gemm_tc2.cuh, complex64 only; null otherwise)
    uint16_t* Rp;         // [nbmax] B planes of the row panel R (64 x nP), bplanes layout with 4 k-chunks
    uint16_t* Xp;         // [2][nbmax] B planes of the pivot block row Xtilde_k,: (64 x nP), ping-pong on k
    uint16_t* Cp;         // [2][nbmax][6][nP/8][8][8][8] A planes of the column panel X_:,k (nP x 64), ping-pong on k
    uint16_t* Pp;         // [nbmax][6][8][8][8][8] A planes of the pivot-block inverse P (64 x 64)
    uint16_t* Tp;         // [nfreq*M][6][nP/8][nP/8][8][8] A planes of the finished block inverses
    size_t rp_stride;     // elements per batch entry of Xp and Rp: B planes of 64 rows
    int nbmax;            // batch capacity (2 * max_freq)
    int gj_drain;         // drain period (chunks) of the leading accumulator in the K = 64 Gauss-Jordan GEMMs
    int inplace;          // TMA-fed engine: X^(k) is updated in place in its T slot (no ping-pong: the batch stays L2 resident)
    cx<R>* snap;          // [nbmax][64*64] copy of X^(k)_{k+1,k+1}: the Cin of the look-ahead pivot CTA (the update overwrites the block in place)
    unsigned long long* trace;  // debugging (UST_TC2_TRACE_UPDATE=step,k): [1024][16] phase timestamps of the update CTAs
    int trace_step, trace_k;
    int prefetch_cin;     // update kernel: L2 prefetch of the X tile at CTA start
    // Frequency groups run as independent launch chains on separate streams: a launch covers the chains of the
    // frequencies [f0, f0 + nbatch / 2) (PH_MID: nbatch); blockIdx.z is local to the group, zb0 + z indexes the per-chain
    // work buffers (Rp, Xp, Cp, Pp, snap, pbuf, scratch) and f0 + chain_freq() the per-frequency arrays.
    int zb0, f0;
    int t_ring;           // FP32 T holds 4 slots per frequency (previous / current row of either chain) instead of all M rows
};

// FP32 block slot of (frequency, block row).  The Schur update only ever reads the previous row of the same chain (the
// middle row: of both chains), so the TMA-fed engine -- whose sweeps read the bf16 planes Tp, never T -- keeps a ring
// of two slots per chain: rows alternate by parity, the middle row takes the down chain's free slot.
template <typename R>
__device__ __forceinline__ cx<R>* t_slot(const FactorArgs<R>& a, int freq, int row) {
    const size_t bs = (size_t)a.g.nP * a.g.nP;
    if (a.t_ring) return a.T + ((size_t)freq * 4 + (row > a.g.mid ? 2 : 0) + (row & 1)) * bs;
    return a.T + ((size_t)freq * a.g.M + row) * bs;
}

// buffer holding X^{(k)} for batch entry z working on block row `row`
template <typename R>
__device__ __forceinline__ cx<R>* gj_buffer(const FactorArgs<R>& a, int z, int freq, int row, int k) {
    const size_t bs = (size_t)a.g.nP * a.g.nP;
    cx<R>* slot = t_slot(a, freq, row);
    if (a.inplace) return slot;
    cx<R>* scr = a.scratch + (size_t)(a.zb0 + z) * bs;
    const int nblk = a.g.nP / GJ_NB;
    const bool k_even = (k & 1) == 0;
    const bool slot_holds_even = (nblk & 1) == 0;  // X^{(nblk)} must land in the T slot
    return (k_even == slot_holds_even) ? slot : scr;
}

// One CTA (16 x 16 threads) = one TS x TS tile of S.  Thread (tx, ty) owns rows a0 + PT*ty .. + PT-1 (contiguous) and
// columns b0 + tx + 16*dx (strided: a half-warp reads / writes 16 consecutive complex values, conflict free and
// coalesced).  The (TS+2)^2 halo tile of T_prev and the tridiagonal coefficients of the tile's rows / columns are staged
// in shared memory, one coupled neighbour (t) at a time; per neighbour a thread first contracts the column coefficients
// (rowacc, PT+2 rows) and then the row coefficients.  TS = 64 for complex64: with 32 x 32 tiles the launch was 8192 CTAs
// of ~1 us of work each and ran at the CTA dispatch rate (74 us for 128 MB of traffic).
template <typename R>
struct SchurTile { static constexpr int TS = sizeof(R) == 4 ? 64 : 32; };

template <typename R>
__device__ __forceinline__ void gj_pivot_body(const FactorArgs<R>& a, int k, int z, unsigned char* smem_raw, const cx<R>* sm_block);

// `pivot0` (TMA-fed engine): the tile (0, 0) of a chain IS pivot block 0 (TS = 64 = GJ_NB), so the CTA that computes it goes
// on to invert it (gj_pivot_body from shared memory) and emits P_0; those CTAs are numbered first so that the 64-step
// inversion runs under the rest of the launch instead of in the k = 0 launch after it.
template <typename R>
__global__ void __launch_bounds__(256, sizeof(R) == 4 ? 3 : 2) schur_kernel(FactorArgs<R> a, int pivot0) {
    constexpr int TS = SchurTile<R>::TS, PT = TS / 16;
    __shared__ cx<R> Tt[TS + 2][TS + 3];
    __shared__ cx<R> lc[TS][3], rc[TS][3];
    pdl_trigger();
    pdl_wait();
    int z = blockIdx.z, bx = blockIdx.x, by = blockIdx.y;
    if (pivot0) {
        const int T = gridDim.x, nb = gridDim.z;
        int L = bx + T * (by + T * z);
        if (L < nb) { z = L; bx = 0; by = 0; }
        else { L -= nb; z = L / (T * T - 1); const int r = L % (T * T - 1) + 1; bx = r % T; by = r / T; }
    }
    const int row = chain_row(a.g, a.phase, z, a.step);
    if (row < 0) return;
    const int freq = (a.f0 + chain_freq(a.phase, z)), dir = chain_dir(a.phase, z);
    const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * 16 + tx;
    const int b0 = bx * TS, a0 = by * TS;
    const int nI = a.g.nI, nP = a.g.nP, M = a.g.M;
    const size_t pl = (size_t)a.g.Nx * a.g.Ny;
    const cx<R>* planes_f = a.planes + (size_t)freq * 9 * pl;
    const int y = row + 1;
    const size_t bs = (size_t)nP * nP;
    const bool on[2] = {(dir == 0 || dir == 2) && row > 0, (dir == 1 || dir == 2) && row < M - 1};
    const bool interior = a0 < nI && b0 < nI;

    // D_i (tridiagonal) or the identity of the padding block
    cx<R> out[PT][PT];
#pragma unroll
    for (int dy = 0; dy < PT; ++dy) {
        const int ai = a0 + PT * ty + dy;
#pragma unroll
        for (int dx = 0; dx < PT; ++dx) {
            const int bi = b0 + tx + 16 * dx;
            cx<R> v = cxzero<R>();
            if (ai < nI && bi < nI) {
                const size_t o = (size_t)y * a.g.Nx + (ai + 1);
                if (bi == ai) v = planes_f[PL_C * pl + o];
                else if (bi == ai - 1) v = planes_f[PL_L * pl + o];
                else if (bi == ai + 1) v = planes_f[PL_R * pl + o];
            } else if (ai == bi) {
                v = cxone<R>();
            }
            out[dy][dx] = v;
        }
    }
    if (interior) {
#pragma unroll 1
        for (int t = 0; t < 2; ++t) {
            if (!on[t]) continue;
            if (t == 1 && on[0]) __syncthreads();  // middle row: the shared tile is reused for the second neighbour
            const cx<R>* Tp = t_slot(a, freq, t == 0 ? row - 1 : row + 1);
            // halo tile: loads in batches of HB before the shared-memory stores (a generic pointer may alias shared memory as
            // far as the compiler knows, so a load-store loop is serialised: 18 exposed L2/HBM latencies per CTA = 17 us);
            // the coefficient loads of the tile's rows / columns go out between the first batch's loads and its stores
            constexpr int NE = (TS + 2) * (TS + 2), HB = sizeof(R) == 4 ? 9 : 5;
#pragma unroll 1
            for (int e0 = tid; e0 < NE; e0 += 256 * HB) {
                cx<R> hv[HB];
#pragma unroll
                for (int j = 0; j < HB; ++j) {
                    const int e = e0 + 256 * j;
                    const int r = e / (TS + 2), c = e % (TS + 2);
                    const int p = a0 - 1 + r, q = b0 - 1 + c;
                    hv[j] = (e < NE && p >= 0 && p < nI && q >= 0 && q < nI) ? Tp[(size_t)p * nP + q] : cxzero<R>();
                }
                if (e0 == tid && tid < 2 * TS) {
                    const int which = tid / TS, idx = tid % TS;
                    cx<R> c0 = cxzero<R>(), c1 = cxzero<R>(), c2 = cxzero<R>();
                    if (which == 0) {  // L[a, a-1..a+1] (t = 0: L_i, t = 1: U_i), row form at grid row y
                        if (a0 + idx < nI) tri3<R>(planes_f, a.g, t == 0 ? TRI_L : TRI_U, false, y, a0 + idx, c0, c1, c2);
                        lc[idx][0] = c0; lc[idx][1] = c1; lc[idx][2] = c2;
                    } else {           // U[b-1..b+1, b] (t = 0: U_{i-1}, t = 1: L_{i+1}), column form
                        if (b0 + idx < nI) tri3<R>(planes_f, a.g, t == 0 ? TRI_UC : TRI_LC, false, t == 0 ? y - 1 : y + 1, b0 + idx, c0, c1, c2);
                        rc[idx][0] = c0; rc[idx][1] = c1; rc[idx][2] = c2;
                    }
                }
#pragma unroll
                for (int j = 0; j < HB; ++j) {
                    const int e = e0 + 256 * j;
                    if (e < NE) Tt[e / (TS + 2)][e % (TS + 2)] = hv[j];
                }
            }
            __syncthreads();
#pragma unroll
            for (int dx = 0; dx < PT; ++dx) {
                const int lb = tx + 16 * dx;
                const cx<R> r0 = rc[lb][0], r1 = rc[lb][1], r2 = rc[lb][2];
                cx<R> rowacc[PT + 2];  // (T_prev U)[a0 + PT*ty - 1 + p, b]
#pragma unroll
                for (int p = 0; p < PT + 2; ++p) {
                    cx<R> s = cxzero<R>();
                    cmac(s, Tt[PT * ty + p][lb], r0);
                    cmac(s, Tt[PT * ty + p][lb + 1], r1);
                    cmac(s, Tt[PT * ty + p][lb + 2], r2);
                    rowacc[p] = s;
                }
#pragma unroll
                for (int dy = 0; dy < PT; ++dy) {
                    const int la = PT * ty + dy;
                    cx<R> s = cxzero<R>();
                    cmac(s, lc[la][0], rowacc[dy]);
                    cmac(s, lc[la][1], rowacc[dy + 1]);
                    cmac(s, lc[la][2], rowacc[dy + 2]);
                    out[dy][dx] = out[dy][dx] - s;
                }
            }
        }
    }
    cx<R>* X0 = gj_buffer(a, z, freq, row, 0);
#pragma unroll
    for (int dy = 0; dy < PT; ++dy) {
        const int ai = a0 + PT * ty + dy;
        if (ai >= nP) continue;
#pragma unroll
        for (int dx = 0; dx < PT; ++dx) {
            const int bi = b0 + tx + 16 * dx;
            if (bi >= nP) continue;
            const bool live = ai < nI && bi < nI;
            X0[(size_t)ai * nP + bi] = (live || ai == bi) ? out[dy][dx] : cxzero<R>();
        }
    }
    if constexpr (sizeof(R) == 4) {
        if (pivot0 && bx == 0 && by == 0) {
            static_assert(TS == GJ_NB, "the first Schur tile must be the first pivot block");
            __syncthreads();  // the halo tile is dead: its storage becomes the block; the scratch of the blocked inversion is dynamic
            extern __shared__ __align__(16) unsigned char schur_dyn[];
            cx<R>* blk = reinterpret_cast<cx<R>*>(&Tt[0][0]);
            static_assert(sizeof(Tt) >= sizeof(cx<R>) * GJ_NB * (GJ_NB + 1), "the pivot block must fit in the halo tile");
#pragma unroll
            for (int dy = 0; dy < PT; ++dy)
#pragma unroll
                for (int dx = 0; dx < PT; ++dx) {
                    const int ai = PT * ty + dy, bi = tx + 16 * dx;
                    blk[ai * (GJ_NB + 1) + bi] = ((ai < nI && bi < nI) || ai == bi) ? out[dy][dx] : cxzero<R>();
                }
            __syncthreads();
            gj_pivot_blocked(a, z, reinterpret_cast<cx<float>*>(blk), reinterpret_cast<cx<float>*>(schur_dyn), tid);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Pivot: P = inv(X_kk) by unpivoted Gauss-Jordan, one CTA per chain (the latency-bound part of the
// factorisation: 64 dependent steps).  The block lives in REGISTERS: thread (i = tid/4, q = tid%4) holds
// columns 16q..16q+15 of row i of G = X_kk^T (the inverse of a transpose is the transpose of the inverse;
// the row-panel kernel wants P[r][kk] = G[kk][r] with unit stride).  Per step p the four owners of row p
// scale and publish it through a double-buffered shared row (ONE barrier per step); every thread takes its
// multiplier G[i][p] (the pivot itself for the owners) from its row partner with a shuffle and updates 16 entries.
// grid = (1, 1, nbatch), 256 threads, dynamic smem = gj_pivot_smem<R>().
// ---------------------------------------------------------------------------------------------
template <typename R>
constexpr int gj_pivot_qs() { return sizeof(R) == 4 ? 18 : 17; }  // padded quarter stride: the four quarters of a row land in different banks
template <typename R>
constexpr size_t gj_pivot_smem() { return sizeof(cx<R>) * (2 * 4 * gj_pivot_qs<R>() + (sizeof(R) == 4 ? GJ_NB * (GJ_NB + 1) : 0)); }

// With `sm_block` the 64 x 64 block is taken from shared memory (row stride GJ_NB + 1) instead of X: the look-ahead CTAs
// of the update launch form the next pivot block there (tc2_gj_update_kernel).
template <typename R>
__device__ __forceinline__ void gj_pivot_body(const FactorArgs<R>& a, int k, int z, unsigned char* smem_raw, const cx<R>* sm_block) {
    constexpr int QS = sizeof(R) == 4 ? 18 : 17;
    cx<R>(*rowbuf)[4 * QS] = reinterpret_cast<cx<R>(*)[4 * QS]>(smem_raw);  // [2][4 quarters][QS] scaled pivot rows, double buffered
    const int row = chain_row(a.g, a.phase, z, a.step);
    if (row < 0) return;
    const int freq = (a.f0 + chain_freq(a.phase, z));
    const int nP = a.g.nP;
    const cx<R>* __restrict__ Xc = gj_buffer(a, z, freq, row, k);
    const int k0 = k * GJ_NB;
    const int tid = threadIdx.x + threadIdx.y * blockDim.x;  // (16, 16) block when called from the Schur kernel
    const int i = tid >> 2, q = tid & 3, lane = tid & 31;
    cx<R> g[16];
    if (sm_block) {  // the region may be reused once the block is in registers
#pragma unroll
        for (int c = 0; c < 16; ++c) g[c] = sm_block[(16 * q + c) * (GJ_NB + 1) + i];
        __syncthreads();
    } else {
#pragma unroll
        for (int c = 0; c < 16; ++c) g[c] = Xc[(size_t)(k0 + 16 * q + c) * nP + k0 + i];  // G[i][16q+c] = X_kk[16q+c][i]
    }
    bool bad = false;
    if constexpr (sizeof(R) == 4) {
        // complex64: the row is held as packed pairs (re[c], re[c+1]) / (im[c], im[c+1]) and updated with the packed FP32 FMA of
        // sm_100 (fma.rn.f32x2: two IEEE FMAs per instruction), the published pivot row is SoA [re x 16 | im x 16] per quarter
        // so that a 16-byte shared-memory read yields two pairs: 32 packed FMAs + 8 reads per step instead of 64 FMAs + 8 reads.
        // The CTA is issue bound (2 warps per scheduler, ~200 instructions per step before), not latency bound.
        typedef unsigned long long u64;
        auto pk = [](float lo, float hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; };
        auto lo = [](u64 v) { float x, y; asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(v)); return x; };
        auto hi = [](u64 v) { float x, y; asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(v)); return y; };
        auto fma2 = [](u64 x, u64 y, u64 w) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(x), "l"(y), "l"(w)); return d; };
        auto mul2 = [](u64 x, u64 y) { u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(x), "l"(y)); return d; };
        constexpr int QF = 36;  // floats per quarter in the row buffer: 16 re + 16 im + 4 pad (= QS complex: same footprint)
        float(*rbf)[4 * QF] = reinterpret_cast<float(*)[4 * QF]>(smem_raw);
        u64 gre[8], gim[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { gre[j] = pk(g[2 * j].re, g[2 * j + 1].re); gim[j] = pk(g[2 * j].im, g[2 * j + 1].im); }
#pragma unroll 1
        for (int pq = 0; pq < 4; ++pq) {
#pragma unroll
            for (int pp = 0; pp < 16; ++pp) {
                const int p = 16 * pq + pp;
                float* rb = rbf[p & 1] + QF * q;
                // G[i][p] lives in register pp of the row partner that owns column quarter pq
                const float sre = (pp & 1) ? hi(gre[pp >> 1]) : lo(gre[pp >> 1]);
                const float sim = (pp & 1) ? hi(gim[pp >> 1]) : lo(gim[pp >> 1]);
                const float mre = __shfl_sync(0xffffffffu, sre, (lane & ~3) | pq);
                const float mim = __shfl_sync(0xffffffffu, sim, (lane & ~3) | pq);
                const bool own = (q == pq);
                if (i == p) {  // scale the pivot row by 1 / pivot, publish it
                    const float mag = mre * mre + mim * mim;
                    if (!(mag > 0.f) || isinf(mag)) bad = true;
                    const cx<float> ip = crecip(cx<float>(mre, mim));
                    const u64 ipre = pk(ip.re, ip.re), ipim = pk(ip.im, ip.im), nipim = pk(-ip.im, -ip.im);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const u64 nre = fma2(gim[j], nipim, mul2(gre[j], ipre));  // re*ip.re - im*ip.im
                        const u64 nim = fma2(gim[j], ipre, mul2(gre[j], ipim));   // re*ip.im + im*ip.re
                        gre[j] = nre; gim[j] = nim;
                    }
                    if (own) {  // the pivot entry itself becomes 1 / pivot
                        gre[pp >> 1] = (pp & 1) ? pk(lo(gre[pp >> 1]), ip.re) : pk(ip.re, hi(gre[pp >> 1]));
                        gim[pp >> 1] = (pp & 1) ? pk(lo(gim[pp >> 1]), ip.im) : pk(ip.im, hi(gim[pp >> 1]));
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        *reinterpret_cast<ulonglong2*>(rb + 4 * j) = make_ulonglong2(gre[2 * j], gre[2 * j + 1]);
                        *reinterpret_cast<ulonglong2*>(rb + 16 + 4 * j) = make_ulonglong2(gim[2 * j], gim[2 * j + 1]);
                    }
                }
                __syncthreads();
                if (i != p) {
                    if (own) {  // pivot column: X~ has e_p there
                        gre[pp >> 1] = (pp & 1) ? pk(lo(gre[pp >> 1]), 0.f) : pk(0.f, hi(gre[pp >> 1]));
                        gim[pp >> 1] = (pp & 1) ? pk(lo(gim[pp >> 1]), 0.f) : pk(0.f, hi(gim[pp >> 1]));
                    }
                    const u64 nmre = pk(-mre, -mre), pmim = pk(mim, mim), nmim = pk(-mim, -mim);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const ulonglong2 rr = *reinterpret_cast<const ulonglong2*>(rb + 4 * j);
                        const ulonglong2 ri = *reinterpret_cast<const ulonglong2*>(rb + 16 + 4 * j);
                        gre[2 * j] = fma2(pmim, ri.x, fma2(nmre, rr.x, gre[2 * j]));          // re -= m.re*r.re - m.im*r.im
                        gre[2 * j + 1] = fma2(pmim, ri.y, fma2(nmre, rr.y, gre[2 * j + 1]));
                        gim[2 * j] = fma2(nmim, rr.x, fma2(nmre, ri.x, gim[2 * j]));          // im -= m.re*r.im + m.im*r.re
                        gim[2 * j + 1] = fma2(nmim, rr.y, fma2(nmre, ri.y, gim[2 * j + 1]));
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            g[2 * j] = cx<R>(lo(gre[j]), lo(gim[j]));
            g[2 * j + 1] = cx<R>(hi(gre[j]), hi(gim[j]));
        }
    } else {
#pragma unroll 1
    for (int pq = 0; pq < 4; ++pq) {
#pragma unroll
        for (int pp = 0; pp < 16; ++pp) {
            const int p = 16 * pq + pp;
            cx<R>* rb = rowbuf[p & 1];
            // G[i][p] lives in register pp of the row partner that owns column quarter pq: the multiplier of row i,
            // and for the owners of row p the pivot itself
            cx<R> m;
            m.re = __shfl_sync(0xffffffffu, g[pp].re, (lane & ~3) | pq);
            m.im = __shfl_sync(0xffffffffu, g[pp].im, (lane & ~3) | pq);
            const bool own = (q == pq);
            if (i == p) {  // scale the pivot row, publish it
                const R mag = m.re * m.re + m.im * m.im;
                if (!(mag > R(0)) || isinf(mag)) bad = true;  // zero, NaN or overflowing pivot
                const cx<R> ip = crecip(m);
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    g[c] = (own && c == pp) ? ip : g[c] * ip;
                    rb[QS * q + c] = g[c];
                }
            }
            __syncthreads();
            if (i != p) {
                if (own) g[pp] = cxzero<R>();  // pivot column: X~ has e_p there
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const cx<R> rj = rb[QS * q + c];
                    g[c].re = fma(-m.re, rj.re, g[c].re); g[c].re = fma(m.im, rj.im, g[c].re);
                    g[c].im = fma(-m.re, rj.im, g[c].im); g[c].im = fma(-m.im, rj.re, g[c].im);
                }
            }
        }
    }
    }
    if (bad) atomicOr(a.status, 1);
    if constexpr (sizeof(R) == 4) {
        if (a.Pp) {
            // TMA-fed engine: P goes out as bf16 x 3 A planes.  g holds G = P^T (thread = column of P), a 16-byte plane
            // chunk is 8 consecutive columns of one row of P: transpose through shared memory.
            cx<R>(*tileP)[GJ_NB + 1] = reinterpret_cast<cx<R>(*)[GJ_NB + 1]>(smem_raw + sizeof(cx<R>) * 2 * 4 * QS);
            __syncthreads();
#pragma unroll
            for (int c = 0; c < 16; ++c) tileP[i][16 * q + c] = g[c];  // tileP[col of P][row of P]
            __syncthreads();
            uint16_t* dstm = a.Pp + (size_t)(a.zb0 + z) * tc2::NPL_A * GJ_NB * GJ_NB;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int e = tid + 256 * h;
                const int r = e & 63, J = e >> 6;
                float re[8], im[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) { cx<R> v = tileP[8 * J + c][r]; re[c] = v.re; im[c] = v.im; }
                tc2::store_a8(dstm + ((size_t)(r >> 3) * 8 + J) * 64 + (r & 7) * 8, (size_t)GJ_NB * GJ_NB, re, im);
            }
            return;
        }
    }
    cx<R>* Pg = a.pbuf + (size_t)(a.zb0 + z) * GJ_NB * GJ_NB;
#pragma unroll
    for (int c = 0; c < 16; ++c) Pg[i * GJ_NB + 16 * q + c] = g[c];
}

// ---------------------------------------------------------------------------------------------
// Blocked pivot inversion (TMA-fed engine, complex64): P = inv(X_kk), 64 x 64, in place in shared memory.
//
// The register version above runs 64 strictly sequential steps of ~200 instructions with a CTA barrier each (33 us alone,
// 48 us next to a tile CTA): it is the critical path of an update launch as soon as the batch is small (strong scaling,
// one frequency per GPU) and holds one CTA slot per chain for most of the launch otherwise.  Here the same unpivoted
// Gauss-Jordan elimination is blocked by 16: per block step the CTA inverts the 16 x 16 diagonal block (inv16_cta: one entry
// per thread, 16 sequential steps of one barrier each), then forms the row panel R = P_bb * A~[b,:] and applies the rank-16
// update A~ - A[:,b] R as register-tiled complex GEMMs on packed FP32 FMAs -- 4 x fewer instructions than the unblocked
// form.  Mathematically the same elimination order as the unblocked form; rounding differs.
//   A       [64][65] complex, holds X_kk on entry and P on exit
//   scratch Pbuf [16][17] | Pbuf2 [16][17] | Cbuf [64][17] | Rbuf [16][65]      (gj_pivot2_scratch_bytes)
// ---------------------------------------------------------------------------------------------
constexpr int PB = 16;
constexpr int PV_LD = GJ_NB + 1;
constexpr size_t gj_pivot2_scratch_elems = 2 * PB * (PB + 1) + GJ_NB * (PB + 1) + PB * PV_LD;
constexpr size_t gj_pivot2_scratch_bytes = sizeof(cx<float>) * gj_pivot2_scratch_elems;
constexpr size_t gj_pivot2_smem_bytes = sizeof(cx<float>) * GJ_NB * PV_LD + gj_pivot2_scratch_bytes;  // block + scratch (stand-alone pivot CTAs)

typedef unsigned long long u64p;  // two packed FP32 values: (re, im) of one complex number, or a broadcast pair
__device__ __forceinline__ u64p pk2(float lo, float hi) { u64p r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpk2(u64p v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ u64p fma2p(u64p x, u64p y, u64p w) { u64p d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(x), "l"(y), "l"(w)); return d; }

// Inverse of a 16 x 16 complex block by the whole CTA (256 threads = one entry each), unpivoted Gauss-Jordan.  An earlier form ran
// on one warp (row per lane pair, pivot row published through shared memory, __syncwarp per step): a lone warp exposes the latency
// of every instruction of its ~100-instruction step (3.1-5.5 us per block alone, 5-10 us next to a tile CTA: 17 of the 28 us of a
// pivot inversion); with one entry per thread a step is three broadcast reads, the reciprocal, two multiply-adds, one store and one
// barrier.  The block ping-pongs between two shared buffers (read step p from buf[p & 1], write buf[(p + 1) & 1]), so one
// barrier per step suffices; after 16 steps the inverse is back in buf0.  Returns true on a zero / non-finite pivot.
__device__ __forceinline__ bool inv16_cta(const cx<float>* __restrict__ src, int ld, cx<float>* __restrict__ buf0, cx<float>* __restrict__ buf1, int tid) {
    typedef cx<float> C;
    const int r = tid >> 4, c = tid & 15;
    constexpr int LD = PB + 1;
    C v = src[r * ld + c];
    buf0[r * LD + c] = v;
    __syncthreads();
    bool bad = false;
#pragma unroll
    for (int p = 0; p < PB; ++p) {
        const C* __restrict__ s = (p & 1) ? buf1 : buf0;
        C* __restrict__ d = (p & 1) ? buf0 : buf1;
        const C piv = s[p * LD + p], m = s[r * LD + p], pr = s[p * LD + c];
        const float mag = piv.re * piv.re + piv.im * piv.im;
        if (!(mag > 0.f) || isinf(mag)) bad = true;
        const float sc = __frcp_rn(mag);  // correctly rounded, like 1.f / mag
        const C ip(piv.re * sc, -piv.im * sc);
        const C sv = (c == p) ? ip : pr * ip;  // scaled pivot row, the pivot entry itself becomes 1 / pivot
        if (r == p) {
            v = sv;
        } else {
            if (c == p) v = cxzero<float>();   // pivot column: A~ has e_p there
            v.re = fmaf(-m.re, sv.re, v.re); v.re = fmaf(m.im, sv.im, v.re);
            v.im = fmaf(-m.re, sv.im, v.im); v.im = fmaf(-m.im, sv.re, v.im);
        }
        d[r * LD + c] = v;
        __syncthreads();
    }
    return bad;
}

__device__ __forceinline__ void gj_pivot_blocked(const FactorArgs<float>& a, int z, cx<float>* __restrict__ A, cx<float>* __restrict__ scratch, int tid,
                                                 unsigned long long* stamps = nullptr) {
    typedef cx<float> C;
    // debugging (UST_TC2_TRACE_UPDATE): phase stamps of the traced launch's pivot CTAs: [0] start, then per block step: diagonal
    // block inverted, panels formed, update applied
#define PIV_STAMP(i) do { if (stamps && tid == 0) stamps[i] = tc2::gtime(); } while (0)
    PIV_STAMP(0);
    C* Pbuf = scratch;                          // [16][17]
    C* Pbuf2 = Pbuf + PB * (PB + 1);            // [16][17] ping-pong partner of Pbuf during the diagonal-block inversion
    C* Cbuf = Pbuf2 + PB * (PB + 1);            // [64][17]
    C* Rbuf = Cbuf + GJ_NB * (PB + 1);          // [16][65]
    const int ty = tid >> 4, tx = tid & 15;
    bool bad = false;
#pragma unroll 1
    for (int b = 0; b < GJ_NB / PB; ++b) {
        const int b0 = PB * b;
        bad |= inv16_cta(A + b0 * PV_LD + b0, PV_LD, Pbuf, Pbuf2, tid);  // ends with a barrier
        PIV_STAMP(1 + 3 * b);
        // column panel C = A[:, b] -> Cbuf (the update overwrites those entries), row panel R = P * A~[b, :] -> Rbuf
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int i = tid >> 2, kk = (tid & 3) * 4 + j;
            Cbuf[i * (PB + 1) + kk] = A[i * PV_LD + b0 + kk];
        }
        {
            C acc[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[j] = cxzero<float>();
#pragma unroll
            for (int kk = 0; kk < PB; ++kk) {
                const C pv = Pbuf[ty * (PB + 1) + kk];
#pragma unroll
                for (int j = 0; j < 4; ++j) cmac(acc[j], pv, A[(b0 + kk) * PV_LD + tx + 16 * j]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) Rbuf[ty * PV_LD + tx + 16 * j] = (j == b) ? Pbuf[ty * (PB + 1) + tx] : acc[j];  // A~[b, b] = I
        }
        __syncthreads();
        PIV_STAMP(2 + 3 * b);
        // rows of block b take R (4 entries per thread); every other row i: A[i, :] <- A~[i, :] - C[i, :] R with A~[i, b-columns] = 0.
        // The 48 other rows are dealt 3 per thread (x 4 columns) so that all eight warps carry the same load (with 4 rows per
        // thread the two warps that own block b's rows idled through the phase and the other six set its length).
#pragma unroll
        for (int j = 0; j < 4; ++j) A[(b0 + ty) * PV_LD + tx + 16 * j] = Rbuf[ty * PV_LD + tx + 16 * j];
        {
            int rws[3];
#pragma unroll
            for (int ri = 0; ri < 3; ++ri) { const int r3 = 3 * ty + ri; rws[ri] = r3 + (r3 >= b0 ? PB : 0); }
            u64p acc[3][4];
#pragma unroll
            for (int ri = 0; ri < 3; ++ri)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const C v = (j == b) ? cxzero<float>() : A[rws[ri] * PV_LD + tx + 16 * j];
                    acc[ri][j] = pk2(v.re, v.im);
                }
#pragma unroll 4
            for (int kk = 0; kk < PB; ++kk) {
                u64p rv[4], rs[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const C v = Rbuf[kk * PV_LD + tx + 16 * j];
                    rv[j] = pk2(v.re, v.im);     // ( r.re,  r.im)
                    rs[j] = pk2(-v.im, v.re);    // (-r.im,  r.re)
                }
#pragma unroll
                for (int ri = 0; ri < 3; ++ri) {
                    const C cv = Cbuf[rws[ri] * (PB + 1) + kk];
                    const u64p cr = pk2(-cv.re, -cv.re), ci = pk2(-cv.im, -cv.im);
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[ri][j] = fma2p(ci, rs[j], fma2p(cr, rv[j], acc[ri][j]));  // -= c * r
                }
            }
#pragma unroll
            for (int ri = 0; ri < 3; ++ri)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    C v;
                    unpk2(acc[ri][j], v.re, v.im);
                    A[rws[ri] * PV_LD + tx + 16 * j] = v;
                }
        }
        __syncthreads();
        PIV_STAMP(3 + 3 * b);
    }
    if (bad && tid == 0) atomicOr(a.status, 1);
    // P goes out as bf16 x 3 A planes: a 16-byte plane chunk is 8 consecutive columns of one row of P
    uint16_t* dstm = a.Pp + (size_t)(a.zb0 + z) * tc2::NPL_A * GJ_NB * GJ_NB;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int e = tid + 256 * h;
        const int r = e & 63, J = e >> 6;
        float re[8], im[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) { const C v = A[r * PV_LD + 8 * J + c]; re[c] = v.re; im[c] = v.im; }
        tc2::store_a8(dstm + ((size_t)(r >> 3) * 8 + J) * 64 + (r & 7) * 8, (size_t)GJ_NB * GJ_NB, re, im);
    }
}

// stand-alone form: the block is fetched from X^(k) in global memory first (pivot launches without look-ahead)
__device__ __forceinline__ void gj_pivot_blocked_global(const FactorArgs<float>& a, int k, int z, unsigned char* smem_raw, int tid) {
    const int row = chain_row(a.g, a.phase, z, a.step);
    if (row < 0) return;
    const int freq = a.f0 + chain_freq(a.phase, z);
    const int nP = a.g.nP, k0 = k * GJ_NB;
    const cx<float>* __restrict__ Xc = gj_buffer(a, z, freq, row, k);
    cx<float>* A = reinterpret_cast<cx<float>*>(smem_raw);
    for (int e = tid; e < GJ_NB * GJ_NB; e += 256) A[(e >> 6) * PV_LD + (e & 63)] = Xc[(size_t)(k0 + (e >> 6)) * nP + k0 + (e & 63)];
    __syncthreads();
    gj_pivot_blocked(a, z, A, A + GJ_NB * PV_LD, tid);
}

// complex128 form of the blocked pivot inversion (stand-alone launches: the complex128 path has no look-ahead): the same
// elimination as gj_pivot_blocked -- 16 x 16 diagonal blocks inverted by the whole CTA with one entry per thread and a barrier per
// scalar step, row / column panels, rank-16 update dealt 3 rows per thread -- in FP64 FMAs.  The register version it replaces
// (gj_pivot_body, 64 CTA-wide steps of ~200 instructions) took 49 us per launch, a quarter of a complex128 evaluation.
//   smem: A [64][65] | Pbuf, Pbuf2 [16][17] | Cbuf [64][17] | Rbuf [16][65]   complex128  (gj_pivot_f64_smem_bytes)
constexpr size_t gj_pivot_f64_smem_bytes = sizeof(cx<double>) * (GJ_NB * PV_LD + 2 * PB * (PB + 1) + GJ_NB * (PB + 1) + PB * PV_LD);
// With `form` the kernel runs one pivot step AHEAD, beside update k-1 on a side stream: the block is not read from X^(k) (which that
// update is still writing) but formed from X^(k-1), which the update only reads (the FMA path ping-pongs between two buffers),
// and the row panel R_{k-1} already in place:  X^(k)_kk = X^(k-1)_kk - X^(k-1)_{k,k-1} R_{k-1}[:, k]  as four rank-16 updates
// staged through the panel buffers.  Not bit-identical to what update k-1 writes for that block (different summation order,
// ~1e-16 relative) -- immaterial at complex128's 1e-10 bar, where the complex64 path needs the same arithmetic (DESIGN 4.2).
__device__ __forceinline__ void gj_pivot_blocked_f64(const FactorArgs<double>& a, int k, int z, unsigned char* smem_raw, int tid, int form) {
    typedef cx<double> C;
    const int row = chain_row(a.g, a.phase, z, a.step);
    if (row < 0) return;
    const int freq = a.f0 + chain_freq(a.phase, z);
    const int nP = a.g.nP, k0 = k * GJ_NB;
    const C* __restrict__ Xc = gj_buffer(a, z, freq, row, form ? k - 1 : k);
    C* A = reinterpret_cast<C*>(smem_raw);
    C* Pbuf = A + GJ_NB * PV_LD;
    C* Pbuf2 = Pbuf + PB * (PB + 1);
    C* Cbuf = Pbuf2 + PB * (PB + 1);
    C* Rbuf = Cbuf + GJ_NB * (PB + 1);
    const int ty = tid >> 4, tx = tid & 15;
    for (int e = tid; e < GJ_NB * GJ_NB; e += 256) A[(e >> 6) * PV_LD + (e & 63)] = Xc[(size_t)(k0 + (e >> 6)) * nP + k0 + (e & 63)];
    if (form) {
        const C* __restrict__ Xn = gj_buffer(a, z, freq, row, k);  // holds R_{k-1} in block row k-1
        const int km = k0 - GJ_NB;
#pragma unroll 1
        for (int kc = 0; kc < GJ_NB / PB; ++kc) {
            __syncthreads();
            for (int e = tid; e < GJ_NB * PB; e += 256) Cbuf[(e >> 4) * (PB + 1) + (e & 15)] = Xc[(size_t)(k0 + (e >> 4)) * nP + km + PB * kc + (e & 15)];
            for (int e = tid; e < PB * GJ_NB; e += 256) Rbuf[(e >> 6) * PV_LD + (e & 63)] = Xn[(size_t)(km + PB * kc + (e >> 6)) * nP + k0 + (e & 63)];
            __syncthreads();
            C acc[4][4];  // rows 4 ty .., columns tx + 16 j
#pragma unroll
            for (int ri = 0; ri < 4; ++ri)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[ri][j] = A[(4 * ty + ri) * PV_LD + tx + 16 * j];
#pragma unroll 4
            for (int kk = 0; kk < PB; ++kk) {
                C rv[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) rv[j] = Rbuf[kk * PV_LD + tx + 16 * j];
#pragma unroll
                for (int ri = 0; ri < 4; ++ri) {
                    const C cv = Cbuf[(4 * ty + ri) * (PB + 1) + kk];
                    const C ncv(-cv.re, -cv.im);
#pragma unroll
                    for (int j = 0; j < 4; ++j) cmac(acc[ri][j], ncv, rv[j]);
                }
            }
#pragma unroll
            for (int ri = 0; ri < 4; ++ri)
#pragma unroll
                for (int j = 0; j < 4; ++j) A[(4 * ty + ri) * PV_LD + tx + 16 * j] = acc[ri][j];
        }
    }
    __syncthreads();
    bool bad = false;
#pragma unroll 1
    for (int b = 0; b < GJ_NB / PB; ++b) {
        const int b0 = PB * b;
        {   // diagonal block b: one entry per thread, ping-pong Pbuf / Pbuf2, one barrier per step; the inverse ends in Pbuf
            constexpr int LD = PB + 1;
            C v = A[(b0 + ty) * PV_LD + b0 + tx];
            Pbuf[ty * LD + tx] = v;
            __syncthreads();
#pragma unroll
            for (int p = 0; p < PB; ++p) {
                const C* __restrict__ s = (p & 1) ? Pbuf2 : Pbuf;
                C* __restrict__ d = (p & 1) ? Pbuf : Pbuf2;
                const C piv = s[p * LD + p], m = s[ty * LD + p], pr = s[p * LD + tx];
                const double mag = piv.re * piv.re + piv.im * piv.im;
                if (!(mag > 0.0) || isinf(mag)) bad = true;
                const C ip = crecip(piv);
                const C sv = (tx == p) ? ip : pr * ip;
                if (ty == p) {
                    v = sv;
                } else {
                    if (tx == p) v = cxzero<double>();
                    v.re = fma(-m.re, sv.re, v.re); v.re = fma(m.im, sv.im, v.re);
                    v.im = fma(-m.re, sv.im, v.im); v.im = fma(-m.im, sv.re, v.im);
                }
                d[ty * LD + tx] = v;
                __syncthreads();
            }
        }
        // column panel C = A[:, b] -> Cbuf, row panel R = P * A~[b, :] -> Rbuf
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int i = tid >> 2, kk = (tid & 3) * 4 + j;
            Cbuf[i * (PB + 1) + kk] = A[i * PV_LD + b0 + kk];
        }
        {
            C acc[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[j] = cxzero<double>();
#pragma unroll
            for (int kk = 0; kk < PB; ++kk) {
                const C pv = Pbuf[ty * (PB + 1) + kk];
#pragma unroll
                for (int j = 0; j < 4; ++j) cmac(acc[j], pv, A[(b0 + kk) * PV_LD + tx + 16 * j]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) Rbuf[ty * PV_LD + tx + 16 * j] = (j == b) ? Pbuf[ty * (PB + 1) + tx] : acc[j];  // A~[b, b] = I
        }
        __syncthreads();
        // rows of block b take R; the 48 other rows (3 per thread): A[i, :] <- A~[i, :] - C[i, :] R with A~[i, b-columns] = 0
#pragma unroll
        for (int j = 0; j < 4; ++j) A[(b0 + ty) * PV_LD + tx + 16 * j] = Rbuf[ty * PV_LD + tx + 16 * j];
        {
            int rws[3];
#pragma unroll
            for (int ri = 0; ri < 3; ++ri) { const int r3 = 3 * ty + ri; rws[ri] = r3 + (r3 >= b0 ? PB : 0); }
            C acc[3][4];
#pragma unroll
            for (int ri = 0; ri < 3; ++ri)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[ri][j] = (j == b) ? cxzero<double>() : A[rws[ri] * PV_LD + tx + 16 * j];
#pragma unroll 4
            for (int kk = 0; kk < PB; ++kk) {
                C rv[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) rv[j] = Rbuf[kk * PV_LD + tx + 16 * j];
#pragma unroll
                for (int ri = 0; ri < 3; ++ri) {
                    const C cv = Cbuf[rws[ri] * (PB + 1) + kk];
                    const C ncv(-cv.re, -cv.im);
#pragma unroll
                    for (int j = 0; j < 4; ++j) cmac(acc[ri][j], ncv, rv[j]);  // -= c * r
                }
            }
#pragma unroll
            for (int ri = 0; ri < 3; ++ri)
#pragma unroll
                for (int j = 0; j < 4; ++j) A[rws[ri] * PV_LD + tx + 16 * j] = acc[ri][j];
        }
        __syncthreads();
    }
    if (bad && tid == 0) atomicOr(a.status, 1);
    // the row-panel kernel wants G = P^T: Pg[i][j] = P[j][i]
    C* Pg = a.pbuf + (size_t)(a.zb0 + z) * GJ_NB * GJ_NB;
    for (int e = tid; e < GJ_NB * GJ_NB; e += 256) Pg[e] = A[(e & 63) * PV_LD + (e >> 6)];
}

template <typename R>
__global__ void __launch_bounds__(256, 1) gj_pivot_kernel(FactorArgs<R> a, int k, int form = 0) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    pdl_trigger();
    pdl_wait();
    if constexpr (sizeof(R) == 4) {
        if (a.Pp) { gj_pivot_blocked_global(a, k, blockIdx.z, smem_raw, threadIdx.x); return; }
        gj_pivot_body<R>(a, k, blockIdx.z, smem_raw, nullptr);
    } else {
        gj_pivot_blocked_f64(a, k, blockIdx.z, smem_raw, threadIdx.x, form);
    }
}

// Row panel: R_j = P * Xtilde_kj written into block row k of X'.  grid = (nblk, 1, nbatch), 256 threads,
// dynamic smem = 2 * 64x64 complex.
template <typename R>
constexpr size_t gj_rowpanel_smem() {  // double: four planes (re / im of G and of the tile), rows padded by 8 (DMMA fragment loads)
    return sizeof(R) == 8 ? 4 * sizeof(double) * GJ_NB * (GJ_NB + 8) : 2 * sizeof(cx<R>) * GJ_NB * GJ_NB;
}
template <typename R>
__global__ void __launch_bounds__(256) gj_rowpanel_kernel(FactorArgs<R> a, int k) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int z = blockIdx.z;
    const int row = chain_row(a.g, a.phase, z, a.step);
    if (row < 0) return;
    const int freq = (a.f0 + chain_freq(a.phase, z));
    const int nP = a.g.nP;
    const cx<R>* __restrict__ Xc = gj_buffer(a, z, freq, row, k);
    cx<R>* __restrict__ Xn = gj_buffer(a, z, freq, row, k + 1);
    const cx<R>* __restrict__ Pg = a.pbuf + (size_t)(a.zb0 + z) * GJ_NB * GJ_NB;
    const int k0 = k * GJ_NB, j0 = blockIdx.x * GJ_NB;
    const int tid = threadIdx.x;
    if constexpr (sizeof(R) == 8) {
        // complex128: the 64 x 64 x 64 product on the FP64 tensor-core instruction (see gemm_simt.cuh): A[m][kk] = P[m][kk] =
        // G[kk][m] (the pivot kernel stores G = P^T), B[kk][n] = X~_kj[kk][n]; warp grid 2 x 4, a warp owns 4 x 2 tiles of 8 x 8
        constexpr int LD = GJ_NB + 8;
        double(*Gr)[LD] = reinterpret_cast<double(*)[LD]>(smem_raw);
        double(*Gi)[LD] = Gr + GJ_NB;
        double(*Tr)[LD] = Gi + GJ_NB;
        double(*Ti)[LD] = Tr + GJ_NB;
        for (int e = tid; e < GJ_NB * GJ_NB; e += 256) {
            const int r = e / GJ_NB, c = e % GJ_NB;
            const cx<R> g = Pg[e];
            Gr[r][c] = g.re; Gi[r][c] = g.im;
            cx<R> tv;
            if (j0 == k0) tv = (r == c) ? cxone<R>() : cxzero<R>();
            else tv = Xc[(size_t)(k0 + r) * nP + j0 + c];
            Tr[r][c] = tv.re; Ti[r][c] = tv.im;
        }
        __syncthreads();
        const int lane = tid & 31, warp = tid >> 5;
        const int wm = (warp & 1) * 32, wn = (warp >> 1) * 16, fr = lane >> 2, fk = lane & 3;
        double cr[4][2][2], ci[4][2][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) { cr[i][j][0] = cr[i][j][1] = 0.0; ci[i][j][0] = ci[i][j][1] = 0.0; }
#pragma unroll 4
        for (int k4 = 0; k4 < GJ_NB; k4 += 4) {
            double ar[4], ai[4], br[2], bi[2], nbi[2];
#pragma unroll
            for (int i = 0; i < 4; ++i) { ar[i] = Gr[k4 + fk][wm + 8 * i + fr]; ai[i] = Gi[k4 + fk][wm + 8 * i + fr]; }
#pragma unroll
            for (int j = 0; j < 2; ++j) { br[j] = Tr[k4 + fk][wn + 8 * j + fr]; bi[j] = Ti[k4 + fk][wn + 8 * j + fr]; nbi[j] = -bi[j]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    dmma884(cr[i][j][0], cr[i][j][1], ar[i], br[j]);
                    dmma884(cr[i][j][0], cr[i][j][1], ai[i], nbi[j]);
                    dmma884(ci[i][j][0], ci[i][j][1], ar[i], bi[j]);
                    dmma884(ci[i][j][0], ci[i][j][1], ai[i], br[j]);
                }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q)
                    Xn[(size_t)(k0 + wm + 8 * i + fr) * nP + j0 + wn + 8 * j + 2 * fk + q] = cx<R>(cr[i][j][q], ci[i][j][q]);
        return;
    } else {
    cx<R>(*G)[GJ_NB] = reinterpret_cast<cx<R>(*)[GJ_NB]>(smem_raw);                                   // G[kk][r] = P[r][kk]
    cx<R>(*Tl)[GJ_NB] = reinterpret_cast<cx<R>(*)[GJ_NB]>(smem_raw + sizeof(cx<R>) * GJ_NB * GJ_NB);  // Xtilde_kj tile
    for (int e = tid; e < GJ_NB * GJ_NB; e += 256) {
        int r = e / GJ_NB, c = e % GJ_NB;
        G[r][c] = Pg[e];
        cx<R> tv;
        if (j0 == k0) tv = (r == c) ? cxone<R>() : cxzero<R>();
        else tv = Xc[(size_t)(k0 + r) * nP + j0 + c];
        Tl[r][c] = tv;
    }
    __syncthreads();
    const int tx = tid & 15, ty = tid >> 4;
    cx<R> acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) acc[i][jj] = cxzero<R>();
#pragma unroll 8
    for (int kk = 0; kk < GJ_NB; ++kk) {
        cx<R> av[4], bv[4];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            av[2 * c] = G[kk][c * 32 + ty * 2];
            av[2 * c + 1] = G[kk][c * 32 + ty * 2 + 1];
            bv[2 * c] = Tl[kk][c * 32 + tx * 2];
            bv[2 * c + 1] = Tl[kk][c * 32 + tx * 2 + 1];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) cmac(acc[i][jj], av[i], bv[jj]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int r = (i >> 1) * 32 + ty * 2 + (i & 1);
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
            int c = (jj >> 1) * 32 + tx * 2 + (jj & 1);
            Xn[(size_t)(k0 + r) * nP + j0 + c] = acc[i][jj];
        }
    }
    }
}

// X'_ij = Xtilde_ij - X_ik R_j for block rows i != k.  grid = (nblk, nblk-1, nbatch).
template <typename R>
__global__ void __launch_bounds__(256) gj_update_kernel(FactorArgs<R> a, int k) {
    __shared__ GemmSmem<R, GJ_NB, GJ_NB> sm;
    const int z = blockIdx.z;
    const int row = chain_row(a.g, a.phase, z, a.step);
    if (row < 0) return;
    const int freq = (a.f0 + chain_freq(a.phase, z));
    const int nP = a.g.nP;
    const cx<R>* Xc = gj_buffer(a, z, freq, row, k);
    cx<R>* Xn = gj_buffer(a, z, freq, row, k + 1);
    const int ib = blockIdx.y + (blockIdx.y >= k ? 1 : 0);
    GemmTile<R> t;
    t.A = Xc + k * GJ_NB; t.lda = nP;
    t.B = Xn + (size_t)k * GJ_NB * nP; t.ldb = nP;
    t.Cin = Xc; t.ldcin = nP;
    t.Cout = Xn; t.ldc = nP;
    t.M = nP; t.N = nP; t.K = GJ_NB; t.Mstore = nP;
    t.m0 = ib * GJ_NB; t.n0 = blockIdx.x * GJ_NB;
    t.mask_lo = k * GJ_NB; t.mask_hi = (k + 1) * GJ_NB;
    t.sgn = R(-1);
    cgemm_tile<R, GJ_NB, GJ_NB, false>(t, sm);
}

// Column panel X_:,k (nP x 64, FP32) -> bf16 x 3 A planes of the TMA-fed update.  grid = (nP/32, 1, nbatch), 256 threads:
// thread = (block row I, block column J, row r in the block), a warp writes 512 contiguous bytes per plane.
__device__ __forceinline__ void gj_colsplit_body(const FactorArgs<float>& a, int k, int z, int bx, int tid) {
    const int row = chain_row(a.g, a.phase, z, a.step);
    if (row < 0) return;
    const int freq = (a.f0 + chain_freq(a.phase, z));
    const int nP = a.g.nP;
    const cx<float>* __restrict__ Xc = gj_buffer(a, z, freq, row, k);
    const int I = bx * 4 + (tid >> 6), J = (tid >> 3) & 7, r = tid & 7;
    const int rr = I * 8 + r;
    if (rr >= nP) return;
    const cx<float>* src = Xc + (size_t)rr * nP + k * GJ_NB + J * 8;
    float re[8], im[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) { cx<float> v = src[c]; re[c] = v.re; im[c] = v.im; }
    uint32_t wr[3][4], wi[3][4];
#pragma unroll
    for (int qd = 0; qd < 4; ++qd) {
        tc::Split3 sr = tc::split2(re[2 * qd], re[2 * qd + 1]);
        tc::Split3 si = tc::split2(im[2 * qd], im[2 * qd + 1]);
#pragma unroll
        for (int sp = 0; sp < 3; ++sp) { wr[sp][qd] = sr.w[sp]; wi[sp][qd] = si.w[sp]; }
    }
    const size_t plane = (size_t)nP * GJ_NB;  // elements per plane
    uint16_t* dst = a.Cp + ((size_t)(k & 1) * a.nbmax + a.zb0 + z) * tc2::NPL_A * plane + ((size_t)I * 8 + J) * 64 + r * 8;
#pragma unroll
    for (int sp = 0; sp < 3; ++sp) {
        *reinterpret_cast<uint4*>(dst + sp * plane) = make_uint4(wr[sp][0], wr[sp][1], wr[sp][2], wr[sp][3]);
        *reinterpret_cast<uint4*>(dst + (3 + sp) * plane) = make_uint4(wi[sp][0], wi[sp][1], wi[sp][2], wi[sp][3]);
    }
}

// k = 0 preparation of the TMA-fed engine in ONE launch (pivot block 0 is inverted by the Schur launch): CTA role by blockIdx.x --
//   [0, nrow)            B planes of the pivot block row 0 (gj_rowsplit, 128 columns per CTA)
//   [nrow, nrow + ncol)  A planes of block column 0 (gj_colsplit, 32 rows per CTA)
// grid = (nrow + ncol, 1, nbatch), 256 threads.
__device__ __forceinline__ void gj_rowsplit_body(const FactorArgs<float>& a, int k, int z, int tn, int r);
__global__ void __launch_bounds__(256) gj_k0_kernel(FactorArgs<float> a, int nrow) {
    pdl_trigger();
    pdl_wait();
    const int z = blockIdx.z, bx = blockIdx.x;
    if (bx < nrow) {
        if (threadIdx.x < 128) gj_rowsplit_body(a, 0, z, bx, threadIdx.x);
    } else {
        gj_colsplit_body(a, 0, z, bx - nrow, threadIdx.x);
    }
}

// Pivot block row of X^(k) (64 x nP, FP32) with block column k replaced by the identity -> B planes Xp of the TMA-fed
// row panel.  Only used for k = 0 (later block rows are emitted by the update kernel's epilogue).
// grid = (ceil(nP/128), 1, nbatch), 128 threads: thread = column, loop over the 8 groups of 8 rows.
__device__ __forceinline__ void gj_rowsplit_body(const FactorArgs<float>& a, int k, int z, int tn, int r) {
    const int row = chain_row(a.g, a.phase, z, a.step);
    if (row < 0) return;
    const int freq = (a.f0 + chain_freq(a.phase, z));
    const int nP = a.g.nP;
    const cx<float>* __restrict__ Xc = gj_buffer(a, z, freq, row, k);
    const int k0 = k * GJ_NB;
    const int n = tn * tc2::TN + r;
    uint16_t* base = a.Xp + ((size_t)(k & 1) * a.nbmax + a.zb0 + z) * a.rp_stride;
    for (int kg = 0; kg < 8; ++kg) {
        float re[8], im[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            cx<float> v = cxzero<float>();
            if (n < nP) {
                if (n >= k0 && n < k0 + GJ_NB) v = cx<float>((n - k0 == 8 * kg + c) ? 1.f : 0.f, 0.f);
                else v = Xc[(size_t)(k0 + 8 * kg + c) * nP + n];
            }
            re[c] = v.re; im[c] = v.im;
        }
        tc2::store_b8(base + ((size_t)tn * (GJ_NB / tc2::KC) + (kg >> 1)) * (tc2::B_STAGE / 2), r, kg & 1, re, im);
    }
}

// emission targets shared by the two TMA-fed Gauss-Jordan kernels: the next column panel (or, after the last block
// step, the finished inverse as sweep operand planes)
__device__ __forceinline__ void gj_emit_a(const FactorArgs<float>& a, tc2::Tc2Tile& t, int z, int freq, int row, int k, int row_off) {
    const int nP = a.g.nP, nblk = nP / GJ_NB;
    t.ea_row_off = row_off;
    if (k + 1 < nblk) {
        const size_t plane = (size_t)nP * GJ_NB;
        t.ea_planes = a.Cp + ((size_t)((k + 1) & 1) * a.nbmax + a.zb0 + z) * tc2::NPL_A * plane;
        t.ea_plane_elems = (unsigned)plane; t.ea_nbc = GJ_NB / 8;
        t.ea_n_lo = (k + 1) * GJ_NB; t.ea_n_hi = (k + 2) * GJ_NB; t.ea_col_off = (k + 1) * GJ_NB;
        t.ea_zero_from = 0x7fffffff;
    } else {
        const size_t mat = (size_t)freq * a.g.M + row;
        t.ea_planes = a.Tp + mat * (size_t)tc2::NPL_A * nP * nP;
        t.ea_plane_elems = (unsigned)(nP * nP); t.ea_nbc = nP / 8;
        t.ea_n_lo = 0; t.ea_n_hi = nP; t.ea_col_off = 0;
        t.ea_zero_from = a.g.nI;
    }
}

// TMA-fed tensor-core row panel: R = P * Xtilde_k,: -> block row k of X' (FP32), B planes of R for the update and the
// rows of the next column panel that lie in block row k.  One 64 x 64 tile (block column blockIdx.x) per CTA on the
// two-CTAs-per-SM form of the engine (gemm_tc2h.cuh): grid = (nP/64 [+1 snapshot CTA], 1, nbatch), 256 threads.
__global__ void __launch_bounds__(tc2::NUM_THREADS_H, 2)
tc2_gj_rowpanel_kernel(FactorArgs<float> a, int k, float bias_fix, const __grid_constant__ CUtensorMap pmap) {
    extern __shared__ __align__(1024) unsigned char tc2_smem[];
    constexpr int TW = tc2::TNH;
    pdl_trigger();
    const int z = blockIdx.z;
    const int row = chain_row(a.g, a.phase, z, a.step);
    if (row < 0) { pdl_wait(); return; }  // an early exit must not let the grid complete before its predecessor
    const int freq = (a.f0 + chain_freq(a.phase, z));
    const int nP = a.g.nP;
    if (blockIdx.x * TW >= nP) {
        // extra CTA: snapshot of X^(k)_{k+1,k+1} (the Cin of the look-ahead pivot CTA of the next update launch, which
        // overwrites that block in place).  64 x 64 complex = 2048 16-byte words; all loads of a thread are issued before
        // its stores (a load-store loop through two global pointers is serialised by possible aliasing, which made this
        // one CTA the longest of the launch).
        pdl_wait();
        const cx<float>* __restrict__ Xc = gj_buffer(a, z, freq, row, k);
        cx<float>* __restrict__ S = a.snap + (size_t)(a.zb0 + z) * GJ_NB * GJ_NB;
        const int k1 = (k + 1) * GJ_NB;
        constexpr int PER = GJ_NB * GJ_NB / 2 / 256;  // 8 words per thread
        float4 v[PER];
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int w = threadIdx.x + 256 * j, r = w >> 5, c2 = w & 31;
            v[j] = *reinterpret_cast<const float4*>(Xc + (size_t)(k1 + r) * nP + k1 + 2 * c2);
        }
#pragma unroll
        for (int j = 0; j < PER; ++j) reinterpret_cast<float4*>(S)[threadIdx.x + 256 * j] = v[j];
        return;
    }
    tc2::Tc2Tile t;
    tc2::tile_no_emit(t);
    t.bplanes = a.Xp + ((size_t)(k & 1) * a.nbmax + a.zb0 + z) * a.rp_stride;
    t.amat = a.zb0 + z;
    t.Cin = nullptr; t.ldcin = nP;
    t.Cout = gj_buffer(a, z, freq, row, k + 1) + (size_t)k * GJ_NB * nP; t.ldc = nP;
    t.M = GJ_NB; t.N = nP; t.K = GJ_NB; t.Mstore = GJ_NB;
    t.m0 = 0; t.n0 = blockIdx.x * TW;
    t.mask_lo = 0; t.mask_hi = 0; t.skip_lo = 0; t.skip_hi = 0;
    t.sgn = 1.f;
    t.bias_fix = bias_fix;
    t.drain_every = a.gj_drain;
    t.eb_planes = a.Rp + (size_t)(a.zb0 + z) * a.rp_stride; t.eb_m_lo = 0; t.eb_id_lo = 0; t.eb_id_hi = 0;
    gj_emit_a(a, t, z, freq, row, k, k * GJ_NB);
    tc2::cgemm_tile_h(t, &pmap, tc2_smem);
}

// TMA-fed tensor-core update: X' = Xtilde - X_:,k R over the whole matrix except the pivot block row; the epilogue also
// emits the next pivot block row (B planes) and the next column panel (A planes), or the finished inverse.
// 128 x 64 tiles, two CTAs per SM (gemm_tc2h.cuh), 256 threads, 1-D grid of up to two CTA roles:
//   [nbatch look-ahead pivot CTAs]  (pivot_next)  form and invert pivot block k+1 beside the tiles
//   [nbatch * ceil(nP/128) * nP/64 tile CTAs]
__global__ void __launch_bounds__(tc2::NUM_THREADS_H, 2)
tc2_gj_update_kernel(FactorArgs<float> a, int k, float bias_fix, int pivot_next, const __grid_constant__ CUtensorMap cmap) {
    extern __shared__ __align__(1024) unsigned char tc2_smem[];
    constexpr int TW = tc2::TNH;
    // With pivot_next the first nbatch CTAs are look-ahead pivot CTAs: CTA z forms and inverts the NEXT pivot
    // block of chain z while the other CTAs run the rank-64 update, so the latency-bound inversion hides behind the update
    // instead of preceding the next row panel.
    pdl_trigger();
    int bid = blockIdx.x;
    if (pivot_next) {
        if (bid < a.nbatch) {
            // The next pivot block is formed by the SAME tensor-core arithmetic as the update tile that owns it (same
            // operand planes, chunking, draining): a 128 x 64 product whose Cin is the snapshot of X^(k)_{k+1,k+1}
            // and whose result stays in shared memory.  Forming it with FP32 FMAs from the snapshot instead is more
            // accurate per entry but no longer consistent with the rest of block row k+1, and costs a factor 1.4 in
            // the wavefield error at 512^2 (tools/exp_accuracy.py: 9.5e-6 vs 6.7e-6).
            static_assert(tc2::CH_LD == GJ_NB + 1, "pivot body reads the staged tile with row stride GJ_NB + 1");
            const int z = bid, kb = k + 1, nP = a.g.nP;
            const int row = chain_row(a.g, a.phase, z, a.step);
            if (row < 0) { pdl_wait(); return; }
            tc2::Tc2Tile t;
            tc2::tile_no_emit(t);
            t.bplanes = a.Rp + (size_t)(a.zb0 + z) * a.rp_stride;
            t.amat = (k & 1) * a.nbmax + a.zb0 + z;
            const cx<float>* S1 = a.snap + (size_t)(a.zb0 + z) * GJ_NB * GJ_NB;  // X^(k)_{k+1,k+1}
            t.Cin = S1 - (size_t)(kb * GJ_NB) * GJ_NB - kb * GJ_NB; t.ldcin = GJ_NB;
            t.Cout = nullptr; t.ldc = nP; t.keep = 1;
            t.M = nP; t.N = nP; t.K = GJ_NB; t.Mstore = nP;
            t.m0 = (kb >> 1) * tc2::TM; t.n0 = kb * GJ_NB;
            t.mask_lo = 0; t.mask_hi = 0;
            t.skip_lo = (kb ^ 1) * GJ_NB; t.skip_hi = t.skip_lo + GJ_NB;  // the sibling block of the 128-row tile is not needed
            t.sgn = -1.f; t.bias_fix = bias_fix; t.drain_every = a.gj_drain;
            const bool traced = a.trace && a.step == a.trace_step && k == a.trace_k && z < 24;
            if (traced) {  // debugging: pivot CTAs use trace rows 1000 + z, their end-of-inversion stamp goes to column 17
                t.trace = a.trace + 16 * (1000 + z);
                if (threadIdx.x == 0) { unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); a.trace[16 * 1024 + 1000 + z] = smid; }
            }
            tc2::cgemm_tile_h(t, &cmap, tc2_smem);
            __syncthreads();
            unsigned char* smem_al = tc2_smem + ((128u - (tc::smem_u32(tc2_smem) & 127u)) & 127u);
            // the staged 128 x 65 tile holds the block (rows 64 (kb & 1) ..): invert it where it lies, scratch behind the tile
            cx<float>* blk = reinterpret_cast<cx<float>*>(smem_al) + (size_t)(kb & 1) * GJ_NB * tc2::CH_LD;
            cx<float>* scr = reinterpret_cast<cx<float>*>(smem_al) + (size_t)tc2::TM * tc2::CH_LD;
            static_assert((size_t)tc2::TM * tc2::CH_LD * sizeof(cx<float>) + gj_pivot2_scratch_bytes <= (size_t)tc2::STAGES_H * tc2::STAGE_H,
                          "pivot scratch must fit behind the staging tile inside the operand ring");
            gj_pivot_blocked(a, z, blk, scr, threadIdx.x, traced ? a.trace + 18 * 1024 + 16 * z : nullptr);
            if (traced && threadIdx.x == 0) a.trace[17 * 1024 + 1000 + z] = tc2::gtime();
            return;
        }
        bid -= a.nbatch;
    }
    const int nP = a.g.nP, nblk = nP / GJ_NB;
    const int tiles_m = (nP + tc2::TM - 1) / tc2::TM, tiles = (nP + TW - 1) / TW;
    const int z = bid / (tiles_m * tiles);
    const int rem = bid % (tiles_m * tiles);
    const int mt = rem / tiles, nt = rem % tiles;
    const int row = chain_row(a.g, a.phase, z, a.step);
    if (row < 0) { pdl_wait(); return; }
    const int freq = (a.f0 + chain_freq(a.phase, z));
    tc2::Tc2Tile t;
    tc2::tile_no_emit(t);
    t.bplanes = a.Rp + (size_t)(a.zb0 + z) * a.rp_stride;
    t.amat = (k & 1) * a.nbmax + a.zb0 + z;
    t.Cin = gj_buffer(a, z, freq, row, k); t.ldcin = nP;
    t.Cout = gj_buffer(a, z, freq, row, k + 1); t.ldc = nP;
    t.M = nP; t.N = nP; t.K = GJ_NB; t.Mstore = nP;
    t.m0 = mt * tc2::TM; t.n0 = nt * TW;
    t.mask_lo = k * GJ_NB; t.mask_hi = (k + 1) * GJ_NB;
    t.skip_lo = k * GJ_NB; t.skip_hi = (k + 1) * GJ_NB;
    t.sgn = -1.f;
    t.bias_fix = bias_fix;
    t.drain_every = a.gj_drain;
    gj_emit_a(a, t, z, freq, row, k, 0);
    if (k + 1 < nblk) {
        t.eb_planes = a.Xp + ((size_t)((k + 1) & 1) * a.nbmax + a.zb0 + z) * a.rp_stride;
        t.eb_m_lo = (k + 1) * GJ_NB; t.eb_id_lo = (k + 1) * GJ_NB; t.eb_id_hi = (k + 2) * GJ_NB;
    }
    if (a.trace && a.step == a.trace_step && k == a.trace_k && bid < 900) {
        t.trace = a.trace + 16 * bid;
        if (threadIdx.x == 0) { unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); a.trace[16 * 1024 + bid] = smid; }
    }
    t.prefetch_cin = a.prefetch_cin;
    tc2::cgemm_tile_h(t, &cmap, tc2_smem);
}

}  // namespace ust
