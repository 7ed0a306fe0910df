// gemm_tc2h.cuh -- the TMA-fed tcgen05 complex GEMM of gemm_tc2.cuh as a 128 x 64 tile with 256 threads, sized so that
// TWO CTAs are resident per SM.
//
// Why: the rank-64 Gauss-Jordan kernels (K = 64: four k-chunks) spend a third of a CTA's life each in loading, in the
// MMA / drain loop and in the write-out (in-situ trace, tools/exp_update_trace.py: 1.9 / 4.7 / 7 us of 14.7 us), and a
// 608-thread CTA with a 196 KB operand ring has the SM to itself, so nothing overlaps.  Two smaller co-resident CTAs let
// the hardware overlap one tile's write-out with the other's loads and MMAs.  What bounds the CTA size:
//   registers  warp w lives in SM sub-partition w % 4 (16384 registers each): 2 x 8 warps = 4 per sub-partition leaves
//              128 registers per thread; any extra role warp (9 or 10 per CTA) puts 6 on one sub-partition = 80 registers,
//              too few for the 64 FP32 accumulators a drain thread holds.  So all eight warps are drain warps and the
//              three service roles ride on them: warp 0 lane 0 = TMA producer + issuer of the leading product (D1),
//              warp 1 lane 0 = issuer of the five correction products (D2), warp 2 = TMEM allocation;
//   TMEM       D1 + D2 = 2 x 2 x 64 columns = 256 per CTA, 512 per SM;
//   smem       3 stages x 36 KB (A: 6 planes x 128 x 16, B: 3 planes x (64 re + 64 im) x 16) + barriers = 108.6 KB.
// Operand layouts in HBM are those of gemm_tc2.cuh (B planes are stored per 128-column tile: a 64-column half is two
// contiguous 2 KB pieces per plane, re rows and im rows).  Same arithmetic as gemm_tc2.cuh with drain_every = 1: the
// leading product of every 16-k chunk is drained to FP32 registers, corrections accumulate in D2, first-order bias fix.
#pragma once
#include "gemm_tc2.cuh"

namespace ust {
namespace tc2 {

constexpr int TNH = 64;
constexpr int BH_PLANE = 2 * TNH * KC * 2;                  // 4096 B
constexpr int BH_STAGE = NPL_B * BH_PLANE;                  // 12288 B
constexpr int STAGE_H = A_STAGE + BH_STAGE;                 // 36864 B
constexpr int STAGES_H = 3;
constexpr int NUM_THREADS_H = 256;
constexpr int NUM_WARPS_H = 8;
constexpr int CH_LD = TNH + 1;
constexpr int SMEM_BYTES_H = STAGES_H * STAGE_H + 128 + 128 + 384;  // ring + alignment slack + barriers + tile descriptor
static_assert(TM * CH_LD * 8 <= STAGES_H * STAGE_H, "epilogue staging tile must fit in the operand ring");
static_assert(2 * (SMEM_BYTES_H + 1024) <= 227 * 1024, "two CTAs per SM");
constexpr uint32_t TMEM_COLS_H = 256;                       // D1 = cols [0,128), D2 = cols [128,256)
constexpr uint32_t IDESC_N64 = IDESC_BASE | ((64u >> 3) << 17);

__device__ __forceinline__ void cgemm_tile_h(const Tc2Tile& t_in, const CUtensorMap* amap, unsigned char* smem_raw) {
    typedef cx<float> C;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) TC2_TRACE(0);
    if (tid == 0) asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)amap) : "memory");  // descriptor fetch overlaps the set-up
    const uint32_t smem_base = (smem_u32(smem_raw) + 127u) & ~127u;
    unsigned char* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t bar_base = smem_base + STAGES_H * STAGE_H;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES_H + s); };
    const uint32_t d1_full = bar_base + 8u * (2 * STAGES_H);
    const uint32_t d1_empty = bar_base + 8u * (2 * STAGES_H + 1);
    const uint32_t d2_full = bar_base + 8u * (2 * STAGES_H + 2);
    const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES_H + 3);
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_al + (tmem_slot - smem_base));
    Tc2Tile* t_sh = reinterpret_cast<Tc2Tile*>(smem_al + STAGES_H * STAGE_H + 128);
    if (tid == 0) *t_sh = t_in;
    const Tc2Tile& t = *t_sh;

    if (warp == 2) {
        if (lane == 0) {
            for (int s = 0; s < STAGES_H; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 2); }
            mbar_init(d1_full, 1);
            mbar_init(d1_empty, NUM_WARPS_H);
            mbar_init(d2_full, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS_H) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_acc = *tmem_slot_ptr;
    pdl_wait();
    if (warp == 0) TC2_TRACE(1);
    const uint32_t D1 = tmem_acc, D2 = tmem_acc + 2 * TNH;
    const int nk = (t.K + KC - 1) / KC;
    const int D = t.drain_every < 1 ? 1 : (t.drain_every > nk ? nk : t.drain_every);  // D1 is drained every D chunks

    // B source of this 64-column half: chunk c of the 128-column tile tn, plane p: re rows at +2048*half, im rows at +4096+2048*half
    const unsigned char* bsrc = reinterpret_cast<const unsigned char*>(t.bplanes) + (size_t)(t.n0 / TN) * nk * B_STAGE + ((t.n0 % TN) / TNH) * 2048;
    const int am0 = t.m0, amat = t.amat;
    // one chunk = 1 tensor copy (A) + 6 bulk copies (B), issued warp-convergently by warp 0 (one elected lane)
    auto load_chunk = [&](int c) {
        const int s = c % STAGES_H;
        const uint32_t sa = smem_base + s * STAGE_H, sb = sa + A_STAGE;
        mbar_expect_tx_e(full_bar(s), STAGE_H);
        tma_load_5d_e(sa, amap, full_bar(s), 0, (c * KC) >> 3, am0 >> 3, 0, amat);  // box {64, 2, 16, 6, 1}
        const unsigned char* bc = bsrc + (size_t)c * B_STAGE;
#pragma unroll
        for (int p = 0; p < NPL_B; ++p) {
            bulk_load_e(sb + p * BH_PLANE, bc + p * B_PLANE, 2048, full_bar(s));
            bulk_load_e(sb + p * BH_PLANE + 2048, bc + p * B_PLANE + 4096, 2048, full_bar(s));
        }
    };
    // first fill of the ring: chunk 0 by warp 0 (which then issues the leading products), the other stages by warp 2 (idle after
    // the TMEM allocation) -- issuing the 8 copies of a chunk takes an elected lane ~0.35 us, and with all three chunks on warp 0
    // the first MMA waited for the copies of chunks 1 and 2 to be ISSUED
    if (warp == 0) {
        load_chunk(0);
        TC2_TRACE(2);
    } else if (warp == 2) {
        for (int c = 1; c < nk && c < STAGES_H; ++c) load_chunk(c);
    }
    if (t.Cin && tid >= 128 && t.prefetch_cin) {
        // the tile of Cin is read only after the MMA loop: ask L2 for it now so that the HBM reads run under the loop
        const int rr = tid - 128, m = t.m0 + rr;
        const int ncols = t.N - t.n0 < TNH ? t.N - t.n0 : TNH;
        if (m < t.Mstore && !(m >= t.skip_lo && m < t.skip_hi) && ncols > 0 && ((ncols * 8) & 15) == 0 && ((t.ldcin & 1) == 0) && ((t.n0 & 1) == 0))
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"((uint64_t)(t.Cin + (size_t)m * t.ldcin + t.n0)), "r"((uint32_t)(ncols * 8)) : "memory");
    }

    const uint32_t id1 = IDESC_N128, id2 = IDESC_N64 | IDESC_ANEG, id3 = IDESC_N64;
    // descriptors of stage 0, built once (two make_desc per MMA cost a lone thread more than the MMA issue itself)
    uint64_t dAr[3], dAi[3], dB[3], dBi[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        dAr[i] = make_desc(smem_base + i * A_PLANE, 128u, 256u);
        dAi[i] = make_desc(smem_base + (3 + i) * A_PLANE, 128u, 256u);
        dB[i] = make_desc(smem_base + A_STAGE + i * BH_PLANE, 128u, 256u);
        dBi[i] = make_desc(smem_base + A_STAGE + i * BH_PLANE + (TNH / 8) * 256, 128u, 256u);
    }
    auto issue = [&](uint32_t d, uint64_t so, int i, int j, uint32_t acc_first) {
        umma_e(d, dAr[i] + so, dB[j] + so, id1, acc_first);    // [Cr|Ci] += Ar * [Br|Bi]
        umma_e(d, dAi[i] + so, dBi[j] + so, id2, 1u);          // Cr -= Ai * Bi
        umma_e(d + TNH, dAi[i] + so, dB[j] + so, id3, 1u);     // Ci += Ai * Br
    };

    const int q = warp & 3, cg = warp >> 2;
    const uint32_t lane_addr = ((uint32_t)(q * 32)) << 16;
    float acc_re[32], acc_im[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) { acc_re[j] = 0.f; acc_im[j] = 0.f; }

    for (int c = 0; c < nk; ++c) {
        const int s = c % STAGES_H;
        const uint32_t use = (uint32_t)(c / STAGES_H);
        if (warp < 2) {
            // issuer roles, executed warp-convergently (one elected lane issues, see umma_e)
            const uint64_t so = (uint64_t)((uint32_t)(s * STAGE_H) >> 4);
            mbar_wait(full_bar(s), use & 1u);
            if (warp == 0) {
                if (c == 0) TC2_TRACE(3);
                if (c > 0 && c % D == 0) mbar_wait(d1_empty, (uint32_t)(c / D - 1) & 1u);
                if (c == nk - 1) TC2_TRACE(8);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                issue(D1, so, 0, 0, c % D == 0 ? 0u : 1u);
                if ((c + 1) % D == 0 || c == nk - 1) umma_commit_e(d1_full);
                umma_commit_e(empty_bar(s));
                if (c == 0) TC2_TRACE(4);
            } else {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                issue(D2, so, 0, 1, c > 0 ? 1u : 0u);
                issue(D2, so, 1, 0, 1u);
                issue(D2, so, 0, 2, 1u);
                issue(D2, so, 2, 0, 1u);
                issue(D2, so, 1, 1, 1u);
                umma_commit_e(empty_bar(s));
                if (c == nk - 1) { TC2_TRACE(9); umma_commit_e(d2_full); }
            }
            __syncwarp();
        }
        // ---------------- every warp: drain D1 (chunks c-D+1..c) into FP32 registers ----------------
        if ((c + 1) % D == 0 || c == nk - 1) {
        mbar_wait(d1_full, (uint32_t)(c / D) & 1u);
        if (warp == 3 && c == 0) TC2_TRACE(5);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            uint32_t vr[8], vi[8];
            tmem_ld8(D1 + lane_addr + (uint32_t)(32 * cg + 8 * h), vr);
            tmem_ld8(D1 + lane_addr + (uint32_t)(TNH + 32 * cg + 8 * h), vi);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (h == 3) {
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(d1_empty);
                if (warp == 3 && c == 0) TC2_TRACE(6);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                acc_re[8 * h + j] += __uint_as_float(vr[j]);
                acc_im[8 * h + j] += __uint_as_float(vi[j]);
            }
        }
        }
        // refill the slot of chunk c once both issuers' MMAs on it have completed
        if (warp == 0 && c + STAGES_H < nk) {
            mbar_wait(empty_bar(s), use & 1u);
            load_chunk(c + STAGES_H);
        }
    }
    // ---------------- epilogue: add the correction accumulator, stage the tile in shared memory ----------------
    mbar_wait(d2_full, 0);
    if (warp == 3) TC2_TRACE(10);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    C* stage = reinterpret_cast<C*>(smem_al);
    {
        const int r = q * 32 + lane;
        const float bias = t.bias_fix * (float)D;  // the truncation bias grows linearly with the chunks accumulated per drain
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            uint32_t vr[8], vi[8];
            tmem_ld8(D2 + lane_addr + (uint32_t)(32 * cg + 8 * h), vr);
            tmem_ld8(D2 + lane_addr + (uint32_t)(TNH + 32 * cg + 8 * h), vi);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float ar = acc_re[8 * h + j], ai = acc_im[8 * h + j];
                const float cr = fmaf(ar, bias, __uint_as_float(vr[j]));
                const float ci = fmaf(ai, bias, __uint_as_float(vi[j]));
                stage[(size_t)r * CH_LD + 32 * cg + 8 * h + j] = C(ar + cr, ai + ci);
            }
        }
    }
    if (warp == 3) TC2_TRACE(11);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {  // the accumulators are in shared memory: give the TMEM columns back early (the co-resident CTA may be waiting)
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"(TMEM_COLS_H) : "memory");
    }
    if (warp == 3) TC2_TRACE(15);
    const Tc2Tile tl = *t_sh;
    // ---------------- coalesced write-out: one warp per row, 2 complex per lane ----------------
    const bool emit = tl.ea_planes != nullptr || tl.eb_planes != nullptr || tl.keep;  // keep: the caller reads the finished tile from shared memory
    const bool vec_ok = ((tl.ldc & 1) == 0) && ((((uintptr_t)tl.Cout) & 15) == 0) && (tl.n0 % 2 == 0) &&
                        (!tl.Cin || (((tl.ldcin & 1) == 0) && ((((uintptr_t)tl.Cin) & 15) == 0)));
    if (vec_ok && tl.n0 + TNH <= tl.N) {
        constexpr int RPW = TM / NUM_WARPS_H;  // 16 rows per warp, loads of all of them in flight before the first use
        float4 cin[RPW];
        unsigned live = 0;
        const int nloc = lane * 2, n = tl.n0 + nloc;
#pragma unroll
        for (int j = 0; j < RPW; ++j) {
            const int m = tl.m0 + warp + NUM_WARPS_H * j;
            const bool lv = m < tl.Mstore && !(m >= tl.skip_lo && m < tl.skip_hi);
            live |= (lv ? 1u : 0u) << j;
            cin[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (lv && tl.Cin) cin[j] = *reinterpret_cast<const float4*>(tl.Cin + (size_t)m * tl.ldcin + n);
        }
        const bool z0 = n >= tl.mask_lo && n < tl.mask_hi, z1 = n + 1 >= tl.mask_lo && n + 1 < tl.mask_hi;
#pragma unroll
        for (int j = 0; j < RPW; ++j) {
            const int rr = warp + NUM_WARPS_H * j;
            const int m = tl.m0 + rr;
            if (!((live >> j) & 1u)) continue;
            const C a0 = stage[(size_t)rr * CH_LD + nloc], a1 = stage[(size_t)rr * CH_LD + nloc + 1];
            float4 c = cin[j];
            if (z0) { c.x = 0.f; c.y = 0.f; }
            if (z1) { c.z = 0.f; c.w = 0.f; }
            c.x += tl.sgn * a0.re; c.y += tl.sgn * a0.im; c.z += tl.sgn * a1.re; c.w += tl.sgn * a1.im;
            if (tl.Cout) *reinterpret_cast<float4*>(tl.Cout + (size_t)m * tl.ldc + n) = c;
            if (emit) { stage[(size_t)rr * CH_LD + nloc] = C(c.x, c.y); stage[(size_t)rr * CH_LD + nloc + 1] = C(c.z, c.w); }
        }
    } else {
        for (int rr = warp; rr < TM; rr += NUM_WARPS_H) {
            const int m = tl.m0 + rr;
            if (m >= tl.Mstore || (m >= tl.skip_lo && m < tl.skip_hi)) continue;
            const int nloc = lane * 2, n = tl.n0 + nloc;
            if (n >= tl.N) continue;
            const C a0 = stage[(size_t)rr * CH_LD + nloc], a1 = stage[(size_t)rr * CH_LD + nloc + 1];
            C c0 = cxzero<float>(), c1 = cxzero<float>();
            if (tl.Cin) {
                const C* ci = tl.Cin + (size_t)m * tl.ldcin + n;
                c0 = ci[0];
                if (n + 1 < tl.N) c1 = ci[1];
                if (n >= tl.mask_lo && n < tl.mask_hi) c0 = cxzero<float>();
                if (n + 1 >= tl.mask_lo && n + 1 < tl.mask_hi) c1 = cxzero<float>();
            }
            c0.re += tl.sgn * a0.re; c0.im += tl.sgn * a0.im;
            c1.re += tl.sgn * a1.re; c1.im += tl.sgn * a1.im;
            if (tl.Cout) {
                C* co = tl.Cout + (size_t)m * tl.ldc + n;
                co[0] = c0;
                if (n + 1 < tl.N) co[1] = c1;
            }
            if (emit) { stage[(size_t)rr * CH_LD + nloc] = c0; stage[(size_t)rr * CH_LD + nloc + 1] = c1; }
        }
    }
    if (warp == 3) TC2_TRACE(12);
    if (emit) {
        // ---------------- emit the finished tile as operand planes (layouts of gemm_tc2.cuh) ----------------
        __syncthreads();
        if (tl.eb_planes && tl.eb_m_lo >= tl.m0 && tl.eb_m_lo < tl.m0 + TM) {
            const int r0 = tl.eb_m_lo - tl.m0;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int e = tid + NUM_THREADS_H * h;
                const int nloc = e & (TNH - 1), kg = e >> 6;
                const int n = tl.n0 + nloc;
                float re[8], im[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    C v = stage[(size_t)(r0 + 8 * kg + c) * CH_LD + nloc];
                    if (n >= tl.eb_id_lo && n < tl.eb_id_hi) v = C((n - tl.eb_id_lo == 8 * kg + c) ? 1.f : 0.f, 0.f);
                    if (n >= tl.N) v = cxzero<float>();
                    re[c] = v.re; im[c] = v.im;
                }
                uint16_t* chunk = tl.eb_planes + ((size_t)(n / TN) * (64 / KC) + (kg >> 1)) * (B_STAGE / 2);
                store_b8(chunk, n % TN, kg & 1, re, im);
            }
        }
        if (tl.ea_planes) {
            const int lo = tl.ea_n_lo > tl.n0 ? tl.ea_n_lo : tl.n0;
            const int hi = tl.ea_n_hi < tl.n0 + TNH ? tl.ea_n_hi : tl.n0 + TNH;
            const int nJ = hi > lo ? (hi - lo) >> 3 : 0;
            for (int e = tid; e < nJ * TM; e += NUM_THREADS_H) {
                const int rr = e & (TM - 1), jj = e >> 7;
                const int m = tl.m0 + rr;
                if (m >= tl.Mstore || (m >= tl.skip_lo && m < tl.skip_hi)) continue;
                const int n8 = lo + 8 * jj;
                const int tr = m + tl.ea_row_off, tcol = n8 - tl.ea_col_off;
                float re[8], im[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    C v = stage[(size_t)rr * CH_LD + (n8 - tl.n0) + c];
                    if (tr >= tl.ea_zero_from || tcol + c >= tl.ea_zero_from || n8 + c >= tl.N) v = cxzero<float>();
                    re[c] = v.re; im[c] = v.im;
                }
                uint16_t* dst = tl.ea_planes + ((size_t)(tr >> 3) * tl.ea_nbc + (tcol >> 3)) * 64 + (tr & 7) * 8;
                store_a8(dst, tl.ea_plane_elems, re, im);
            }
        }
    }
    if (warp == 3) TC2_TRACE(13);
    if (warp == 2) TC2_TRACE(14);
}

}  // namespace tc2
}  // namespace ust
