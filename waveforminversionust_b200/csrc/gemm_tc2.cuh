// gemm_tc2.cuh -- TMA-fed, warp-specialised complex64 GEMM on tcgen05 with split operands prepared in HBM.
//
//     Cout = (Cin ? Cin : 0) + sgn * op(A) * B,     op(A) = A  or  conj(A)^T,    complex64 in / out
//
// Why this shape (a first engine, removed after round 1, had every CTA re-read FP32 operands, split them into bf16
// planes with its own ALUs and accumulate everything inside the tensor core): two measured
// problems (tools/exp_tc_accum.py, profiles/): (i) the tensor core adds into its FP32 accumulator with
// truncation, a bias of about -1.7e-9 per accumulated k that compounds coherently over the ~Ny dependent
// block rows (1.8e-4 wavefield error at 512^2); (ii) the eight converting warps, not the MMA pipe, set the pace.
// Here
//   * operands are split ONCE by their producers into bf16 planes laid out as 8x8 "core matrices" (128 B):
//       A planes  [matrix][plane 0..5 = re1,re2,re3,im1,im2,im3][I = row/8][J = col/8][8][8]        (Gauss-Jordan epilogues, a_split_kernel)
//       B planes  [batch][n-tile][k-chunk][plane 0..2][256 rows = (re of 128 columns | im)][16 k]      (tri_apply2 / b_split)
//     so one 5-D TMA tensor copy brings a [128 x 16] (forward, K-major) or [16 x 128] (adjoint, MN-major: the
//     same 8x8 blocks, leading/stride offsets swapped, a_major bit set) slab of all six A planes, and one
//     1-D bulk copy brings the three B planes of a k-chunk;
//   * the leading product a1*b1 of every 16-k chunk goes to its own TMEM accumulator D1 which sixteen drain
//     warps read back (tcgen05.ld) and add to FP32 registers with round-to-nearest, while the five small
//     correction products of the chunk run on the tensor core into D2 (their truncation is 2^-8 smaller);
//   * complex arithmetic needs no duplicated/negated B planes: per plane pair
//       [Cr|Ci] += Ar*[Br|Bi]   (N=256);   Cr += (-Ai)*Bi   (N=128, a_negate);   Ci += Ai*Br   (N=128)
//     (signs of the last two swapped for conj(A));
//   * the epilogue goes through shared memory so global reads/writes of C are row-contiguous.
// Warp roles (608 threads): warp 0 TMA producer, warp 1 TMEM allocator + issuer of the leading products (D1), warp 2
// issuer of the correction products (D2) -- one thread cannot issue 18 MMAs per chunk fast enough (measured 43 ns per
// MMA, tools/exp_tc2_trace.py) and the D1 hand-shake must not sit behind the correction stream --, warps 3..18
// drain/epilogue (warp w owns TMEM lanes 32*(w%4).. and complex columns 32*((w-3)/4)..).
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace ust {
namespace tc2 {

using tc::mbar_arrive;
using tc::mbar_init;
using tc::mbar_wait;
using tc::smem_u32;

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}

constexpr int TM = 128, TN = 128, KC = 16;
constexpr int NPL_A = 6, NPL_B = 3;
constexpr int A_PLANE = TM * KC * 2;                       // 4096 B
constexpr int B_PLANE = 2 * TN * KC * 2;                   // 8192 B
constexpr int A_STAGE = NPL_A * A_PLANE;                   // 24576 B
constexpr int B_STAGE = NPL_B * B_PLANE;                   // 24576 B
constexpr int STAGE_BYTES = A_STAGE + B_STAGE;             // 49152 B
constexpr int STAGES = 4;
constexpr int NUM_EPI_WARPS = 16;
constexpr int FIRST_EPI_WARP = 3;
constexpr int NUM_THREADS = 32 * (FIRST_EPI_WARP + NUM_EPI_WARPS);  // 608
constexpr int C_LD = TN + 1;                               // padded row of the complex staging tile
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 512;  // ring + alignment slack + barriers (128 B) + tile descriptor (384 B)
static_assert(TM * C_LD * 8 <= STAGES * STAGE_BYTES, "epilogue staging tile must fit in the operand ring");
constexpr uint32_t TMEM_COLS = 512;                        // D1 = cols [0,256), D2 = cols [256,512)

// element offset of (row r, k) inside one B plane of one k-chunk (K-major, SWIZZLE_NONE, LBO 128 B, SBO 256 B)
__host__ __device__ __forceinline__ int bplane_off(int r, int k) { return (r >> 3) * 128 + (k >> 3) * 64 + (r & 7) * 8 + (k & 7); }
// number of bf16 elements of the B-plane buffer of one batch entry
__host__ __device__ __forceinline__ size_t bplanes_elems(int kpad, int ncols) {
    return (size_t)((ncols + TN - 1) / TN) * (size_t)(kpad / KC) * (size_t)(B_STAGE / 2);
}
// element offset of entry (row, col) of plane p of an A matrix with leading dimension nP (multiple of 64)
__host__ __device__ __forceinline__ size_t aplane_off(int nP, int p, int row, int col) {
    const int nb = nP >> 3;
    return (size_t)p * nP * nP + ((size_t)(row >> 3) * nb + (col >> 3)) * 64 + (row & 7) * 8 + (col & 7);
}

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(lbo >> 4) << 16;
    d |= (uint64_t)(sbo >> 4) << 32;
    d |= (uint64_t)1 << 46;  // descriptor version (Blackwell); layout_type 0 = SWIZZLE_NONE
    return d;
}
// kind::f16: BF16 x BF16 -> F32, M = 128
constexpr uint32_t IDESC_BASE = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 4) << 24);
constexpr uint32_t IDESC_N256 = IDESC_BASE | ((256u >> 3) << 17);
constexpr uint32_t IDESC_N128 = IDESC_BASE | ((128u >> 3) << 17);
constexpr uint32_t IDESC_ANEG = 1u << 13;
constexpr uint32_t IDESC_AMN = 1u << 15;  // A operand MN-major

__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// Warp-convergent forms: every lane executes the statement with the same operands and one elected lane issues.  Inside
// an `if (lane == 0)` the compiler cannot keep descriptors in uniform registers and wraps each MMA in a waterfall loop
// (ELECT / R2UR.BROADCAST / BRA.U.ANY, ~20 instructions per MMA for a lone thread).
__device__ __forceinline__ void umma_e(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_e(uint32_t bar) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(bar)
        : "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(dst), "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"((uint64_t)src), "r"(bytes), "r"(bar)
                 : "memory");
}

// warp-convergent forms of the copy instructions (same operands in every lane, one elected lane issues; see umma_e)
__device__ __forceinline__ void mbar_expect_tx_e(uint32_t bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\t"
                 "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_5d_e(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
    asm volatile(
        "{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\t"
        "@q cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];\n\t}"
        ::"r"(dst), "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void bulk_load_e(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\t"
                 "@q cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n\t}"
                 ::"r"(dst), "l"((uint64_t)src), "r"(bytes), "r"(bar)
                 : "memory");
}

// three bf16 words (two consecutive values each) of plane 1..3
using tc::split2;
using tc::Split3;

// split 8 consecutive k of one B line (re and im) and store the 16-byte chunks of the three planes.
// `chunk` points at the [3][256][16] block of this (n-tile, k-chunk); r = column within the tile; kh = 0/1 half of the chunk
__device__ __forceinline__ void store_b8(uint16_t* chunk, int r, int kh, const float (&re)[8], const float (&im)[8]) {
    uint32_t wr[3][4], wi[3][4];
#pragma unroll
    for (int qd = 0; qd < 4; ++qd) {
        Split3 sr = split2(re[2 * qd], re[2 * qd + 1]);
        Split3 si = split2(im[2 * qd], im[2 * qd + 1]);
#pragma unroll
        for (int s = 0; s < 3; ++s) { wr[s][qd] = sr.w[s]; wi[s][qd] = si.w[s]; }
    }
#pragma unroll
    for (int s = 0; s < 3; ++s) {
        uint16_t* pl = chunk + s * (B_PLANE / 2);
        *reinterpret_cast<uint4*>(pl + bplane_off(r, kh * 8)) = make_uint4(wr[s][0], wr[s][1], wr[s][2], wr[s][3]);
        *reinterpret_cast<uint4*>(pl + bplane_off(TN + r, kh * 8)) = make_uint4(wi[s][0], wi[s][1], wi[s][2], wi[s][3]);
    }
}

// split 8 consecutive entries of one A row (re and im) and store the 16-byte chunks of the six planes; `dst` points at
// the chunk inside plane 0, planes are `plane_elems` apart
__device__ __forceinline__ void store_a8(uint16_t* dst, size_t plane_elems, const float (&re)[8], const float (&im)[8]) {
    uint32_t wr[3][4], wi[3][4];
#pragma unroll
    for (int qd = 0; qd < 4; ++qd) {
        Split3 sr = split2(re[2 * qd], re[2 * qd + 1]);
        Split3 si = split2(im[2 * qd], im[2 * qd + 1]);
#pragma unroll
        for (int s = 0; s < 3; ++s) { wr[s][qd] = sr.w[s]; wi[s][qd] = si.w[s]; }
    }
#pragma unroll
    for (int s = 0; s < 3; ++s) {
        *reinterpret_cast<uint4*>(dst + s * plane_elems) = make_uint4(wr[s][0], wr[s][1], wr[s][2], wr[s][3]);
        *reinterpret_cast<uint4*>(dst + (3 + s) * plane_elems) = make_uint4(wi[s][0], wi[s][1], wi[s][2], wi[s][3]);
    }
}

// One tile of the product.  A comes through the tensor map (planes of matrix `amat`), B from `bplanes`.
struct Tc2Tile {
    const uint16_t* bplanes;       // B planes of this batch entry
    int amat;                      // matrix index (coordinate 4 of the tensor map)
    const cx<float>* Cin; int ldcin;
    cx<float>* Cout; int ldc;
    int M, N, K;                   // logical sizes (K rounded up to KC inside; planes are zero padded)
    int Mstore;                    // rows m < Mstore are written
    int m0, n0;                    // tile origin
    int mask_lo, mask_hi;          // Cin columns in [mask_lo, mask_hi) read as zero
    int skip_lo, skip_hi;          // output rows in [skip_lo, skip_hi) are left untouched
    float sgn;
    float bias_fix;                // first-order correction of the tensor core's truncation bias on D1 per accumulated chunk (0 = off)
    int drain_every;               // D1 is drained to registers every `drain_every` chunks (1 = every chunk; >= nk = once at the end)
    // Optional: the epilogue also emits the finished tile as split operand planes for the kernels that consume it next
    // (saves a separate split pass over the same data).
    uint16_t* ea_planes;           // A planes (null = off): target entry (row m + ea_row_off, col n - ea_col_off)
    unsigned ea_plane_elems;       //   elements per plane
    int ea_nbc;                    //   8x8 blocks per target row
    int ea_n_lo, ea_n_hi;          //   tile columns n in [ea_n_lo, ea_n_hi) are emitted (multiples of 8)
    int ea_col_off, ea_row_off;
    int ea_zero_from;              //   target rows / columns >= this are written as zero
    uint16_t* eb_planes;           // B planes (null = off), K = 64 rows: k = m - eb_m_lo in [0, 64)
    int eb_m_lo;
    int eb_id_lo, eb_id_hi;        //   columns n in [eb_id_lo, eb_id_hi) are replaced by the identity (Gauss-Jordan pivot column)
    unsigned long long* trace;     // optional phase timestamps of this CTA, 16 slots (tools/exp_tc2_trace.py); null = off
    int prefetch_cin;              // L2 prefetch of the Cin tile when the CTA starts
    int keep;                      // 128 x 64 form: leave the finished tile (Cin + sgn*A*B, live rows) in the shared-memory staging
                                   // tile [128][65] at the 128-byte aligned base of the dynamic shared memory; Cout may be null
    // 128 x 128 form launched as clusters of two or four CTAs (split K): CTA rank r computes its share of the k-chunks, all stage
    // their partial tile, rank 0 adds the others' through distributed shared memory (in rank order) and writes the result (no
    // emission in this mode).
    // For launches with so few tiles that most SMs idle (sweeps of one or two frequencies): the tile's k loop is the launch.
    int ksplit;                    // 0 / 1 = off, 2 / 4 = CTAs per cluster
};
__host__ __device__ __forceinline__ void tile_no_emit(Tc2Tile& t) {
    t.ea_planes = nullptr; t.ea_plane_elems = 0; t.ea_nbc = 0; t.ea_n_lo = 0; t.ea_n_hi = 0; t.ea_col_off = 0; t.ea_row_off = 0;
    t.drain_every = 1; t.ea_zero_from = 0x7fffffff; t.eb_planes = nullptr; t.eb_m_lo = 0; t.eb_id_lo = 0; t.eb_id_hi = 0; t.trace = nullptr; t.prefetch_cin = 0; t.keep = 0; t.ksplit = 0;
}

static_assert(sizeof(Tc2Tile) <= 384, "tile descriptor must fit in its shared-memory slot");

__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long v;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
    return v;
}
#define TC2_TRACE(slot)                                                                               \
    do {                                                                                              \
        if (t_in.trace && lane == 0) t_in.trace[slot] = gtime();                                     \
    } while (0)

__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {  // every thread of both CTAs
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_map(uint32_t saddr, uint32_t rank) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank)); return r;
}
__device__ __forceinline__ cx<float> ld_cluster_c(uint32_t caddr) {
    float x, y; asm volatile("ld.shared::cluster.v2.f32 {%0, %1}, [%2];" : "=f"(x), "=f"(y) : "r"(caddr) : "memory"); return cx<float>(x, y);
}

template <bool TA>
__device__ __forceinline__ void cgemm_tile(const Tc2Tile& t_in, const CUtensorMap* amap, unsigned char* smem_raw) {
    typedef cx<float> C;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) TC2_TRACE(0);
    if (tid == 0) asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)amap) : "memory");  // descriptor fetch overlaps the set-up
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    unsigned char* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t bar_base = smem_base + STAGES * STAGE_BYTES;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
    const uint32_t d1_full = bar_base + 8u * (2 * STAGES);
    const uint32_t d1_empty = bar_base + 8u * (2 * STAGES + 1);
    const uint32_t d2_full = bar_base + 8u * (2 * STAGES + 2);
    const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 3);
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_al + (tmem_slot - smem_base));
    // the tile descriptor lives in shared memory: the drain warps have no registers to spare for it
    Tc2Tile* t_sh = reinterpret_cast<Tc2Tile*>(smem_al + STAGES * STAGE_BYTES + 128);
    if (tid == 0) *t_sh = t_in;
    const Tc2Tile& t = *t_sh;

    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 2); }
            mbar_init(d1_full, 1);
            mbar_init(d1_empty, NUM_EPI_WARPS);
            mbar_init(d2_full, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_acc = *tmem_slot_ptr;
    pdl_wait();  // prologue (barriers, TMEM) overlapped the previous kernel; from here on global memory is touched
    if (warp == 0) TC2_TRACE(1);
    const uint32_t D1 = tmem_acc, D2 = tmem_acc + 2 * TN;
    const int nk_all = (t.K + KC - 1) / KC;  // read after the __syncthreads above
    const int nsplit = t.ksplit > 1 ? t.ksplit : 1;   // CTAs of the cluster that share this tile's k range (1, 2 or 4)
    const bool split = nsplit > 1;
    const uint32_t crank = split ? cluster_ctarank() : 0u;
    const int per = (nk_all + nsplit - 1) / nsplit;
    const int c_first = (int)crank * per;            // this CTA's k-chunks: [c_first, c_first + nk); the host keeps nk >= 1
    const int nk = nk_all - c_first < per ? nk_all - c_first : per;
    const int D = t.drain_every < 1 ? 1 : (t.drain_every > nk ? nk : t.drain_every);
    const int ndrain = (nk + D - 1) / D;
    if (t.Cin && t.prefetch_cin && warp >= FIRST_EPI_WARP && tid - 32 * FIRST_EPI_WARP < TM) {
        // Cin is read only after the MMA loop: ask L2 for the tile now (one row per drain thread; they idle until chunk 0 lands)
        const int m = t.m0 + tid - 32 * FIRST_EPI_WARP;
        const int ncols = t.N - t.n0 < TN ? t.N - t.n0 : TN;
        if (m < t.Mstore && !(m >= t.skip_lo && m < t.skip_hi) && ncols > 0 && ((ncols * 8) & 15) == 0 && ((t.ldcin & 1) == 0) && ((t.n0 & 1) == 0) &&
            ((((uintptr_t)t.Cin) & 15) == 0))
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"((uint64_t)(t.Cin + (size_t)m * t.ldcin + t.n0)), "r"((uint32_t)(ncols * 8)) : "memory");
    }

    if (warp == 0) {
        // ---------------- TMA producer (whole warp, one elected lane issues) ----------------
        {
            const int tn = t.n0 / TN;
            const unsigned char* bsrc = reinterpret_cast<const unsigned char*>(t.bplanes) + (size_t)tn * nk_all * B_STAGE;
            const int m0 = t.m0, amat = t.amat;
            for (int c = 0; c < nk; ++c) {
                const int s = c % STAGES;
                const uint32_t use = (uint32_t)(c / STAGES);
                mbar_wait(empty_bar(s), (use & 1u) ^ 1u);
                const uint32_t sa = smem_base + s * STAGE_BYTES, sb = sa + A_STAGE;
                mbar_expect_tx_e(full_bar(s), STAGE_BYTES);
                if (!TA) tma_load_5d_e(sa, amap, full_bar(s), 0, ((c_first + c) * KC) >> 3, m0 >> 3, 0, amat);   // box {64, 2, 16, 6, 1}
                else     tma_load_5d_e(sa, amap, full_bar(s), 0, m0 >> 3, ((c_first + c) * KC) >> 3, 0, amat);   // box {64, 16, 2, 6, 1}
                bulk_load_e(sb, bsrc + (size_t)(c_first + c) * B_STAGE, B_STAGE, full_bar(s));
                if (c == 0) TC2_TRACE(2);
            }
        }
        __syncwarp();
        if (split) { cluster_sync_all(); cluster_sync_all(); }  // partner barriers of the drain warps' two (staged / read)
    } else if (warp == 1 || warp == 2) {
        // ---------------- MMA issuers: warp 1 = leading product -> D1 (paced by the drain), warp 2 = corrections -> D2 ----------------
        // A descriptors: forward = K-major rows of A ([i16][j2] blocks: SBO 256, LBO 128);
        //                adjoint = MN-major ([i2][j16] blocks: K groups 2048 B apart = LBO, MN groups 128 B apart = SBO)
        const uint32_t a_lbo = TA ? 2048u : 128u, a_sbo = TA ? 128u : 256u;
        const uint32_t amaj = TA ? IDESC_AMN : 0u;
        // product 2: Cr += -+ Ai*Bi ; product 3: Ci += +- Ai*Br   (upper signs: plain A, lower: conj(A))
        const uint32_t id1 = IDESC_N256 | amaj;
        const uint32_t id2 = IDESC_N128 | amaj | (TA ? 0u : IDESC_ANEG);
        const uint32_t id3 = IDESC_N128 | amaj | (TA ? IDESC_ANEG : 0u);
        const bool lead = warp == 1;
        // descriptors of stage 0, built once: a single thread spends ~25 dependent integer instructions (50-70 ns) on two
        // make_desc calls per MMA otherwise, which is what paced the issue; a stage is one 64-bit add away
        uint64_t dAr[3], dAi[3], dB[3], dBi[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            dAr[i] = make_desc(smem_base + i * A_PLANE, a_lbo, a_sbo);
            dAi[i] = make_desc(smem_base + (3 + i) * A_PLANE, a_lbo, a_sbo);
            dB[i] = make_desc(smem_base + A_STAGE + i * B_PLANE, 128u, 256u);
            dBi[i] = make_desc(smem_base + A_STAGE + i * B_PLANE + (TN / 8) * 256, 128u, 256u);
        }
        for (int c = 0; c < nk; ++c) {
            const int s = c % STAGES;
            const uint32_t use = (uint32_t)(c / STAGES);
            mbar_wait(full_bar(s), use & 1u);
            if (lead && c == 0) TC2_TRACE(3);
            if (lead && c > 0 && c % D == 0) mbar_wait(d1_empty, (uint32_t)(c / D - 1) & 1u);
            if (lead && c == 1) TC2_TRACE(7);
            if (lead && c == nk - 1) TC2_TRACE(8);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            {
                const uint64_t so = (uint64_t)((uint32_t)(s * STAGE_BYTES) >> 4);
                auto issue = [&](uint32_t d, int i, int j, uint32_t acc_first) {
                    umma_e(d, dAr[i] + so, dB[j] + so, id1, acc_first);        // [Cr|Ci] += Ar * [Br|Bi]
                    umma_e(d, dAi[i] + so, dBi[j] + so, id2, 1u);              // Cr -+= Ai * Bi
                    umma_e(d + TN, dAi[i] + so, dB[j] + so, id3, 1u);          // Ci +-= Ai * Br   (N=128 reads the Br rows only)
                };
                if (lead) {
                    issue(D1, 0, 0, c % D == 0 ? 0u : 1u);
                    if ((c + 1) % D == 0 || c == nk - 1) umma_commit_e(d1_full);
                    umma_commit_e(empty_bar(s));
                    if (c == 0) TC2_TRACE(4);
                } else {
                    issue(D2, 0, 1, c > 0 ? 1u : 0u);
                    issue(D2, 1, 0, 1u);
                    issue(D2, 0, 2, 1u);
                    issue(D2, 2, 0, 1u);
                    issue(D2, 1, 1, 1u);
                    umma_commit_e(empty_bar(s));
                    if (c == nk - 1) TC2_TRACE(9);
                    if (c == nk - 1) umma_commit_e(d2_full);
                }
            }
            __syncwarp();
        }
        if (split) { cluster_sync_all(); cluster_sync_all(); }
    } else {
        // ---------------- drain warps: D1 -> FP32 registers every chunk ----------------
        const int q = warp & 3, cg = (warp - FIRST_EPI_WARP) >> 2;
        const uint32_t lane_addr = ((uint32_t)(q * 32)) << 16;
        float acc_re[32], acc_im[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) { acc_re[j] = 0.f; acc_im[j] = 0.f; }
        for (int c = 0; c < ndrain; ++c) {
            mbar_wait(d1_full, (uint32_t)c & 1u);
            if (warp == FIRST_EPI_WARP && c == 0) TC2_TRACE(5);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                uint32_t vr[8], vi[8];
                tmem_ld8(D1 + lane_addr + (uint32_t)(32 * cg + 8 * h), vr);
                tmem_ld8(D1 + lane_addr + (uint32_t)(TN + 32 * cg + 8 * h), vi);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (h == 3) {  // D1 has been read completely: hand it back before doing the last additions
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(d1_empty);
                    if (warp == FIRST_EPI_WARP && c == 0) TC2_TRACE(6);
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    acc_re[8 * h + j] += __uint_as_float(vr[j]);
                    acc_im[8 * h + j] += __uint_as_float(vi[j]);
                }
            }
        }
        // ---------------- epilogue: add the correction accumulator, stage the tile in shared memory ----------------
        mbar_wait(d2_full, 0);
        if (warp == FIRST_EPI_WARP) TC2_TRACE(10);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        C* stage = reinterpret_cast<C*>(smem_al);
        const int r = q * 32 + lane;
        const float bias = t.bias_fix * (float)D;  // the truncation bias grows linearly with the chunks accumulated per drain
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            uint32_t vr[8], vi[8];
            tmem_ld8(D2 + lane_addr + (uint32_t)(32 * cg + 8 * h), vr);
            tmem_ld8(D2 + lane_addr + (uint32_t)(TN + 32 * cg + 8 * h), vi);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float ar = acc_re[8 * h + j], ai = acc_im[8 * h + j];
                const float cr = fmaf(ar, bias, __uint_as_float(vr[j]));
                const float ci = fmaf(ai, bias, __uint_as_float(vi[j]));
                stage[(size_t)r * C_LD + 32 * cg + 8 * h + j] = C(ar + cr, ai + ci);
            }
        }
        if (warp == FIRST_EPI_WARP) TC2_TRACE(11);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        asm volatile("bar.sync 1, %0;" ::"n"(NUM_EPI_WARPS * 32) : "memory");
        if (warp == FIRST_EPI_WARP) TC2_TRACE(15);
        // the accumulators are dead now: take a private copy of the tile descriptor so that stores through Cout / the
        // staging tile cannot force re-reads of its fields from shared memory
        const Tc2Tile tl = *t_sh;
        uint32_t peer[3] = {0, 0, 0};
        if (split) {
            cluster_sync_all();  // all partial tiles are staged
#pragma unroll
            for (int pr = 1; pr < 4; ++pr)
                if (pr < nsplit) peer[pr - 1] = cluster_map(smem_u32(stage), (uint32_t)pr);
        }
        if (!split || crank == 0) {
        // ---------------- coalesced write-out: one warp per row, 4 complex per lane ----------------
        const int ew = warp - FIRST_EPI_WARP;
        const bool emit = tl.ea_planes != nullptr || tl.eb_planes != nullptr;
        const bool vec_ok = ((tl.ldc & 1) == 0) && ((((uintptr_t)tl.Cout) & 15) == 0) && (tl.n0 % 2 == 0) &&
                            (!tl.Cin || (((tl.ldcin & 1) == 0) && ((((uintptr_t)tl.Cin) & 15) == 0)));
        if (vec_ok && tl.n0 + TN <= tl.N) {
            // fast path (full-width, aligned tile): all Cin loads of this warp's 8 rows are issued before any is used
            constexpr int RPW = TM / NUM_EPI_WARPS;  // 8 rows per warp
            float4 cin[RPW][2];
            bool live[RPW];
#pragma unroll
            for (int j = 0; j < RPW; ++j) {
                const int m = tl.m0 + ew + NUM_EPI_WARPS * j;
                live[j] = m < tl.Mstore && !(m >= tl.skip_lo && m < tl.skip_hi);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    cin[j][h] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (live[j] && tl.Cin) cin[j][h] = *reinterpret_cast<const float4*>(tl.Cin + (size_t)m * tl.ldcin + tl.n0 + h * 64 + lane * 2);
                }
            }
#pragma unroll
            for (int j = 0; j < RPW; ++j) {
                const int rr = ew + NUM_EPI_WARPS * j;
                const int m = tl.m0 + rr;
                if (!live[j]) continue;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int nloc = h * 64 + lane * 2;
                    const int n = tl.n0 + nloc;
                    C a0 = stage[(size_t)rr * C_LD + nloc], a1 = stage[(size_t)rr * C_LD + nloc + 1];
                    if (split) {
#pragma unroll
                        for (int pr = 0; pr < 3; ++pr) {
                            if (pr + 1 >= nsplit) break;
                            const C b0 = ld_cluster_c(peer[pr] + (uint32_t)(((size_t)rr * C_LD + nloc) * sizeof(C))), b1 = ld_cluster_c(peer[pr] + (uint32_t)(((size_t)rr * C_LD + nloc + 1) * sizeof(C)));
                            a0.re += b0.re; a0.im += b0.im; a1.re += b1.re; a1.im += b1.im;
                        }
                    }
                    float4 c = cin[j][h];
                    if (n >= tl.mask_lo && n < tl.mask_hi) { c.x = 0.f; c.y = 0.f; }
                    if (n + 1 >= tl.mask_lo && n + 1 < tl.mask_hi) { c.z = 0.f; c.w = 0.f; }
                    c.x += tl.sgn * a0.re; c.y += tl.sgn * a0.im; c.z += tl.sgn * a1.re; c.w += tl.sgn * a1.im;
                    *reinterpret_cast<float4*>(tl.Cout + (size_t)m * tl.ldc + n) = c;
                    if (emit) { stage[(size_t)rr * C_LD + nloc] = C(c.x, c.y); stage[(size_t)rr * C_LD + nloc + 1] = C(c.z, c.w); }
                }
            }
        } else
        for (int rr = ew; rr < TM; rr += NUM_EPI_WARPS) {
            const int m = tl.m0 + rr;
            if (m >= tl.Mstore || (m >= tl.skip_lo && m < tl.skip_hi)) continue;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int nloc = h * 64 + lane * 2;
                const int n = tl.n0 + nloc;
                if (n >= tl.N) continue;
                C a0 = stage[(size_t)rr * C_LD + nloc], a1 = stage[(size_t)rr * C_LD + nloc + 1];
                if (split) {
#pragma unroll
                    for (int pr = 0; pr < 3; ++pr) {
                        if (pr + 1 >= nsplit) break;
                        const C b0 = ld_cluster_c(peer[pr] + (uint32_t)(((size_t)rr * C_LD + nloc) * sizeof(C))), b1 = ld_cluster_c(peer[pr] + (uint32_t)(((size_t)rr * C_LD + nloc + 1) * sizeof(C)));
                        a0.re += b0.re; a0.im += b0.im; a1.re += b1.re; a1.im += b1.im;
                    }
                }
                C c0 = cxzero<float>(), c1 = cxzero<float>();
                const bool pair = vec_ok && (n + 1 < tl.N);
                if (tl.Cin) {
                    const C* ci = tl.Cin + (size_t)m * tl.ldcin + n;
                    if (pair) {
                        float4 f = *reinterpret_cast<const float4*>(ci);
                        c0 = C(f.x, f.y); c1 = C(f.z, f.w);
                    } else {
                        c0 = ci[0];
                        if (n + 1 < tl.N) c1 = ci[1];
                    }
                    if (n >= tl.mask_lo && n < tl.mask_hi) c0 = cxzero<float>();
                    if (n + 1 >= tl.mask_lo && n + 1 < tl.mask_hi) c1 = cxzero<float>();
                }
                c0.re += tl.sgn * a0.re; c0.im += tl.sgn * a0.im;
                c1.re += tl.sgn * a1.re; c1.im += tl.sgn * a1.im;
                C* co = tl.Cout + (size_t)m * tl.ldc + n;
                if (pair) {
                    *reinterpret_cast<float4*>(co) = make_float4(c0.re, c0.im, c1.re, c1.im);
                } else {
                    co[0] = c0;
                    if (n + 1 < tl.N) co[1] = c1;
                }
                if (emit) { stage[(size_t)rr * C_LD + nloc] = c0; stage[(size_t)rr * C_LD + nloc + 1] = c1; }
            }
        }
        if (warp == FIRST_EPI_WARP) TC2_TRACE(12);
        if (emit && !split) {
            // ---------------- emit the finished tile as operand planes ----------------
            asm volatile("bar.sync 1, %0;" ::"n"(NUM_EPI_WARPS * 32) : "memory");
            const int et = tid - 32 * FIRST_EPI_WARP;  // 0..511
            if (tl.eb_planes && tl.eb_m_lo >= tl.m0 && tl.eb_m_lo < tl.m0 + TM) {
                // B planes of the 64 rows [eb_m_lo, eb_m_lo+64): task = (column, group of 8 rows)
                const int r0 = tl.eb_m_lo - tl.m0;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int e = et + 512 * h;
                    const int nloc = e & (TN - 1), kg = e >> 7;
                    const int n = tl.n0 + nloc;
                    float re[8], im[8];
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        C v = stage[(size_t)(r0 + 8 * kg + c) * C_LD + nloc];
                        if (n >= tl.eb_id_lo && n < tl.eb_id_hi) v = C((n - tl.eb_id_lo == 8 * kg + c) ? 1.f : 0.f, 0.f);
                        if (n >= tl.N) v = cxzero<float>();
                        re[c] = v.re; im[c] = v.im;
                    }
                    uint16_t* chunk = tl.eb_planes + ((size_t)(tl.n0 / TN) * (64 / KC) + (kg >> 1)) * (B_STAGE / 2);
                    store_b8(chunk, nloc, kg & 1, re, im);
                }
            }
            if (tl.ea_planes) {
                const int lo = tl.ea_n_lo > tl.n0 ? tl.ea_n_lo : tl.n0;
                const int hi = tl.ea_n_hi < tl.n0 + TN ? tl.ea_n_hi : tl.n0 + TN;
                const int nJ = hi > lo ? (hi - lo) >> 3 : 0;
                for (int e = et; e < nJ * TM; e += NUM_EPI_WARPS * 32) {
                    const int rr = e & (TM - 1), jj = e >> 7;
                    const int m = tl.m0 + rr;
                    if (m >= tl.Mstore || (m >= tl.skip_lo && m < tl.skip_hi)) continue;
                    const int n8 = lo + 8 * jj;
                    const int tr = m + tl.ea_row_off, tcol = n8 - tl.ea_col_off;
                    float re[8], im[8];
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        C v = stage[(size_t)rr * C_LD + (n8 - tl.n0) + c];
                        if (tr >= tl.ea_zero_from || tcol + c >= tl.ea_zero_from || n8 + c >= tl.N) v = cxzero<float>();
                        re[c] = v.re; im[c] = v.im;
                    }
                    uint16_t* dst = tl.ea_planes + ((size_t)(tr >> 3) * tl.ea_nbc + (tcol >> 3)) * 64 + (tr & 7) * 8;
                    store_a8(dst, tl.ea_plane_elems, re, im);
                }
            }
        }
        }  // rank 0 / unsplit
        if (split) cluster_sync_all();  // rank 1 keeps its staged tile until rank 0 has read it
    }
    if (warp == FIRST_EPI_WARP) TC2_TRACE(13);
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"(TMEM_COLS) : "memory");
        TC2_TRACE(14);
    }
}

// ---------------------------------------------------------------------------------------------
// operand preparation
// ---------------------------------------------------------------------------------------------
// A planes of a batch of FP32 complex matrices.  src(z) = src0 + z*src_stride (row-major, leading dimension ld);
// entries with row >= rows or col >= cols are written as zero.  Destination matrix index = mat0 + z*mat_step.
// grid = (nP/256, nP/8, nbatch), 256 threads: a warp writes 4 adjacent 8x8 blocks (512 contiguous bytes) per plane.
struct ASplitArgs {
    const cx<float>* src0; size_t src_stride; int ld, rows, cols;
    uint16_t* planes; int nP; int mat0, mat_step;
};
__device__ __forceinline__ void a_split_body(const cx<float>* __restrict__ src, int ld, int rows, int cols, uint16_t* __restrict__ dst, int nP) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int I = blockIdx.y, J = blockIdx.x * 32 + w * 4 + (lane >> 3), r = lane & 7;
    if (J * 8 >= nP) return;
    const int row = I * 8 + r, col0 = J * 8;
    float re[8], im[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        cx<float> v = (row < rows && col0 + c < cols) ? src[(size_t)row * ld + col0 + c] : cxzero<float>();
        re[c] = v.re; im[c] = v.im;
    }
    uint32_t wr[3][4], wi[3][4];
#pragma unroll
    for (int qd = 0; qd < 4; ++qd) {
        Split3 sr = split2(re[2 * qd], re[2 * qd + 1]);
        Split3 si = split2(im[2 * qd], im[2 * qd + 1]);
#pragma unroll
        for (int s = 0; s < 3; ++s) { wr[s][qd] = sr.w[s]; wi[s][qd] = si.w[s]; }
    }
#pragma unroll
    for (int s = 0; s < 3; ++s) {
        *reinterpret_cast<uint4*>(dst + aplane_off(nP, s, row, col0)) = make_uint4(wr[s][0], wr[s][1], wr[s][2], wr[s][3]);
        *reinterpret_cast<uint4*>(dst + aplane_off(nP, 3 + s, row, col0)) = make_uint4(wi[s][0], wi[s][1], wi[s][2], wi[s][3]);
    }
}
__global__ void __launch_bounds__(256) a_split_kernel(ASplitArgs a) {
    const int z = blockIdx.z;
    a_split_body(a.src0 + (size_t)z * a.src_stride, a.ld, a.rows, a.cols,
                 a.planes + (size_t)(a.mat0 + z * a.mat_step) * NPL_A * a.nP * a.nP, a.nP);
}

// B planes of one FP32 complex matrix B[k*ldb + n] (K x N); kpad = K rounded up to KC.  grid = (kpad/8, ceil(N/128)), 128 threads.
__global__ void __launch_bounds__(128) b_split_kernel(const cx<float>* __restrict__ B, int ldb, int K, int N, int kpad, uint16_t* __restrict__ planes) {
    const int kg = blockIdx.x, tn = blockIdx.y, r = threadIdx.x;
    const int n = tn * TN + r;
    float re[8], im[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const int k = kg * 8 + c;
        cx<float> v = (k < K && n < N) ? B[(size_t)k * ldb + n] : cxzero<float>();
        re[c] = v.re; im[c] = v.im;
    }
    uint16_t* chunk = planes + ((size_t)tn * (kpad / KC) + (kg >> 1)) * (B_STAGE / 2);
    store_b8(chunk, r, kg & 1, re, im);
}

// ---------------------------------------------------------------------------------------------
// host: tensor maps over an A-plane buffer
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// maps[0]: forward box {64, 2, 16, 6, 1}; maps[1]: adjoint box {64, 16, 2, 6, 1}
// general form: matrices of `rows` x `cols` entries (multiples of 8), planes of rows*cols elements
inline int make_aplane_maps(uint16_t* planes, int rows, int cols, long long nmat, CUtensorMap maps[2]) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled is unavailable (driver too old?)"); return 1; }
    const cuuint64_t nbr = (cuuint64_t)(rows / 8), nbc = (cuuint64_t)(cols / 8);
    const cuuint64_t pl = (cuuint64_t)rows * cols * 2;
    const cuuint64_t dims[5] = {64, nbc, nbr, (cuuint64_t)NPL_A, (cuuint64_t)nmat};
    const cuuint64_t strides[4] = {128, nbc * 128, pl, (cuuint64_t)NPL_A * pl};  // bytes, dims 1..4
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    const cuuint32_t box_f[5] = {64, 2, 16, (cuuint32_t)NPL_A, 1};
    const cuuint32_t box_a[5] = {64, 16, 2, (cuuint32_t)NPL_A, 1};
    for (int i = 0; i < 2; ++i) {
        CUresult r = enc(&maps[i], CU_TENSOR_MAP_DATA_TYPE_UINT16, 5, planes, dims, strides, i == 0 ? box_f : box_a, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with code " + std::to_string((int)r)); return 1; }
    }
    return 0;
}
inline int make_aplane_maps(uint16_t* planes, int nP, long long nmat, CUtensorMap maps[2]) { return make_aplane_maps(planes, nP, nP, nmat, maps); }

}  // namespace tc2
}  // namespace ust
