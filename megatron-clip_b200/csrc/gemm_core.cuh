// Warp-specialised tcgen05 GEMM core for the ClipLoss path (sm_100a only).
//
//   D[M, N] = A[M, K] * B[N, K]^T      16-bit operands (bf16 or fp16), fp32 accumulation in TMEM
//
// CTAs work in PAIRS (cluster of 2, tcgen05 cta_group::2): a pair computes a 256 x 256 tile with UMMA M=256, N=256,
// K=16.  Each CTA loads its own 128 rows of A and HALF of the B tile, so a pipeline stage is 32 KB per CTA instead of
// 48 KB: the measured refill round trip of a stage is ~1900 cycles against 512 cycles of MMA per K block, so the ring
// needs >= 5 stages to keep the tensor pipe busy, which only fits with the halved B (7 stages STATS, 5 + staging
// otherwise).  One CTA = 10 warps: warp 0 = TMA producer, warp 1 = TMEM allocator and, in the even (leader) CTA, the
// single-thread tcgen05.mma issuer for the pair, warps 2..9 = epilogue for the CTA's own 128 accumulator rows (two
// warps per TMEM lane quarter, one per 128-column half).  Three pipelines: the shared-memory ring (TMA -> MMA, full
// barriers in the leader, empty barriers in both CTAs via multicast commit), a 2-stage TMEM accumulator ring
// (MMA -> epilogue) and the unit's tile loop.  K is streamed in 64-element (128-byte, SWIZZLE_128B) blocks.
//
// Epilogue modes (all read the accumulator with tcgen05.ld, thread == one row of the tile):
//   MODE_STATS : online row max / sum-of-exp / sum-of-exp-times-logit of s*A*B^T over a run of column tiles, plus the
//                positive (diagonal) logit.  This is the logits + cross-entropy forward of loss.py:112-119,135-138
//                without storing the logits; the third statistic gives dlogit_scale without touching the backward.
//   MODE_GRAD  : recompute the tile and write G = 2^14 * (alpha*(P_row - Id) + beta*(P_col - Id)) as fp16 into an
//                L2-resident panel.
//   MODE_OUT   : plain fp32 output (optionally accumulating) - the two gradient GEMMs dX = G*Y and dY = G^T*X.
// GRAD and OUT tiles leave the SM through swizzled shared-memory staging and TMA (store / reduce-add), so the global
// writes are full 128-byte lines issued by the copy engine, not 32 scattered 16-byte stores per warp instruction.
// Operands may be K-major (row-major [rows, K]) or MN-major (row-major [K, rows]); the latter lets the gradient
// GEMMs read Y, X and the G panel in place, without transposes.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math_constants.h>

#include "ptx.cuh"

namespace clipk {

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;
constexpr int A_STAGE_BYTES = BM * BK * 2;   // 16 KB
constexpr int B_STAGE_BYTES = (BN / 2) * BK * 2;   // 16 KB: this CTA's half of the pair's 256-column B tile
constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
constexpr int NUM_EPI_WARPS = 8;
constexpr int NUM_THREADS = 64 + NUM_EPI_WARPS * 32;
constexpr int TMEM_COLS = 512;               // 2 accumulator stages x 256 fp32 columns
constexpr int MISC_BYTES = 1024;
// Epilogue staging: every epilogue warp owns two 4 KB buffers (32 rows x 128 B, SWIZZLE_128B) from which its part of
// the tile leaves through TMA (store of the fp16 G tile, store / reduce-add of the fp32 gradient tile).  The STATS
// kernel writes nothing per tile, so it spends that shared memory on two more pipeline stages instead.
constexpr int STG_BYTES = 4096;
constexpr int STG_TOTAL = NUM_EPI_WARPS * 2 * STG_BYTES;   // 64 KB
__host__ __device__ constexpr int stages_of(int mode) { return mode == 0 ? 7 : 5; }
__host__ __device__ constexpr int smem_bytes_of(int mode) {
    return 1024 /*align slack*/ + stages_of(mode) * STAGE_BYTES + 256 + MISC_BYTES + (mode == 0 ? 0 : STG_TOTAL);
}
constexpr int PARTS_PER_UNIT = 2;            // each 128-column half of a tile keeps its own row statistics
constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;

enum Mode { MODE_STATS = 0, MODE_GRAD = 1, MODE_OUT = 2 };

struct KArgs {
    int M, N;             // output extent (rows of A, rows of B)
    int num_kb;           // K blocks of 64 elements over all segments (= nseg * kb_per_seg)
    // K segments: block kb belongs to segment kb / kb_per_seg; a_off/b_off shift the INNER (contiguous) coordinate of
    // the operand for that segment.  16-bit inputs use one segment; fp32 values are held as two scaled fp16 planes
    // [hi | lo] laid side by side and contracted as three plane pairs (lo.hi, hi.lo, hi.hi - small terms first).
    int nseg, kb_per_seg;
    int a_off[3], b_off[3];
    int a_mn, b_mn;       // operand majors (1 = MN-major)
    int f16;              // operands are fp16 (1) or bf16 (0) - BOTH: an instruction descriptor with a_format != b_format
                          // (fp16 panel x bf16 features) ends in an illegal-instruction error on sm_100a (measured, round 2)
    int a_outer_off, b_outer_off;   // added to the OUTER TMA coordinate (row of a K-major operand, K of an MN-major one)
    int c_col_off, c_row_off;       // added to the epilogue's TMA store coordinates
    int n_tiles;          // ceil(N / BN)
    int tiles_per_unit;   // column tiles swept by one CTA (STATS / GRAD); 1 for OUT
    // STATS / GRAD
    const float* scale;        // device scalar logit_scale
    const float* xs;           // device scalars: true value = stored value * (*xs) for A, (*ys) for B; null = 1
    const float* ys;
    long long diag_offset;     // the positive of row i is column diag_offset + i
    float* part_max;           // [parts][M]  running max of s*log2e*acc      (parts = 2 * gridDim.x)
    float* part_sum;           // [parts][M]  sum 2^(v - max)
    float* part_dot;           // [parts][M]  sum 2^(v - max) * v
    float* pos;                // [M] natural-log units, written by the thread whose run contains the diagonal
    // GRAD
    const float* lse_row;      // [M] natural log
    const float* lse_col;      // [N] natural log
    const float* avec;         // [M] 2^(c - Lr_i), c = global reference of this backward (log2 units), from grad_prep
    const float* bvec;         // [N] 2^(c - Lc_j)
    const float* gref;         // [2]: c, fast-path flag (1 = LSE spread small enough for the one-ex2 path)
    float alpha, beta;
    __half* G;                 // panel of G * 2^14 in fp16, row-major, rows padded to BM and ldg to BN
    int ldg;
    int g_planes;              // 1, or 2 (G split into two fp16 planes, g_plane_stride columns apart)
    int g_plane_stride;
    int g_split;               // meaning of the two planes: 0 = [hi | lo] of one G (22 bits, fp32 features);
                               // 1 = [alpha (P_row - Id) | beta (P_col - Id)]: dX reads the first, dY the second
                               // (local_loss without gather_with_grad, loss.py:53-56)
    // OUT
    float* out;
    int ldo;
    int accumulate;
    const float* oscale0;      // out = acc * (*oscale0) * (*oscale1) * (*oscale2) * oconst   (null pointers count as 1)
    const float* oscale1;
    const float* oscale2;
    float oconst;
};

// ---------------------------------------------------------------------------------------------------- epilogues
struct StatsState {
    float m, l, t, pos_raw;
    bool have_pos;
};

template <bool EDGE>
__device__ __forceinline__ void stats_chunk(const uint32_t (&r)[32], float sc, int col0, int ncols, long long dcol,
                                            StatsState& st) {
    float v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = __uint_as_float(r[k]) * sc;
    if (EDGE) {
#pragma unroll
        for (int k = 0; k < 32; ++k)
            if (col0 + k >= ncols) v[k] = -CUDART_INF_F;
    }
    float cmax = v[0];
#pragma unroll
    for (int k = 1; k < 32; ++k) cmax = fmaxf(cmax, v[k]);
    const float m_new = fmaxf(st.m, cmax);
    if (m_new > -CUDART_INF_F) {
        // all 32 ex2 are issued back to back (MUFU latency is paid once, not per element), then reduced with four
        // independent accumulators
        float e[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) e[k] = ptx::ex2(v[k] - m_new);
        float acc[4] = {0.f, 0.f, 0.f, 0.f}, dot[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < 32; ++k) {
            acc[k & 3] += e[k];
            // masked columns have e == 0 but v == -inf: keep 0 * -inf out of the sum
            dot[k & 3] = fmaf(e[k], (EDGE && col0 + k >= ncols) ? 0.f : v[k], dot[k & 3]);
        }
        const float corr = ptx::ex2(st.m - m_new);
        st.l = st.l * corr + ((acc[0] + acc[1]) + (acc[2] + acc[3]));
        st.t = st.t * corr + ((dot[0] + dot[1]) + (dot[2] + dot[3]));
        st.m = m_new;
    }
    if (EDGE) {
        const bool hit = (dcol >= col0) && (dcol < (long long)col0 + 32) && (dcol < ncols);
        if (__any_sync(0xffffffffu, hit)) {
            const int idx = hit ? int(dcol - col0) : -1;
#pragma unroll
            for (int k = 0; k < 32; ++k)
                if (k == idx) st.pos_raw = __uint_as_float(r[k]);
            st.have_pos = st.have_pos || hit;
        }
    }
}

// 16-byte piece `piece` (0..7) of row `row` (0..31) inside a 32 x 128 B SWIZZLE_128B staging buffer
__device__ __forceinline__ uint32_t stg_addr(uint32_t stg, int row, int piece) {
    return stg + row * 128 + ((piece ^ (row & 7)) << 4);
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// 16 columns of the G tile as fp32 values g[16] (still to be packed).
//   FAST (interior tile and the LSE spread of this backward <= 100 in log2 units): ONE ex2 per element.  With the
//        reference c = min over all row and column LSEs,  E = 2^(v - c),  g = E * (A_i + B_j),
//        A_i = ga * 2^(c - Lr_i) (a register), B_j = gb * 2^(c - Lc_j) (a vector prepared once per backward, read
//        through L1 as warp-uniform float4 loads, issued ONE PIECE AHEAD of their use: loaded where they are used
//        they cost a long-scoreboard stall as long as the piece's sixteen ex2).  v <= min(Lr_i, Lc_j) and the spread bound keep every factor in
//        fp32 range; what underflows is below 2^-126 of a probability.  MUFU runs 16 ex2/clk/SM, so two per element
//        would cost exactly the tile's MMA time - this path halves it and needs no per-tile staging or barrier.
//   exact (tile with positives, columns beyond N, or a wide LSE spread): two ex2 per element, exact masking.
__device__ __forceinline__ void grad16_load_b(const float* __restrict__ bv, float4 (&l4)[4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) l4[j] = __ldg(reinterpret_cast<const float4*>(bv) + j);
}
__device__ __forceinline__ void grad16_fast(const uint32_t (&r)[16], float sc, float cref, float Ai, float gb,
                                            const float4 (&l4)[4], float (&g)[16]) {
    float e[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) e[k] = ptx::ex2(fmaf(__uint_as_float(r[k]), sc, -cref));
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        g[4 * j] = e[4 * j] * fmaf(gb, l4[j].x, Ai);
        g[4 * j + 1] = e[4 * j + 1] * fmaf(gb, l4[j].y, Ai);
        g[4 * j + 2] = e[4 * j + 2] * fmaf(gb, l4[j].z, Ai);
        g[4 * j + 3] = e[4 * j + 3] * fmaf(gb, l4[j].w, Ai);
    }
}
__device__ __forceinline__ void grad16_exact(const uint32_t (&r)[16], float sc, float Lr, float ga, float gb,
                                             const float* __restrict__ lse_col, int col0, int ncols, long long dcol,
                                             float (&g)[16]) {
    const int didx = (dcol >= col0 && dcol < (long long)col0 + 16) ? int(dcol - col0) : -1;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const bool inside = col0 + k < ncols;
        const float lc = inside ? __ldg(lse_col + k) * LOG2E : CUDART_INF_F;
        const float v = __uint_as_float(r[k]) * sc;
        float pr = ptx::ex2(v - Lr), pc = ptx::ex2(v - lc);
        if (k == didx) { pr -= 1.f; pc -= 1.f; }
        g[k] = inside ? ga * pr + gb * pc : 0.f;
    }
}
// the same two, with the row part alpha (P_row - Id) and the column part beta (P_col - Id) kept apart (g_split)
__device__ __forceinline__ void grad16_fast2(const uint32_t (&r)[16], float sc, float cref, float Ai, float gb,
                                             const float4 (&l4)[4], float (&gr)[16], float (&gc)[16]) {
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const float e = ptx::ex2(fmaf(__uint_as_float(r[k]), sc, -cref));
        const float b = (k & 3) == 0 ? l4[k >> 2].x : (k & 3) == 1 ? l4[k >> 2].y : (k & 3) == 2 ? l4[k >> 2].z : l4[k >> 2].w;
        gr[k] = e * Ai;
        gc[k] = e * (gb * b);
    }
}
__device__ __forceinline__ void grad16_exact2(const uint32_t (&r)[16], float sc, float Lr, float ga, float gb,
                                              const float* __restrict__ lse_col, int col0, int ncols, long long dcol,
                                              float (&gr)[16], float (&gc)[16]) {
    const int didx = (dcol >= col0 && dcol < (long long)col0 + 16) ? int(dcol - col0) : -1;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const bool inside = col0 + k < ncols;
        const float lc = inside ? __ldg(lse_col + k) * LOG2E : CUDART_INF_F;
        const float v = __uint_as_float(r[k]) * sc;
        float pr = ptx::ex2(v - Lr), pc = ptx::ex2(v - lc);
        if (k == didx) { pr -= 1.f; pc -= 1.f; }
        gr[k] = inside ? ga * pr : 0.f;
        gc[k] = inside ? gb * pc : 0.f;
    }
}
__device__ __forceinline__ void grad16_store2(const float (&gr)[16], const float (&gc)[16], uint32_t stg, uint32_t stg2, int lane,
                                              int piece0) {
    uint32_t pk[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) pk[k] = ptx::pack_f16x2(gr[2 * k], gr[2 * k + 1]);
    st_shared_v4(stg_addr(stg, lane, piece0), pk[0], pk[1], pk[2], pk[3]);
    st_shared_v4(stg_addr(stg, lane, piece0 + 1), pk[4], pk[5], pk[6], pk[7]);
#pragma unroll
    for (int k = 0; k < 8; ++k) pk[k] = ptx::pack_f16x2(gc[2 * k], gc[2 * k + 1]);
    st_shared_v4(stg_addr(stg2, lane, piece0), pk[0], pk[1], pk[2], pk[3]);
    st_shared_v4(stg_addr(stg2, lane, piece0 + 1), pk[4], pk[5], pk[6], pk[7]);
}
// g[16] -> fp16, into 16-byte pieces [piece0, piece0 + 2) of this row's line of the staging buffer(s): 128-byte rows
// in SWIZZLE_128B order, or (DENSE64) 64-byte rows in SWIZZLE_64B order - the half-size buffers of the A-resident
// recompute kernel
template <bool TWO_PLANES, bool DENSE64 = false>
__device__ __forceinline__ void grad16_store(const float (&g)[16], uint32_t stg, uint32_t stg_lo, int lane, int piece0) {
    uint32_t pk[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) pk[k] = ptx::pack_f16x2(g[2 * k], g[2 * k + 1]);
    if (DENSE64) {
        // 64-byte rows in SWIZZLE_64B order: the 16-byte chunk index is XORed with bits 7..8 of the address = (row / 2) % 4,
        // so the 32 lanes of one store cover all 32 banks four times instead of 8 banks sixteen times
        const int sw = (lane >> 1) & 3;
        st_shared_v4(stg + lane * 64 + ((piece0 ^ sw) << 4), pk[0], pk[1], pk[2], pk[3]);
        st_shared_v4(stg + lane * 64 + (((piece0 + 1) ^ sw) << 4), pk[4], pk[5], pk[6], pk[7]);
        return;
    }
    st_shared_v4(stg_addr(stg, lane, piece0), pk[0], pk[1], pk[2], pk[3]);
    st_shared_v4(stg_addr(stg, lane, piece0 + 1), pk[4], pk[5], pk[6], pk[7]);
    if (TWO_PLANES) {
        // residual plane: g = hi + lo, each piece exactly representable in fp16 (22 bits together)
        uint32_t lo[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float h0 = __half2float(__ushort_as_half((unsigned short)(pk[k] & 0xffffu)));
            const float h1 = __half2float(__ushort_as_half((unsigned short)(pk[k] >> 16)));
            lo[k] = ptx::pack_f16x2(g[2 * k] - h0, g[2 * k + 1] - h1);
        }
        st_shared_v4(stg_addr(stg_lo, lane, piece0), lo[0], lo[1], lo[2], lo[3]);
        st_shared_v4(stg_addr(stg_lo, lane, piece0 + 1), lo[4], lo[5], lo[6], lo[7]);
    }
}

// ---------------------------------------------------------------------------------------------------- CTA body
// The body is split into per-role "unit" functions that carry their pipeline state (ring stage / phase, accumulator
// stage, staging-buffer use) across calls, so the same code serves the one-unit-per-CTA kernels and the persistent
// backward kernel that walks many units per CTA.
struct Cta {
    uint32_t sA, sB, sStg, bar_full, bar_empty, bar_tfull, bar_tempty, bar_afull, bar_aempty, tmem_base;
    uint32_t cta_rank;
    bool leader;
    int warp, lane;
};
struct Pipe {
    int s = 0;          // shared-memory ring stage (producer / MMA)
    uint32_t ph = 0;    // its phase
    int it = 0;         // tiles processed so far (MMA / epilogue): accumulator stage = it & 1
    int stg_use = 0;    // TMA stores issued so far by this epilogue warp
};

// Shared memory: A region (A_BYTES) | NB B stages | epilogue staging | barriers.  The streaming kernels use one A slot
// per stage (A_BYTES = STAGES * A_STAGE_BYTES, NB = STAGES); the A-resident forward keeps all K blocks of its rows.
template <int STAGES, int EXTRA_BYTES, int A_BYTES = STAGES * A_STAGE_BYTES>
__device__ __forceinline__ Cta cta_setup() {
    Cta c;
    c.cta_rank = ptx::cluster_ctarank();   // 0 = leader (issues the pair's MMAs), 1 = peer
    c.leader = (c.cta_rank == 0);
    c.warp = threadIdx.x >> 5;
    c.lane = threadIdx.x & 31;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw_u32 = ptx::smem_u32(smem_raw);
    const uint32_t base = (raw_u32 + 1023u) & ~1023u;
    uint8_t* base_ptr = smem_raw + (base - raw_u32);
    // layout (1024-byte aligned up to the barriers): A stages | B stages | epilogue staging | barriers
    constexpr uint32_t kStg = uint32_t(EXTRA_BYTES);   // epilogue staging (GRAD / OUT) or the column buffer (forward sweep)
    c.sA = base;
    c.sB = c.sA + A_BYTES;
    c.sStg = c.sB + STAGES * B_STAGE_BYTES;
    const uint32_t sBar = c.sStg + kStg;
    c.bar_full = sBar;
    c.bar_empty = sBar + STAGES * 8;
    c.bar_tfull = sBar + 2 * STAGES * 8;
    c.bar_tempty = c.bar_tfull + 16;
    c.bar_afull = c.bar_tempty + 16;
    c.bar_aempty = c.bar_afull + 8;
    const uint32_t sTmemPtr = c.bar_aempty + 8;
    volatile uint32_t* tmem_ptr_gen =
        reinterpret_cast<volatile uint32_t*>(base_ptr + A_BYTES + STAGES * B_STAGE_BYTES + kStg + (2 * STAGES + 6) * 8);

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            ptx::mbar_init(c.bar_full + 8 * s, 1);
            ptx::mbar_init(c.bar_empty + 8 * s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            ptx::mbar_init(c.bar_tfull + 8 * a, 1);
            ptx::mbar_init(c.bar_tempty + 8 * a, 2 * NUM_EPI_WARPS);   // epilogue warps of both CTAs (leader's copy is used)
        }
        ptx::mbar_init(c.bar_afull, 1);
        ptx::mbar_init(c.bar_aempty, 1);
        ptx::fence_barrier_init();
    }
    if (c.warp == 1) {
        ptx::tmem_alloc_pair(sTmemPtr, TMEM_COLS);
        ptx::tmem_relinquish_pair();
    }
    ptx::tc_fence_before();
    ptx::cluster_sync();          // barriers of both CTAs initialised, TMEM allocated, before any remote arrive / TMA
    ptx::tc_fence_after();
    // Programmatic dependent launch: everything above overlapped the tail of the previous kernel in the stream; from
    // here on global memory written by it is read (and memory it reads is overwritten), so wait for it to finish.
    ptx::pdl_launch_dependents();
    ptx::pdl_wait();
    c.tmem_base = *tmem_ptr_gen;
    return c;
}

__device__ __forceinline__ void cta_teardown(const Cta& c) {
    // neither CTA may exit (or free TMEM) while its peer can still read its shared memory or signal its barriers
    ptx::tc_fence_before();
    ptx::cluster_sync();
    if (c.warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc_pair(c.tmem_base, TMEM_COLS);
    }
}

// ------------------------------------------------------------------ TMA producer (one lane of warp 0, both CTAs)
// loads of K block `kb` of segment `seg` for output tile (m_blk, t) into the next ring stage
template <int STAGES>
__device__ __forceinline__ void load_kblock(const Cta& c, Pipe& p, const CUtensorMap* tmA, const CUtensorMap* tmB,
                                            const KArgs& args, int m_blk, int t, int seg, int kb) {
    const int kw = kb * BK;
    const int ao = args.a_off[seg], bo = args.b_off[seg];
    ptx::mbar_wait(c.bar_empty + 8 * p.s, p.ph ^ 1);
    // both CTAs' loads complete on the LEADER's full barrier, which expects the bytes of the pair
    const uint32_t full = c.bar_full + 8 * p.s;
    if (c.leader) ptx::mbar_arrive_expect_tx(full, 2 * STAGE_BYTES);
    const uint32_t a_dst = c.sA + p.s * A_STAGE_BYTES;
    const uint32_t b_dst = c.sB + p.s * B_STAGE_BYTES;
    const int bn0 = t * BN + int(c.cta_rank) * (BN / 2);   // this CTA's half of the B tile
    if (args.a_mn) {
#pragma unroll
        for (int i = 0; i < BM / 64; ++i)
            ptx::tma_load_2d_pair(a_dst + i * 8192, tmA, ao + m_blk * BM + i * 64, args.a_outer_off + kw, full);
    } else {
        ptx::tma_load_2d_pair(a_dst, tmA, ao + kw, args.a_outer_off + m_blk * BM, full);
    }
    if (args.b_mn) {
#pragma unroll
        for (int i = 0; i < BN / 128; ++i)
            ptx::tma_load_2d_pair(b_dst + i * 8192, tmB, bo + bn0 + i * 64, args.b_outer_off + kw, full);
    } else {
        ptx::tma_load_2d_pair(b_dst, tmB, bo + kw, args.b_outer_off + bn0, full);
    }
    if (++p.s == STAGES) { p.s = 0; p.ph ^= 1; }
}

template <int STAGES>
__device__ __forceinline__ void produce_unit(const Cta& c, Pipe& p, const CUtensorMap* tmA, const CUtensorMap* tmB,
                                             const KArgs& args, int m_blk, int t0, int t1) {
    for (int t = t0; t < t1; ++t) {
        for (int kb = 0; kb < args.num_kb; ++kb) {
            const int seg = kb / args.kb_per_seg;
            load_kblock<STAGES>(c, p, tmA, tmB, args, m_blk, t, seg, kb - seg * args.kb_per_seg);
        }
    }
}

// ------------------------------------------------------------------ MMA issuer (one lane of warp 1, leader CTA only)
template <int STAGES>
__device__ __forceinline__ void mma_unit(const Cta& c, Pipe& p, const KArgs& args, int ntiles) {
    const int a_mn = args.a_mn, b_mn = args.b_mn;
    const int num_kb = args.num_kb;
    const uint32_t idesc = ptx::make_idesc_16bit(2 * BM, BN, a_mn, b_mn, /*a_is_bf16=*/!args.f16, /*b_is_bf16=*/!args.f16);
    // K-major SW128: 8-row groups 1024 B apart (SBO); MN-major SW128: 64-wide MN blocks 8192 B apart (LBO),
    // 8-row K groups 1024 B apart (SBO).
    const uint64_t adesc_hi = a_mn ? ptx::make_smem_desc_sw128(8192, 1024) : ptx::make_smem_desc_sw128(16, 1024);
    const uint64_t bdesc_hi = b_mn ? ptx::make_smem_desc_sw128(8192, 1024) : ptx::make_smem_desc_sw128(16, 1024);
    const uint32_t a_kstep = a_mn ? 2048 : 32;   // bytes per UMMA_K = 16 elements
    const uint32_t b_kstep = b_mn ? 2048 : 32;
    for (int t = 0; t < ntiles; ++t, ++p.it) {
        const int a = p.it & 1;
        const uint32_t aph = (p.it >> 1) & 1;
        ptx::mbar_wait(c.bar_tempty + 8 * a, aph ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = c.tmem_base + a * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
            ptx::mbar_wait(c.bar_full + 8 * p.s, p.ph);
            ptx::tc_fence_after();
            const uint32_t a_src = c.sA + p.s * A_STAGE_BYTES;
            const uint32_t b_src = c.sB + p.s * B_STAGE_BYTES;
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
                ptx::mma_f16_ss_pair(d_tmem, ptx::desc_with_addr(adesc_hi, a_src + k * a_kstep),
                                     ptx::desc_with_addr(bdesc_hi, b_src + k * b_kstep), idesc, (kb | k) != 0);
            }
            ptx::mma_commit_pair(c.bar_empty + 8 * p.s);
            if (++p.s == STAGES) { p.s = 0; p.ph ^= 1; }
        }
        ptx::mma_commit_pair(c.bar_tfull + 8 * a);
    }
}

// ------------------------------------------------------------------ epilogue (warps 2..9, both CTAs)
// STATS and OUT tiles (the recompute tiles have their own epilogue below)
template <int MODE>
__device__ __forceinline__ void epilogue_unit(const Cta& c, Pipe& p, const CUtensorMap* tmC, const KArgs& args, int m_blk,
                                              int unit, int t0, int t1, int row_shift = 0) {
    static_assert(MODE == MODE_STATS || MODE == MODE_OUT, "GRAD tiles go through grad_epilogue_unit");
    const int warp = c.warp, lane = c.lane;
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;             // which 128-column half of the tile this warp drains
    const int row = m_blk * BM + q * 32 + lane;
    const bool row_ok = row < args.M;
    const long long dcol = args.diag_offset + row;

    // acc holds the dot product of the STORED operands; dequant = xs*ys turns it into the true x.y
    float sc = 0.f, s_nat = 0.f, oscale = 1.f;
    if (MODE == MODE_STATS) {
        float dequant = 1.f;
        if (args.xs) dequant *= __ldg(args.xs);
        if (args.ys) dequant *= __ldg(args.ys);
        s_nat = __ldg(args.scale) * dequant;      // S = s_nat * acc
        sc = s_nat * LOG2E;
    } else {
        oscale = args.oconst;
        if (args.oscale0) oscale *= __ldg(args.oscale0);
        if (args.oscale1) oscale *= __ldg(args.oscale1);
        if (args.oscale2) oscale *= __ldg(args.oscale2);
    }
    StatsState st{-CUDART_INF_F, 0.f, 0.f, 0.f, false};
    const uint32_t stg0 = c.sStg + (warp - 2) * 2 * STG_BYTES;   // this warp's two staging buffers
    const int accumulate = args.accumulate, ncols = args.N;
    const int c_col_off = args.c_col_off, c_row_off = args.c_row_off + row_shift;   // row_shift: output row of a peer slot

    for (int t = t0; t < t1; ++t, ++p.it) {
        const int a = p.it & 1;
        const uint32_t aph = (p.it >> 1) & 1;
        const int n0 = t * BN;
        ptx::mbar_wait(c.bar_tfull + 8 * a, aph);
        ptx::tc_fence_after();
        const uint32_t taddr = c.tmem_base + a * BN + half * (BN / 2) + (uint32_t(q * 32) << 16);
        // edge tile: contains positives (diagonal entries) of this CTA's rows, or columns beyond N
        const long long d_lo = args.diag_offset + (long long)m_blk * BM;
        const bool edge = (MODE == MODE_STATS) &&
                          (((d_lo + BM - 1 >= n0) && (d_lo < (long long)n0 + BN)) || (n0 + BN > ncols));
        const int colh = n0 + half * (BN / 2);          // first column of this warp's half tile
        const int row0 = m_blk * BM + q * 32;           // first row of this warp

        auto process = [&](const uint32_t (&r)[32], int cidx) {
            const int col0 = colh + cidx * 32;
            if (MODE == MODE_STATS) {
                if (edge) stats_chunk<true>(r, sc, col0, ncols, dcol, st);
                else stats_chunk<false>(r, sc, col0, ncols, dcol, st);
            } else {  // MODE_OUT: 32 fp32 columns = 128 B per row = one staging buffer and one TMA store / reduce
                // before rewriting a staging buffer: at most one older bulk store may still be reading shared memory
                if (lane == 0) ptx::tma_store_wait_read<1>();
                __syncwarp();
                const uint32_t stg = stg0 + (p.stg_use & 1) * STG_BYTES;
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    st_shared_v4(stg_addr(stg, lane, j), __float_as_uint(__uint_as_float(r[4 * j]) * oscale),
                                 __float_as_uint(__uint_as_float(r[4 * j + 1]) * oscale),
                                 __float_as_uint(__uint_as_float(r[4 * j + 2]) * oscale),
                                 __float_as_uint(__uint_as_float(r[4 * j + 3]) * oscale));
                ptx::fence_proxy_async_smem();
                __syncwarp();
                ++p.stg_use;
                if (lane == 0) {
                    // the tensor map clips rows and columns beyond the output matrix
                    if (accumulate) ptx::tma_reduce_add_2d(tmC, stg, c_col_off + col0, c_row_off + row0);
                    else ptx::tma_store_2d(tmC, stg, c_col_off + col0, c_row_off + row0);
                    ptx::tma_store_commit();
                }
            }
        };

        // TMEM loads are double buffered: the load of chunk c+1 is in flight while chunk c is processed, and the
        // accumulator stage goes back to the MMA warp as soon as the last load has landed in registers.
        uint32_t ra[32], rb[32];
        ptx::tmem_ld_32x32(taddr, ra);
        ptx::tmem_ld_wait();
        ptx::tmem_ld_32x32(taddr + 32, rb);
        process(ra, 0);
        ptx::tmem_ld_wait();
        ptx::tmem_ld_32x32(taddr + 64, ra);
        process(rb, 1);
        ptx::tmem_ld_wait();
        ptx::tmem_ld_32x32(taddr + 96, rb);
        process(ra, 2);
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_leader(c.bar_tempty + 8 * a);
        process(rb, 3);
    }

    if (MODE == MODE_STATS) {
        if (row_ok) {
            const size_t slot = (size_t)(unit * PARTS_PER_UNIT + half) * args.M + row;
            args.part_max[slot] = st.m;
            args.part_sum[slot] = st.l;
            args.part_dot[slot] = st.t;
            if (st.have_pos) args.pos[row] = st.pos_raw * s_nat;
        }
    }
}

// Recompute tiles: S tile -> G tile (fp16, x 2^14) -> swizzled staging -> TMA store into the L2-resident panel.
// The tile is drained in 16-column pieces (tcgen05.ld x16, double buffered) to keep the live registers well under the
// 168 a 10-warp CTA allows; four pieces (64 columns = 128 B of fp16 per row) fill one staging buffer = one TMA store.
// NBUF = 4 KB of staging per warp: 2 (two 64-column buffers, one fills while the other leaves; both planes of a
// two-plane G) or 1 (the A-resident recompute kernel, whose shared memory goes to the resident rows: its 4 KB are two
// 32-column half buffers of 64-byte rows, written and stored alternately through a SWIZZLE_64B tensor map).
template <bool TWO_PLANES, int NBUF = 2, bool SPLIT = false>
__device__ __forceinline__ void grad_epilogue_unit(const Cta& c, Pipe& p, const CUtensorMap* tmC, const KArgs& args,
                                                   int m_blk, int t0, int t1) {
    static_assert(NBUF == 2 || !TWO_PLANES, "a two-plane G needs both staging buffers");
    static_assert(TWO_PLANES || !SPLIT, "the row / column split is a two-plane layout");
    const int warp = c.warp, lane = c.lane;
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row = m_blk * BM + q * 32 + lane;
    const bool row_ok = row < args.M;
    const long long dcol = args.diag_offset + row;
    float dequant = 1.f;
    if (args.xs) dequant *= __ldg(args.xs);
    if (args.ys) dequant *= __ldg(args.ys);
    const float sc = __ldg(args.scale) * dequant * LOG2E;
    // G is stored as 2^14 * (alpha*(P_row-Id) + beta*(P_col-Id)) in fp16: |.| <= 2^15 and entries down to
    // ~4e-9 keep the full 11-bit mantissa; logit_scale * gscale * 2^-14 is applied by the gradient GEMMs.
    const float ga = 16384.f * args.alpha, gb = 16384.f * args.beta;
    const float Lr = row_ok ? __ldg(args.lse_row + row) * LOG2E : CUDART_INF_F;   // rows beyond M: every probability is 0
    const float cref = __ldg(args.gref);
    const bool fast = __ldg(args.gref + 1) != 0.f;
    const float Ai = row_ok ? ga * __ldg(args.avec + row) : 0.f;
    const float* __restrict__ bvec = args.bvec;
    const float* __restrict__ lse_col = args.lse_col;
    const int ncols = args.N, plane_stride = args.g_plane_stride;
    const int c_col_off = args.c_col_off, c_row_off = args.c_row_off + m_blk * BM + q * 32;
    const long long d_lo = args.diag_offset + (long long)m_blk * BM;
    const uint32_t stg0 = c.sStg + (warp - 2) * NBUF * STG_BYTES;   // this warp's staging buffer(s)

    for (int t = t0; t < t1; ++t, ++p.it) {
        const int a = p.it & 1;
        const uint32_t aph = (p.it >> 1) & 1;
        const int n0 = t * BN;
        const int colh = n0 + half * (BN / 2);          // first column of this warp's half tile
        if (lane < 4 && t + 1 < t1) {
            // pull the B_j / LSE values of this warp's half of the NEXT tile (512 B) into L1 ahead of their use
            const int cn = colh + BN + lane * 32;
            if (cn + 32 <= ncols) {
                asm volatile("prefetch.global.L1 [%0];" ::"l"(bvec + cn));
                asm volatile("prefetch.global.L1 [%0];" ::"l"(lse_col + cn));
            }
        }
        // edge tile: contains positives (diagonal entries) of this CTA's rows, or columns beyond N
        const bool exact = !fast || ((d_lo + BM - 1 >= n0) && (d_lo < (long long)n0 + BN)) || (n0 + BN > ncols);
        // B_j of the piece in hand and of the next one (fast tiles only; the exact form reads lse_col itself); the
        // first piece's are on their way while this warp waits for the accumulator
        float4 bq[2][4];
        if (!exact) grad16_load_b(bvec + colh, bq[0]);
        ptx::mbar_wait(c.bar_tfull + 8 * a, aph);
        ptx::tc_fence_after();
        const uint32_t taddr = c.tmem_base + a * BN + half * (BN / 2) + (uint32_t(q * 32) << 16);

        uint32_t stg = 0, stg_lo = 0;
        auto piece = [&](const uint32_t (&r)[16], int pi) {
            const int col0 = colh + pi * 16;
            const float4 (&bcur)[4] = bq[pi & 1];
            if (!exact && pi + 1 < 8) grad16_load_b(bvec + col0 + 16, bq[(pi + 1) & 1]);
            if (NBUF == 1) {
                // half buffers of 32 columns: two pieces each
                if ((pi & 1) == 0) {
                    if (lane == 0) ptx::tma_store_wait_read<1>();
                    __syncwarp();
                    stg = stg0 + (p.stg_use & 1) * (STG_BYTES / 2);
                }
                float g[16];
                if (exact) grad16_exact(r, sc, Lr, ga, gb, lse_col + col0, col0, ncols, dcol, g);
                else grad16_fast(r, sc, cref, Ai, gb, bcur, g);
                grad16_store<false, true>(g, stg, 0, lane, (pi & 1) * 2);
                if (pi & 1) {
                    ptx::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        ptx::tma_store_2d(tmC, stg, c_col_off + col0 - 16, c_row_off);
                        ptx::tma_store_commit();
                    }
                    ++p.stg_use;
                }
                return;
            }
            if ((pi & 3) == 0) {
                // (re)use of a staging buffer: at most one older bulk store may still be reading shared memory; with
                // two planes both buffers are written, so nothing of this warp may still be in flight
                if (lane == 0) {
                    if (TWO_PLANES) ptx::tma_store_wait_read<0>();
                    else ptx::tma_store_wait_read<1>();
                }
                __syncwarp();
                stg = stg0 + (p.stg_use & 1) * STG_BYTES;
                stg_lo = stg0 + ((p.stg_use + 1) & 1) * STG_BYTES;
            }
            if (SPLIT) {
                float gr[16], gc[16];
                if (exact) grad16_exact2(r, sc, Lr, ga, gb, lse_col + col0, col0, ncols, dcol, gr, gc);
                else grad16_fast2(r, sc, cref, Ai, gb, bcur, gr, gc);
                grad16_store2(gr, gc, stg, stg_lo, lane, (pi & 3) * 2);
            } else {
                float g[16];
                if (exact) grad16_exact(r, sc, Lr, ga, gb, lse_col + col0, col0, ncols, dcol, g);
                else grad16_fast(r, sc, cref, Ai, gb, bcur, g);
                grad16_store<TWO_PLANES>(g, stg, stg_lo, lane, (pi & 3) * 2);
            }
            if ((pi & 3) == 3) {
                ptx::fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    ptx::tma_store_2d(tmC, stg, c_col_off + col0 - 48, c_row_off);
                    if (TWO_PLANES) ptx::tma_store_2d(tmC, stg_lo, c_col_off + plane_stride + col0 - 48, c_row_off);
                    ptx::tma_store_commit();
                }
                p.stg_use += TWO_PLANES ? 2 : 1;
            }
        };

        uint32_t ra[16], rb[16];
        ptx::tmem_ld_32x16(taddr, ra);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int pi = 0; pi < 8; pi += 2) {
            ptx::tmem_ld_32x16(taddr + (pi + 1) * 16, rb);
            piece(ra, pi);
            ptx::tmem_ld_wait();
            if (pi + 2 < 8) {
                ptx::tmem_ld_32x16(taddr + (pi + 2) * 16, ra);
            } else {
                // the last load has landed: the accumulator stage goes back to the MMA warp
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive_leader(c.bar_tempty + 8 * a);
            }
            piece(rb, pi + 1);
            if (pi + 2 < 8) ptx::tmem_ld_wait();
        }
    }
}

// Before the CTA exits: the bulk stores of this epilogue warp have READ their shared-memory source.  Their global
// writes may still be in flight - the grid does not complete before they have been performed, so the next kernel of
// the stream sees them - which lets slow destinations (peer accumulators over NVLink) drain under the next kernel.
__device__ __forceinline__ void epilogue_drain(const Cta& c) {
    if (c.lane == 0) ptx::tma_store_wait_read<0>();
    __syncwarp();
}
// all bulk stores of this epilogue warp complete (writes performed): before publishing them to other CTAs of the SAME grid
__device__ __forceinline__ void epilogue_drain_complete(const Cta& c) {
    if (c.lane == 0) ptx::tma_store_wait<0>();
    __syncwarp();
}
// ---------------------------------------------------------------------------------------------------- kernels
// One unit per CTA pair: grid = (2 * m_pairs, units), cluster (2, 1, 1).
template <int MODE, int F16>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmC, const KArgs args) {
    constexpr int STAGES = stages_of(MODE);
    const Cta c = cta_setup<STAGES, MODE != MODE_STATS ? STG_TOTAL : 0>();
    const int m_blk = int(blockIdx.x);          // = 2 * m_pair + cta_rank
    const int unit = int(blockIdx.y);
    const int t0 = unit * args.tiles_per_unit;
    const int t1 = min(args.n_tiles, t0 + args.tiles_per_unit);
    Pipe p;
    if (c.warp == 0) {
        if (c.lane == 0) {
            ptx::prefetch_tmap(&tmA);
            ptx::prefetch_tmap(&tmB);
            produce_unit<STAGES>(c, p, &tmA, &tmB, args, m_blk, t0, t1);
        }
    } else if (c.warp == 1) {
        if (c.lane == 0 && c.leader) mma_unit<STAGES>(c, p, args, t1 - t0);
    } else {
        if (MODE == MODE_GRAD) {
            if (args.g_planes == 2 && args.g_split) grad_epilogue_unit<true, 2, true>(c, p, &tmC, args, m_blk, t0, t1);
            else if (args.g_planes == 2) grad_epilogue_unit<true>(c, p, &tmC, args, m_blk, t0, t1);
            else grad_epilogue_unit<false>(c, p, &tmC, args, m_blk, t0, t1);
        } else {
            epilogue_unit<MODE == MODE_GRAD ? MODE_OUT : MODE>(c, p, &tmC, args, m_blk, unit, t0, t1);
        }
        if (MODE != MODE_STATS) epilogue_drain(c);
    }
    cta_teardown(c);
}

// ---------------------------------------------------------------------------------------------------- forward sweep
// Persistent forward kernel: one CTA pair per SM pair walks work items (256 rows x a run of column tiles).
//
// A-resident (ARES, K <= 512).  The 128 rows of A a CTA needs stay in shared memory for a whole run of column tiles
// (128 KB) and only the B half-tiles stream (16 KB per K block and CTA), which halves the L2 -> SM traffic of the
// mainloop.  For longer K (d = 768, 1024) the same kernel streams A with B, one K block per stage.
//
// Single sweep.  The forward needs the log-sum-exp of every ROW and of every COLUMN of the block (loss.py:135-138 takes
// the cross-entropy of logits_per_image and of logits_per_text).  Both come from ONE pass over the tiles when the
// logits are bounded: with u >= |v| for every logit v (log2 units; u = s * max|x_i| * max|y_j| * log2(e) from the row
// norms) ONE exponential per element, e = 2^(v - c) with the global reference c = u - 90, serves both directions: it
// never overflows (e <= 2^90, sums of 2^20 terms and their products with |v - c| < 2^8 stay below 2^127), and every
// element within 2^-24 of ANY possible row or column maximum (>= -u) is a normal fp32 number as long as
// -2u - 24 + 90 >= -126, i.e. u <= 96 (logit_scale * norms <= 66).  Sums are then plain additions (no running
// maximum, no rescaling) and partial sums can be merged in any order.
// The accumulator is read in the 16x256b fragment layout (a thread holds 2 rows x 8 columns of a 16-lane half-chunk),
// which makes the column sums cheap: 3 additions over the 4 rows a thread sees per chunk, then a 3-step butterfly over
// the 8 threads that share the columns; the 4 lane-quarter warps are merged through shared memory and every CTA
// writes one partial (sum, dot) per column and 128-row block, summed later by fwd_merge_kernel.
// When the bound does not hold (logit_scale * norms > ~66) the same launch runs the exact online-max row sweep
// instead and a second launch with the operands swapped produces the column statistics; when it holds the second
// launch exits at once.  The decision is taken on the device from device scalars: no host synchronisation.
constexpr int ARES_KB = 8;                       // resident K blocks (K <= 512)
constexpr int FWD_STAGES = 5;
constexpr int COLBUF_BYTES = 2 * 2 * 4 * 128 * 2 * 4;   // [tile parity][half][lane quarter][128 columns][sum, dot]
__host__ __device__ constexpr int smem_bytes_fwd(bool ares = true) {
    return 1024 + (ares ? ARES_KB : FWD_STAGES) * A_STAGE_BYTES + FWD_STAGES * B_STAGE_BYTES + COLBUF_BYTES + 256 + MISC_BYTES;
}
constexpr float FWD_SAFE_U = 96.f;               // -2u - 24 + FWD_REF_SHIFT >= -126
constexpr float FWD_REF_SHIFT = 90.f;            // reference c = u - 90: uses the overflow headroom of fp32 as well
constexpr float FWD_POS_MARGIN = 175.f;          // rule (b) of fwd_bound: 90 + 102 - 17 (terms of up to 2^17 rows may flush)

struct FwdArgs {
    int M, N;                  // rows of A (X), rows of B (Y)
    int num_kb;                // K blocks (<= ARES_KB in the A-resident kernel)
 int n_tiles, m_pairs;
    int n_clusters;            // clusters of the launch (the part index of a unit is derived from it)
    int pass;                  // 0: X rows against Y columns; 1: the swapped launch (exact mode only)
    int force_exact;           // operands are not plain bf16: no norm bound
    const float* scale;
    const float* xs;           // dequant scalars of the operands (null = 1)
    const float* ys;
    const float* stats;        // [nstat][STAT_WORDS] operand statistics (one row per data-parallel rank, see OperandStats);
    int nstat;                 //   only read when !force_exact
    int stats_rank;            // row of THIS rank: its max |x_i|^2 bounds the rows of the block, every row's max |y_j|^2 the columns
    int use_minpos;            // the positives' lower bound covers every row and column of the problem (see fwd_bound)
    float* mode_out;           // word [5] of this rank's statistics row: 1 = single sweep taken, 0 = exact two-sweep form
    long long diag_offset;
    float* part_max;           // [max parts * 2][M]; part = cluster - first cluster that touches the row pair
    float* part_sum;
    float* part_dot;
    float* pos;                // [M] or null
    float* colpart_sum;        // [2 * m_pairs][ldc]   (pass 0, single sweep)
    float* colpart_dot;
    int ldc;
};

// Operand statistics, one row of STAT_WORDS floats per rank, filled by prep_kernel (clipk.cu):
//   [0] max_i |x_i|^2   [1] max_j |y_j|^2   [2] max |x_ij|   [3] max |y_ij|      (bit patterns of non-negative floats;
//                                                                                  +Inf bits when a NaN / Inf was seen)
//   [4] min_i x_i . y_i over the rank's positive pairs, as an order-REVERSING unsigned code whose maximum is taken
//       (0 = no pair seen; decoded by stat_min_pos)
//   [5] written by fwd_merge_kernel: 1 when the forward took the single sweep, 0 for the exact two-sweep form
constexpr int STAT_WORDS = 8;
__host__ __device__ __forceinline__ int float_to_ordered(float f) {
#ifdef __CUDA_ARCH__
    const int i = __float_as_int(f);
#else
    int i; memcpy(&i, &f, 4);
#endif
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float ordered_to_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

__device__ __forceinline__ float stat_min_pos(float word) {
    const unsigned int u = __float_as_uint(word);
    if (u == 0u) return CUDART_INF_F;                 // no positive pair was seen
    return ordered_to_float(int((~u) ^ 0x80000000u));
}

// The reference c of the single sweep (log2 units) and whether the single sweep is allowed; identical in every thread of
// every CTA of both launches and of the merge kernel.  With u >= |v| for every logit v (from the row norms) and
// c = u - 90 nothing overflows.  What must not happen is that the terms that matter for some row or column flush to
// zero: the sweep is allowed when
//   (a) u <= 96: every logit lies within 192 of any possible maximum, or
//   (b) every row and every column is known to hold a logit >= u - 175: its own positive.  min_i x_i . y_i over ALL
//       pairs of the problem (all ranks) is part of the statistics; with it a trained model at logit_scale = 100
//       (u = 144 for unit vectors) keeps the single sweep as long as no positive pair has a cosine below -0.21.
//       A column's partial sum on a rank that holds none of its large terms may then lose terms below 2^-126 * 2^c:
//       at least 2^85 times smaller than the column's positive, i.e. below fp32 resolution even summed over 2^20 rows.
__device__ __forceinline__ bool fwd_bound(const FwdArgs& a, float* c_out) {
    if (a.force_exact) { *c_out = 0.f; return false; }
    float ny2 = 0.f, minpos = CUDART_INF_F;
    for (int r = 0; r < a.nstat; ++r) {
        const float* st = a.stats + r * STAT_WORDS;
        ny2 = fmaxf(ny2, __ldg(st + 1));
        minpos = fminf(minpos, stat_min_pos(__ldg(st + 4)));
    }
    const float nx2 = __ldg(a.stats + a.stats_rank * STAT_WORDS);
    const float s = __ldg(a.scale);
    const float u = fabsf(s) * sqrtf(nx2) * sqrtf(ny2) * (LOG2E * 1.001f);
    *c_out = u - FWD_REF_SHIFT;
    const bool by_norm = u <= FWD_SAFE_U;                                     // false for NaN / Inf
    const bool by_pos = a.use_minpos && s > 0.f && u < 1e30f && s * LOG2E * minpos >= u - FWD_POS_MARGIN;
    return by_norm || by_pos;
}

// one 16-lane half-chunk (2 rows x 8 columns per thread) of the single sweep
template <bool EDGE>
__device__ __forceinline__ void rowcol_half(const uint32_t (&r)[16], float sc, float u, float& l0, float& t0, float& l1,
                                            float& t1, float (&cs)[8], float (&cd)[8], bool first, int col0, int ncols,
                                            bool ok0, bool ok1, long long dcol0, long long dcol1, float s_nat, float* pos,
                                            int row0, int row1) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const float xa = fmaf(__uint_as_float(r[4 * k + j]), sc, -u);
            const float xb = fmaf(__uint_as_float(r[4 * k + 2 + j]), sc, -u);
            float ea = ptx::ex2(xa), eb = ptx::ex2(xb);
            if (EDGE) {
                const int col = col0 + 8 * k + j;
                const bool cok = col < ncols;
                if (!(cok && ok0)) ea = 0.f;
                if (!(cok && ok1)) eb = 0.f;
                if (pos && cok && ok0 && col == dcol0) pos[row0] = __uint_as_float(r[4 * k + j]) * s_nat;
                if (pos && cok && ok1 && col == dcol1) pos[row1] = __uint_as_float(r[4 * k + 2 + j]) * s_nat;
            }
            l0 += ea; t0 = fmaf(ea, xa, t0);
            l1 += eb; t1 = fmaf(eb, xb, t1);
            const int cc = 2 * k + j;
            if (first) { cs[cc] = ea + eb; cd[cc] = fmaf(ea, xa, eb * xb); }
            else { cs[cc] += ea + eb; cd[cc] = fmaf(ea, xa, fmaf(eb, xb, cd[cc])); }
        }
    }
}

// Work distribution of the A-resident sweeps: the tiles of the block, in row-pair-major order (flat index = m_pair *
// n_tiles + column tile), are cut into n equal contiguous ranges, one per cluster; a range is walked as "units" =
// runs of column tiles inside one row pair (the resident rows of A are swapped at a row-pair boundary).
struct SweepGeom {
    int num_kb, n_tiles, m_pairs;
};
__host__ __device__ __forceinline__ long long sweep_begin(long long total, int cluster, int n) { return total * cluster / n; }
// cluster whose range contains flat tile f
__host__ __device__ __forceinline__ int sweep_cluster_of(long long total, long long f, int n) {
    return int(((f + 1) * n + total - 1) / total - 1);
}
struct SweepUnit { int m_pair, t0, t1; };
struct SweepWalk {
    long long f, f1;
    int n_tiles;
    __device__ __forceinline__ SweepWalk(const SweepGeom& g, int cluster, int n) {
        const long long total = (long long)g.m_pairs * g.n_tiles;
        f = sweep_begin(total, cluster, n);
        f1 = sweep_begin(total, cluster + 1, n);
        n_tiles = g.n_tiles;
    }
    __device__ __forceinline__ bool next(SweepUnit& u) {
        if (f >= f1) return false;
        u.m_pair = int(f / n_tiles);
        u.t0 = int(f - (long long)u.m_pair * n_tiles);
        u.t1 = int(min((long long)n_tiles, u.t0 + (f1 - f)));
        f += u.t1 - u.t0;
        return true;
    }
};

// TMA producer of a sweep (one lane of warp 0, both CTAs).  ARES: the rows of A are loaded once per unit and stay in
// shared memory; otherwise (K > 512) A streams with B, one K block per stage.
template <int STAGES, bool ARES = true>
__device__ __forceinline__ void sweep_produce(const Cta& c, Pipe& p, const CUtensorMap* tmA, const CUtensorMap* tmB,
                                              const SweepGeom& g, int cluster, int n_clusters) {
    SweepWalk w(g, cluster, n_clusters);
    SweepUnit u;
    uint32_t it_n = 0;
    for (; w.next(u); ++it_n) {
        const int m_blk = 2 * u.m_pair + int(c.cta_rank);
        if (ARES) {
            // the resident rows of A may be replaced once every MMA of the previous unit has completed
            if (it_n > 0) ptx::mbar_wait(c.bar_aempty, (it_n - 1) & 1);
            if (c.leader) ptx::mbar_arrive_expect_tx(c.bar_afull, 2 * g.num_kb * A_STAGE_BYTES);
            for (int kb = 0; kb < g.num_kb; ++kb)
                ptx::tma_load_2d_pair(c.sA + kb * A_STAGE_BYTES, tmA, kb * BK, m_blk * BM, c.bar_afull);
        }
        for (int t = u.t0; t < u.t1; ++t) {
            const int bn0 = t * BN + int(c.cta_rank) * (BN / 2);
            for (int kb = 0; kb < g.num_kb; ++kb) {
                ptx::mbar_wait(c.bar_empty + 8 * p.s, p.ph ^ 1);
                const uint32_t full = c.bar_full + 8 * p.s;
                if (c.leader) ptx::mbar_arrive_expect_tx(full, 2 * (ARES ? B_STAGE_BYTES : STAGE_BYTES));
                if (!ARES) ptx::tma_load_2d_pair(c.sA + p.s * A_STAGE_BYTES, tmA, kb * BK, m_blk * BM, full);
                ptx::tma_load_2d_pair(c.sB + p.s * B_STAGE_BYTES, tmB, kb * BK, bn0, full);
                if (++p.s == STAGES) { p.s = 0; p.ph ^= 1; }
            }
        }
    }
}

// MMA issuer of a sweep (one lane of warp 1, leader CTA)
template <int STAGES, int F16, bool ARES = true>
__device__ __forceinline__ void sweep_mma(const Cta& c, Pipe& p, const SweepGeom& g, int cluster, int n_clusters) {
    const uint32_t idesc = ptx::make_idesc_16bit(2 * BM, BN, 0, 0, !F16, !F16);
    const uint64_t desc_hi = ptx::make_smem_desc_sw128(16, 1024);
    SweepWalk w(g, cluster, n_clusters);
    SweepUnit u;
    uint32_t it_n = 0;
    for (; w.next(u); ++it_n) {
        if (ARES) {
            ptx::mbar_wait(c.bar_afull, it_n & 1);
            ptx::tc_fence_after();
        }
        for (int t = u.t0; t < u.t1; ++t, ++p.it) {
            const int a = p.it & 1;
            const uint32_t aph = (p.it >> 1) & 1;
            ptx::mbar_wait(c.bar_tempty + 8 * a, aph ^ 1);
            ptx::tc_fence_after();
            const uint32_t d_tmem = c.tmem_base + a * BN;
            for (int kb = 0; kb < g.num_kb; ++kb) {
                ptx::mbar_wait(c.bar_full + 8 * p.s, p.ph);
                ptx::tc_fence_after();
                const uint32_t a_src = c.sA + (ARES ? kb : p.s) * A_STAGE_BYTES;
                const uint32_t b_src = c.sB + p.s * B_STAGE_BYTES;
#pragma unroll
                for (int k = 0; k < BK / 16; ++k) {
                    ptx::mma_f16_ss_pair(d_tmem, ptx::desc_with_addr(desc_hi, a_src + k * 32),
                                         ptx::desc_with_addr(desc_hi, b_src + k * 32), idesc, (kb | k) != 0);
                }
                ptx::mma_commit_pair(c.bar_empty + 8 * p.s);
                if (++p.s == STAGES) { p.s = 0; p.ph ^= 1; }
            }
            ptx::mma_commit_pair(c.bar_tfull + 8 * a);
        }
        if (ARES) ptx::mma_commit_pair(c.bar_aempty);   // both CTAs' producers wait on their own copy
    }
}

template <int F16, bool ARES>
__global__ void __launch_bounds__(NUM_THREADS, 1)
fwd_sweep_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const FwdArgs args) {
    constexpr int STAGES = FWD_STAGES;
    float u = 0.f;
    const bool safe = fwd_bound(args, &u);
    // the launch of the swapped pass has nothing to do when the single sweep is taken: leave before any barrier, TMEM or
    // cluster state exists (uniform over the grid; the statistics it read were complete before the first launch began)
    if (safe && args.pass == 1) return;
    const Cta c = cta_setup<STAGES, COLBUF_BYTES, (ARES ? ARES_KB : STAGES) * A_STAGE_BYTES>();
    const uint32_t colbuf = c.sStg;
    const bool single = safe && args.pass == 0;
    const int cluster = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    Pipe p;
    const SweepGeom geom{args.num_kb, args.n_tiles, args.m_pairs};
    const long long total_tiles = (long long)args.m_pairs * args.n_tiles;
    {
        if (c.warp == 0) {
            if (c.lane == 0) {
                ptx::prefetch_tmap(&tmA);
                ptx::prefetch_tmap(&tmB);
                sweep_produce<STAGES, ARES>(c, p, &tmA, &tmB, geom, cluster, n_clusters);
            }
        } else if (c.warp == 1) {
            if (c.lane == 0 && c.leader) sweep_mma<STAGES, F16, ARES>(c, p, geom, cluster, n_clusters);
        } else if (!single) {
            // ---- exact mode: online-max row statistics, one row per thread (same code as the streaming STATS kernel)
            KArgs ka{};
            ka.M = args.M; ka.N = args.N; ka.scale = args.scale; ka.xs = args.xs; ka.ys = args.ys;
            ka.diag_offset = args.diag_offset; ka.part_max = args.part_max; ka.part_sum = args.part_sum;
            ka.part_dot = args.part_dot; ka.pos = args.pos;
            SweepWalk w(geom, cluster, n_clusters);
            SweepUnit un;
            while (w.next(un)) {
                const int m_blk = 2 * un.m_pair + int(c.cta_rank);
                const int part = cluster - sweep_cluster_of(total_tiles, (long long)un.m_pair * args.n_tiles, n_clusters);
                epilogue_unit<MODE_STATS>(c, p, &tmA, ka, m_blk, part, un.t0, un.t1);
            }
        } else {
            // ---- single sweep: row and column statistics of every tile
            const int warp = c.warp, lane = c.lane;
            const int q = warp & 3, half = (warp - 2) >> 2;
            const int g = lane >> 2, cq = 2 * (lane & 3);
            float dequant = 1.f;
            if (args.xs) dequant *= __ldg(args.xs);
            if (args.ys) dequant *= __ldg(args.ys);
            const float s_nat = __ldg(args.scale) * dequant;
            const float sc = s_nat * LOG2E;
            const int ncols = args.N, M = args.M;
            float* const pos = args.pos;
            // column of the chunk this lane owns after the butterfly, and its slot in the column buffer
            const int own_col = 8 * (g >> 1) + cq + (g & 1);
            SweepWalk w(geom, cluster, n_clusters);
            SweepUnit un;
            while (w.next(un)) {
                const int m_pair = un.m_pair, t0 = un.t0, t1 = un.t1;
                const int m_blk = 2 * m_pair + int(c.cta_rank);
                const int part = cluster - sweep_cluster_of(total_tiles, (long long)m_pair * args.n_tiles, n_clusters);
                const int rbase = m_blk * BM + q * 32;             // rows rbase + {g, 8 + g, 16 + g, 24 + g}
                float l[4] = {0.f, 0.f, 0.f, 0.f}, tt[4] = {0.f, 0.f, 0.f, 0.f};
                const bool row_edge = (m_blk + 1) * BM > M;
                const long long d_lo = args.diag_offset + (long long)m_blk * BM;
                for (int t = t0; t < t1; ++t, ++p.it) {
                    const int a = p.it & 1;
                    const uint32_t aph = (p.it >> 1) & 1;
                    const int n0 = t * BN;
                    const int colh = n0 + half * (BN / 2);
                    ptx::mbar_wait(c.bar_tfull + 8 * a, aph);
                    ptx::tc_fence_after();
                    const uint32_t taddr = c.tmem_base + a * BN + half * (BN / 2) + (uint32_t(q * 32) << 16);
                    const bool edge = row_edge || (n0 + BN > ncols) ||
                                      (pos && (d_lo + BM - 1 >= n0) && (d_lo < (long long)n0 + BN));
                    const uint32_t cbuf = colbuf + uint32_t(((((t & 1) * 2 + half) * 4 + q) * 128) * 8);
                    float cs[8], cd[8];
                    auto half_chunk = [&](const uint32_t (&r)[16], int hc) {
                        const int h = hc & 1, chunk = hc >> 1;
                        const int col0 = colh + chunk * 32 + cq;
                        const int r0 = rbase + 16 * h + g, r1 = r0 + 8;
                        if (edge)
                            rowcol_half<true>(r, sc, u, l[2 * h], tt[2 * h], l[2 * h + 1], tt[2 * h + 1], cs, cd, h == 0, col0,
                                              ncols, r0 < M, r1 < M, args.diag_offset + r0, args.diag_offset + r1, s_nat, pos,
                                              r0, r1);
                        else
                            rowcol_half<false>(r, sc, u, l[2 * h], tt[2 * h], l[2 * h + 1], tt[2 * h + 1], cs, cd, h == 0, col0,
                                               ncols, true, true, 0, 0, s_nat, nullptr, 0, 0);
                        if (h == 1) {
                            // butterfly over the 8 lanes that hold the same columns (lane bits 4, 3, 2): after the
                            // three steps this lane owns column `own_col` of the chunk
#pragma unroll
                            for (int step = 0; step < 3; ++step) {
                                const int n = 4 >> step;                  // values kept per quantity
                                const int mask = 16 >> step;
                                const bool up = (lane & mask) != 0;
#pragma unroll
                                for (int i = 0; i < n; ++i) {
                                    const float ks = up ? cs[i + n] : cs[i], ss = up ? cs[i] : cs[i + n];
                                    const float kd = up ? cd[i + n] : cd[i], sd = up ? cd[i] : cd[i + n];
                                    cs[i] = ks + __shfl_xor_sync(0xffffffffu, ss, mask);
                                    cd[i] = kd + __shfl_xor_sync(0xffffffffu, sd, mask);
                                }
                            }
                            asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(cbuf + uint32_t((chunk * 32 + own_col) * 8)),
                                         "f"(cs[0]), "f"(cd[0]) : "memory");
                        }
                    };
                    // TMEM loads are double buffered; half-chunk hc = 2 * chunk + h covers lanes 16h.. of the quarter
                    uint32_t ra[16], rb[16];
                    ptx::tmem_ld_16x256b_x4(taddr, ra);
                    ptx::tmem_ld_wait();
#pragma unroll
                    for (int hc = 0; hc < 8; hc += 2) {
                        ptx::tmem_ld_16x256b_x4(taddr + (hc >> 1) * 32 + (16u << 16), rb);
                        half_chunk(ra, hc);
                        ptx::tmem_ld_wait();
                        if (hc + 2 < 8) {
                            ptx::tmem_ld_16x256b_x4(taddr + ((hc + 2) >> 1) * 32, ra);
                        } else {
                            ptx::tc_fence_before();
                            __syncwarp();
                            if (lane == 0) ptx::mbar_arrive_leader(c.bar_tempty + 8 * a);
                        }
                        half_chunk(rb, hc + 1);
                        if (hc + 2 < 8) ptx::tmem_ld_wait();
                    }
                    // merge the four lane quarters of this half: thread (q, lane) sums column q * 32 + lane
                    ptx::named_bar_sync(1 + half, 128);
                    {
                        const int idx = q * 32 + lane;
                        const uint32_t src = colbuf + uint32_t((((t & 1) * 2 + half) * 4 * 128 + idx) * 8);
                        float S = 0.f, D = 0.f;
#pragma unroll
                        for (int qq = 0; qq < 4; ++qq) {
                            float x, y;
                            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(x), "=f"(y) : "r"(src + qq * 128 * 8));
                            S += x; D += y;
                        }
                        {
                            const size_t o = (size_t)m_blk * args.ldc + colh + idx;
                            args.colpart_sum[o] = S;
                            args.colpart_dot[o] = D;
                        }
                    }
                }
                // row statistics of the item: merge the 4 lanes that share the rows, lane (lane & 3) == 0 writes
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    l[i] += __shfl_xor_sync(0xffffffffu, l[i], 1);
                    tt[i] += __shfl_xor_sync(0xffffffffu, tt[i], 1);
                    l[i] += __shfl_xor_sync(0xffffffffu, l[i], 2);
                    tt[i] += __shfl_xor_sync(0xffffffffu, tt[i], 2);
                }
                if ((lane & 3) == 0) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int row = rbase + 8 * i + g;
                        if (row < M) {
                            const size_t slot = (size_t)(part * PARTS_PER_UNIT + half) * M + row;
                            args.part_max[slot] = u;
                            args.part_sum[slot] = l[i];
                            args.part_dot[slot] = fmaf(u, l[i], tt[i]);   // sum e * v with v = x + u
                        }
                    }
                }
            }
        }
    }
    cta_teardown(c);
}

// Recompute (GRAD) tiles of one panel as an A-resident persistent sweep: same mainloop as the forward sweep (rows of X
// resident, 4 B stages, one staging buffer per epilogue warp), G tiles leave through TMA stores.  One-plane operands
// and G only (bf16 / fp16 features with K <= 512); everything else takes the streaming gemm_kernel<MODE_GRAD>.
constexpr int GRAD_SWEEP_STAGES = 4;
constexpr int GRAD_SWEEP_STG = NUM_EPI_WARPS * STG_BYTES;   // 32 KB
__host__ __device__ constexpr int smem_bytes_grad_sweep() {
    return 1024 + ARES_KB * A_STAGE_BYTES + GRAD_SWEEP_STAGES * B_STAGE_BYTES + GRAD_SWEEP_STG + 256 + MISC_BYTES;
}

template <int F16>
__global__ void __launch_bounds__(NUM_THREADS, 1)
grad_sweep_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmC, const KArgs args, const SweepGeom geom) {
    constexpr int STAGES = GRAD_SWEEP_STAGES;
    const Cta c = cta_setup<STAGES, GRAD_SWEEP_STG, ARES_KB * A_STAGE_BYTES>();
    const int cluster = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    Pipe p;
    if (c.warp == 0) {
        if (c.lane == 0) {
            ptx::prefetch_tmap(&tmA);
            ptx::prefetch_tmap(&tmB);
            sweep_produce<STAGES>(c, p, &tmA, &tmB, geom, cluster, n_clusters);
        }
    } else if (c.warp == 1) {
        if (c.lane == 0 && c.leader) sweep_mma<STAGES, F16>(c, p, geom, cluster, n_clusters);
    } else {
        SweepWalk w(geom, cluster, n_clusters);
        SweepUnit un;
        while (w.next(un)) grad_epilogue_unit<false, 1>(c, p, &tmC, args, 2 * un.m_pair + int(c.cta_rank), un.t0, un.t1);
        epilogue_drain(c);
    }
    cta_teardown(c);
}

// The two gradient GEMMs of one panel in ONE launch, so that their tiles together fill the SMs:
// pairs [0, jobs0) run job 0 (dX = G * Yg), the rest run job 1 (dY = G^T * Xg).  A pair is one 256 x 256 output tile.
// Fused gradient GEMM + reduce-scatter (data-parallel ranks of one NVLink domain).  The rows of dY (the gradient on
// the GATHERED text features) belong to their home ranks: rank o owns global rows [o * rows_per_rank, +rows_per_rank).
// With peers.world > 0 every dY tile is written straight into the owner's memory through its peer-mapped address -
// over NVLink for remote owners - into the slot reserved for THIS source rank (plain TMA stores: reductions over
// NVLink were measured ~3x slower), and the CTA does not wait for the remote writes: they drain while the next
// panel is being recomputed.  The owner sums its `world` slots afterwards (finish_grad_kernel).  The separate
// reduce-scatter of loss.py's all_gather backward and its 4 * N * d byte input buffer disappear.
constexpr int MAX_PEERS = 8;
struct PeerOut {
    CUtensorMap map[MAX_PEERS];   // fp32 [rows_per_rank, d] slot of this source rank in the memory of every owner
    int world;                    // 0 = job 1 writes through tmC1 (single GPU, or the NCCL reduce-scatter path)
    int rows_per_rank;            // multiple of 128: a CTA's 128 output rows never straddle two owners
};

template <int F16>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmB0,
                 const __grid_constant__ CUtensorMap tmC0, const KArgs args0,
                 const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmB1,
                 const __grid_constant__ CUtensorMap tmC1, const KArgs args1, const int jobs0, const int jobs1,
                 const int dy_first, const __grid_constant__ PeerOut peers) {
    constexpr int STAGES = stages_of(MODE_OUT);
    const Cta c = cta_setup<STAGES, STG_TOTAL>();
    // cluster (2, 1, 1): one job per CTA pair = a 256 x 256 output tile.  The hardware dispatches the pairs in index
    // order, so the kind with the LONGER jobs goes first (longest-first keeps the tail short); when those are the dY
    // jobs their stores - the ones that cross NVLink in the fused reduce-scatter - also drain under the dX jobs
    const int jj = blockIdx.x >> 1;
    const bool first = dy_first ? (jj >= jobs1) : (jj < jobs0);
    const int j = dy_first ? (first ? jj - jobs1 : jj + jobs0) : jj;     // index in the [dX jobs | dY jobs] numbering
    const KArgs& args = first ? args0 : args1;
    const CUtensorMap* tmA = first ? &tmA0 : &tmA1;
    const CUtensorMap* tmB = first ? &tmB0 : &tmB1;
    const CUtensorMap* tmC = first ? &tmC0 : &tmC1;
    const int k = first ? j : j - jobs0;
    const int m_blk = 2 * (k / args.n_tiles) + int(c.cta_rank);
    const int t0 = k % args.n_tiles;
    int row_shift = 0;
    if (!first && peers.world > 0) {
        const int grow = args.c_row_off + m_blk * BM;           // first global dY row of this CTA
        const int owner = min(grow / peers.rows_per_rank, peers.world - 1);
        tmC = &peers.map[owner];
        row_shift = -owner * peers.rows_per_rank;   // args.accumulate stays: first row panel stores, later ones add
    }
    Pipe p;
    if (c.warp == 0) {
        if (c.lane == 0) {
            ptx::prefetch_tmap(tmA);
            ptx::prefetch_tmap(tmB);
            produce_unit<STAGES>(c, p, tmA, tmB, args, m_blk, t0, t0 + 1);
        }
    } else if (c.warp == 1) {
        if (c.lane == 0 && c.leader) mma_unit<STAGES>(c, p, args, 1);
    } else {
        epilogue_unit<MODE_OUT>(c, p, tmC, args, m_blk, t0, t0, t0 + 1, row_shift);
        epilogue_drain(c);
    }
    cta_teardown(c);
}

// ---------------------------------------------------------------------------------------------------- SigLIP
// Pairwise sigmoid loss (open_clip's SigLipLoss) over the tiles of S = X Y^T:
//   l_ij = s x_i.y_j + t,  z_ij = +1 at the positive (column diag_offset + i), -1 elsewhere,
//   loss = (1/b) sum_ij softplus(-z_ij l_ij),   g_ij = sigma(l_ij) - [j is the positive].
// Every element is independent: no row or column log-sum-exp, no shared reference, no column statistics.  Both kernels
// are the A-resident persistent sweep of the ClipLoss forward (sweep_produce / sweep_mma / SweepWalk) with an epilogue
// of their own, one thread per row and 128-column half (the tcgen05.ld 32x32b layout).  Per (part, half, row) they
// write plain partial sums that small kernels merge in a fixed order: the results are bit-reproducible, no atomics.
struct SigArgs {
    int M, N;                  // rows (b) and columns of this call's block
    const float* scale;        // device scalar s (already exponentiated)
    const float* bias;         // device scalar t; null = 0
    long long diag_offset;     // the positive of row i is column diag_offset + i
    float* part_a;             // [parts][M]  forward: sum softplus(-z l) / ln 2      recompute: sum g
    float* part_b;             // [parts][M]  forward: max negative l * log2(e)       recompute: sum g * x.y
    float* pos;                // [M] forward: positive logit (natural units)
    const float* p2e;          // recompute: device scalar 2^e, the power of two the fp16 G panel carries
};
constexpr int SIG_GRAD_STAGES_STREAM = 6;        // B (and A) stages of the recompute when K > 512: same smem as ARES
__host__ __device__ constexpr int smem_bytes_sig_fwd(bool ares) {
    return 1024 + (ares ? ARES_KB : FWD_STAGES) * A_STAGE_BYTES + FWD_STAGES * B_STAGE_BYTES + 256 + MISC_BYTES;
}
__host__ __device__ constexpr int sig_grad_stages(bool ares) { return ares ? GRAD_SWEEP_STAGES : SIG_GRAD_STAGES_STREAM; }
__host__ __device__ constexpr int smem_bytes_sig_grad(bool ares) {
    return 1024 + (ares ? ARES_KB : SIG_GRAD_STAGES_STREAM) * A_STAGE_BYTES + sig_grad_stages(ares) * B_STAGE_BYTES +
           GRAD_SWEEP_STG + 256 + MISC_BYTES;
}

// log2(1 + e) for e in [0, 1], on the FMA pipe: e * P(e) with P a degree-8 fit of log2(1 + e) / e at Chebyshev nodes.
// Relative error <= 2e-7 in fp32 over every normal e, so small terms keep their value: lg2(1 + e) would round 1 + e
// to 1 and drop every term below 2^-24, and a well-separated batch's loss is a sum of N such terms per row.
__device__ __forceinline__ float sig_log2_1p(float e) {
    float p = 7.395402063e-03f;
    p = fmaf(p, e, -4.194501042e-02f);
    p = fmaf(p, e, 1.118320748e-01f);
    p = fmaf(p, e, -1.962389499e-01f);
    p = fmaf(p, e, 2.752211988e-01f);
    p = fmaf(p, e, -3.582990766e-01f);
    p = fmaf(p, e, 4.806788862e-01f);
    p = fmaf(p, e, -7.213395238e-01f);
    p = fmaf(p, e, 1.442695022e+00f);
    return p * e;
}
__device__ __forceinline__ float sig_rcp(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// 32 columns of one row of the forward, log2 units: with u = -z l log2(e),
//   softplus(-z l) / ln 2 = max(u, 0) + log2(1 + 2^-|u|)
// ONE MUFU op per element (the ex2; 2^-|u| never overflows, and terms down to 2^-126 stay normal), the log on the FMA
// pipe.  EDGE: the chunk may hold the row's positive, or columns >= N (read as zeros by TMA, masked here).
template <bool EDGE>
__device__ __forceinline__ void sig_fwd_chunk(const uint32_t (&r)[32], float sc2, float t2, int col0, int ncols,
                                              long long dcol, float (&acc)[4], float& mneg, float& pos_raw, bool& have_pos) {
    const int didx = (EDGE && dcol >= col0 && dcol < (long long)col0 + 32) ? int(dcol - col0) : -1;
#pragma unroll
    for (int k = 0; k < 32; ++k) {
        const float v = fmaf(__uint_as_float(r[k]), sc2, t2);      // l * log2(e)
        const bool is_pos = EDGE && k == didx;
        const bool inside = !EDGE || col0 + k < ncols;
        const float u = is_pos ? -v : v;
        float sp = fmaxf(u, 0.f) + sig_log2_1p(ptx::ex2(-fabsf(u)));
        if (EDGE) {
            if (!inside) sp = 0.f;
            if (is_pos) { pos_raw = __uint_as_float(r[k]); have_pos = true; }
        }
        acc[k & 3] += sp;
        if (!is_pos && inside) mneg = fmaxf(mneg, v);
    }
}

// One unit (a run of column tiles of one 128-row block) of the forward epilogue; writes the row's partial sums of the unit
// into slot (part, half).  Same accumulator hand-off as epilogue_unit.
__device__ __forceinline__ void sig_fwd_epilogue_unit(const Cta& c, Pipe& p, const SigArgs& args, int m_blk, int part, int t0,
                                                      int t1) {
    const int warp = c.warp, lane = c.lane;
    const int q = warp & 3, half = (warp - 2) >> 2;
    const int row = m_blk * BM + q * 32 + lane;
    const long long dcol = args.diag_offset + row;
    const float s = __ldg(args.scale), t = args.bias ? __ldg(args.bias) : 0.f;
    const float sc2 = s * LOG2E, t2 = t * LOG2E;
    const int ncols = args.N;
    const long long d_lo = args.diag_offset + (long long)m_blk * BM;
    float acc[4] = {0.f, 0.f, 0.f, 0.f}, mneg = -CUDART_INF_F, pos_raw = 0.f;
    bool have_pos = false;
    for (int tt = t0; tt < t1; ++tt, ++p.it) {
        const int a = p.it & 1;
        const uint32_t aph = (p.it >> 1) & 1;
        const int n0 = tt * BN;
        const int colh = n0 + half * (BN / 2);
        // edge tile: contains positives of this CTA's rows, or columns beyond N
        const bool edge = ((d_lo + BM - 1 >= n0) && (d_lo < (long long)n0 + BN)) || (n0 + BN > ncols);
        ptx::mbar_wait(c.bar_tfull + 8 * a, aph);
        ptx::tc_fence_after();
        const uint32_t taddr = c.tmem_base + a * BN + half * (BN / 2) + (uint32_t(q * 32) << 16);
        auto process = [&](const uint32_t (&r)[32], int cidx) {
            const int col0 = colh + cidx * 32;
            if (edge) sig_fwd_chunk<true>(r, sc2, t2, col0, ncols, dcol, acc, mneg, pos_raw, have_pos);
            else sig_fwd_chunk<false>(r, sc2, t2, col0, ncols, dcol, acc, mneg, pos_raw, have_pos);
        };
        uint32_t ra[32], rb[32];
        ptx::tmem_ld_32x32(taddr, ra);
        ptx::tmem_ld_wait();
        ptx::tmem_ld_32x32(taddr + 32, rb);
        process(ra, 0);
        ptx::tmem_ld_wait();
        ptx::tmem_ld_32x32(taddr + 64, ra);
        process(rb, 1);
        ptx::tmem_ld_wait();
        ptx::tmem_ld_32x32(taddr + 96, rb);
        process(ra, 2);
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_leader(c.bar_tempty + 8 * a);
        process(rb, 3);
    }
    if (row < args.M) {
        const size_t slot = (size_t)(part * PARTS_PER_UNIT + half) * args.M + row;
        args.part_a[slot] = (acc[0] + acc[1]) + (acc[2] + acc[3]);
        args.part_b[slot] = mneg;
        if (have_pos) args.pos[row] = fmaf(pos_raw, s, t);
    }
}

template <bool ARES>
__global__ void __launch_bounds__(NUM_THREADS, 1)
siglip_fwd_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const SigArgs args,
                  const SweepGeom geom) {
    constexpr int STAGES = FWD_STAGES;
    const Cta c = cta_setup<STAGES, 0, (ARES ? ARES_KB : STAGES) * A_STAGE_BYTES>();
    const int cluster = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    Pipe p;
    if (c.warp == 0) {
        if (c.lane == 0) {
            ptx::prefetch_tmap(&tmA);
            ptx::prefetch_tmap(&tmB);
            sweep_produce<STAGES, ARES>(c, p, &tmA, &tmB, geom, cluster, n_clusters);
        }
    } else if (c.warp == 1) {
        if (c.lane == 0 && c.leader) sweep_mma<STAGES, 0, ARES>(c, p, geom, cluster, n_clusters);
    } else {
        const long long total = (long long)geom.m_pairs * geom.n_tiles;
        SweepWalk w(geom, cluster, n_clusters);
        SweepUnit un;
        while (w.next(un)) {
            const int part = cluster - sweep_cluster_of(total, (long long)un.m_pair * geom.n_tiles, n_clusters);
            sig_fwd_epilogue_unit(c, p, args, 2 * un.m_pair + int(c.cta_rank), part, un.t0, un.t1);
        }
    }
    cta_teardown(c);
}

// 16 columns of one row of the recompute: g = sigma(l) - [positive], times 2^e, into g[16] (fp32, still to be packed).
// With e = exp(-|l|) (ex2) and r = 1 / (1 + e) (rcp) - TWO MUFU ops per element:
//   sigma(l) = r for l >= 0, e * r for l < 0     (never overflows: e <= 1; no 1 - x cancellation)
//   at the positive g = -sigma(-l), not sigma(l) - 1: a well-classified positive (l = 20) keeps g = -2e-9 instead of
//   the 0 or 2^-24 multiples sigma(l) - 1 gives in fp32.
// The row sums of g and g * x.y (dlogit_bias, dlogit_scale) are taken from the unscaled fp32 values.
template <bool EDGE>
__device__ __forceinline__ void sig_grad16(const uint32_t (&r)[16], float sc2, float t2, float p2e, int col0, int ncols,
                                           long long dcol, bool row_ok, float& sg, float& sgx, float (&g)[16]) {
    const int didx = (EDGE && dcol >= col0 && dcol < (long long)col0 + 16) ? int(dcol - col0) : -1;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const float xy = __uint_as_float(r[k]);
        const float v = fmaf(xy, sc2, t2);                 // l * log2(e)
        const float e = ptx::ex2(-fabsf(v));
        const float big = sig_rcp(1.f + e), small = e * big;
        float gk = v >= 0.f ? big : small;                 // NaN logits take `small` = NaN
        if (EDGE) {
            if (k == didx) gk = -(v >= 0.f ? small : big);
            if (!row_ok || col0 + k >= ncols) gk = 0.f;
        }
        sg += gk;
        sgx = fmaf(gk, xy, sgx);
        g[k] = gk * p2e;
    }
}

// One unit of the recompute epilogue: the G tile leaves through the same half-size SWIZZLE_64B staging and TMA stores as
// grad_epilogue_unit<false, 1>; the row sums of the unit go to slot (part, half).
__device__ __forceinline__ void sig_grad_epilogue_unit(const Cta& c, Pipe& p, const CUtensorMap* tmC, const SigArgs& args,
                                                       int m_blk, int part, int t0, int t1) {
    const int warp = c.warp, lane = c.lane;
    const int q = warp & 3, half = (warp - 2) >> 2;
    const int row = m_blk * BM + q * 32 + lane;
    const bool row_ok = row < args.M;
    const long long dcol = args.diag_offset + row;
    const float sc2 = __ldg(args.scale) * LOG2E, t2 = (args.bias ? __ldg(args.bias) : 0.f) * LOG2E;
    const float p2e = __ldg(args.p2e);
    const int ncols = args.N;
    const int c_row_off = m_blk * BM + q * 32;
    const long long d_lo = args.diag_offset + (long long)m_blk * BM;
    const bool row_edge = (m_blk + 1) * BM > args.M;
    const uint32_t stg0 = c.sStg + (warp - 2) * STG_BYTES;
    float sg = 0.f, sgx = 0.f;
    for (int tt = t0; tt < t1; ++tt, ++p.it) {
        const int a = p.it & 1;
        const uint32_t aph = (p.it >> 1) & 1;
        const int n0 = tt * BN;
        const int colh = n0 + half * (BN / 2);
        // edge tile: positives of this CTA's rows, columns beyond N or rows beyond M (all masked to g = 0)
        const bool edge = row_edge || ((d_lo + BM - 1 >= n0) && (d_lo < (long long)n0 + BN)) || (n0 + BN > ncols);
        ptx::mbar_wait(c.bar_tfull + 8 * a, aph);
        ptx::tc_fence_after();
        const uint32_t taddr = c.tmem_base + a * BN + half * (BN / 2) + (uint32_t(q * 32) << 16);
        uint32_t stg = 0;
        auto piece = [&](const uint32_t (&r)[16], int pi) {
            const int col0 = colh + pi * 16;
            if ((pi & 1) == 0) {
                // half buffers of 32 columns, two pieces each: at most one older bulk store may still read this warp's
                // other half
                if (lane == 0) ptx::tma_store_wait_read<1>();
                __syncwarp();
                stg = stg0 + (p.stg_use & 1) * (STG_BYTES / 2);
            }
            float g[16];
            if (edge) sig_grad16<true>(r, sc2, t2, p2e, col0, ncols, dcol, row_ok, sg, sgx, g);
            else sig_grad16<false>(r, sc2, t2, p2e, col0, ncols, dcol, row_ok, sg, sgx, g);
            grad16_store<false, true>(g, stg, 0, lane, (pi & 1) * 2);
            if (pi & 1) {
                ptx::fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    ptx::tma_store_2d(tmC, stg, col0 - 16, c_row_off);
                    ptx::tma_store_commit();
                }
                ++p.stg_use;
            }
        };
        uint32_t ra[16], rb[16];
        ptx::tmem_ld_32x16(taddr, ra);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int pi = 0; pi < 8; pi += 2) {
            ptx::tmem_ld_32x16(taddr + (pi + 1) * 16, rb);
            piece(ra, pi);
            ptx::tmem_ld_wait();
            if (pi + 2 < 8) {
                ptx::tmem_ld_32x16(taddr + (pi + 2) * 16, ra);
            } else {
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive_leader(c.bar_tempty + 8 * a);
            }
            piece(rb, pi + 1);
            if (pi + 2 < 8) ptx::tmem_ld_wait();
        }
    }
    if (row_ok) {
        const size_t slot = (size_t)(part * PARTS_PER_UNIT + half) * args.M + row;
        args.part_a[slot] = sg;
        args.part_b[slot] = sgx;
    }
}

// Recompute of one G panel: rows of X resident (ARES, K <= 512) or streamed with Y (K > 512), G tiles out through TMA.
template <bool ARES>
__global__ void __launch_bounds__(NUM_THREADS, 1)
siglip_grad_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ CUtensorMap tmC, const SigArgs args, const SweepGeom geom) {
    constexpr int STAGES = sig_grad_stages(ARES);
    const Cta c = cta_setup<STAGES, GRAD_SWEEP_STG, (ARES ? ARES_KB : STAGES) * A_STAGE_BYTES>();
    const int cluster = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    Pipe p;
    if (c.warp == 0) {
        if (c.lane == 0) {
            ptx::prefetch_tmap(&tmA);
            ptx::prefetch_tmap(&tmB);
            sweep_produce<STAGES, ARES>(c, p, &tmA, &tmB, geom, cluster, n_clusters);
        }
    } else if (c.warp == 1) {
        if (c.lane == 0 && c.leader) sweep_mma<STAGES, 0, ARES>(c, p, geom, cluster, n_clusters);
    } else {
        const long long total = (long long)geom.m_pairs * geom.n_tiles;
        SweepWalk w(geom, cluster, n_clusters);
        SweepUnit un;
        while (w.next(un)) {
            const int part = cluster - sweep_cluster_of(total, (long long)un.m_pair * geom.n_tiles, n_clusters);
            sig_grad_epilogue_unit(c, p, &tmC, args, 2 * un.m_pair + int(c.cta_rank), part, un.t0, un.t1);
        }
        epilogue_drain(c);
    }
    cta_teardown(c);
}

}  // namespace clipk
