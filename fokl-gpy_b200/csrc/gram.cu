// gram.cu -- K2: Gram / projection update on the FP64 tensor pipe (sm_100a, mma.sync DMMA).
//
// Replaces XtX = X'X and Xty = X'y of the reference (src/FoKL/FoKLRoutines.py:1492-1494), which
// recomputes the full P x P product on every `gibbs` call.  Here only the block that is new when C
// columns are appended is formed:   block = [X_old  X_new  y]' X_new     ((P_old + C + 1) x C)
// and of its symmetric X_new' X_new part only the 8 x 8 fragments on or above the diagonal.
//
// Work decomposition (gram_plan.h): the needed fragments are grouped into 2 x 2-fragment blocks and the blocks into
// tiles of <= 4 blocks per warp; a CTA (16 warps, 4 blocks = 16 DMMA accumulators per warp) owns one tile for one
// contiguous range of rows.  X is column-major, so both MMA operands are contiguous along the reduction (row) index: the CTA
// streams KB-row slabs of the tile's distinct operand columns ("slots", each staged ONCE however many blocks use it)
// into shared memory with cp.async (3/4-stage ring, [slot][KB + 4] layout = conflict-free fragment loads) and issues
// mma.sync.m8n8k4.f64 from there.  Grid = tiles x row splits ~ one CTA per resident slot; the per-split accumulators go to a
// workspace in fragment order (coalesced 16-byte stores) and gram_reduce_kernel sums them in a fixed order
// (deterministic, no atomics) while scattering to the (P_old + C + 1) x C block.
#include "fokl_ctx.cuh"
#include "gram_plan.h"
#include <cuda.h>            // CUtensorMap types only: the encoder is fetched through cudaGetDriverEntryPoint
#include <algorithm>
#include <stdlib.h>
#include <string.h>

namespace {

using fokl::GramBlockMeta;
using fokl::GramTileMeta;
using fokl::kGramBlocksPerWarp;

constexpr int kMaxStages = 4;            // cp.async ring depth: 4, or 3 when that buys a deeper slab
constexpr int kMaxStagesTma = 8;         // TMA ring depth
constexpr int kPad = 4;                     // row stride KB + 4 doubles: fragment loads hit 16 distinct 8-byte banks

struct GramParams {
    const double *X;
    const double *y;
    int64_t ld, n;
    int p;                                  // p_old + c: slot source p means y
    int kb;                                 // rows per pipeline stage: 16 ... 256
    int kb_shift;                           // log2(kb / 2)
    int stages;                             // ring depth (3 or 4)
    int max_slots;                          // shared-memory stage = max_slots * (kb + 4) doubles
    int64_t rows_per_split;
    const GramTileMeta *tiles;
    const int32_t *slot_src;
    const GramBlockMeta *blocks;
    double *part;                           // [split][tile][64 blocks][4 fragments][64]
    int n_tiles;
    int tile_blocks;                        // workspace stride: warps * 4 blocks per tile
};

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem, int src_bytes)
{
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void dmma_m8n8k4(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// D += A * B on one 8 x 8 x 4 fragment, executed only where `on` is non-zero.  The predicate lives inside the asm so
// the compiler neither branches around the warp-synchronous instruction nor re-converges after it; `on` is
// warp-uniform (it comes from the block's fragment mask).
template <unsigned BIT>
__device__ __forceinline__ void dmma_m8n8k4_if(double &c0, double &c1, double a, double b, unsigned on)
{
#ifdef FOKL_GRAM_MASK_BRANCH
    if (on & BIT) dmma_m8n8k4(c0, c1, a, b);
    return;
#endif
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .b32 t;\n"
        "and.b32 t, %4, %5;\n"
        "setp.ne.u32 p, t, 0;\n"
        "@p mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
        "}\n"
        : "+d"(c0), "+d"(c1)
        : "d"(a), "d"(b), "r"(on), "n"(BIT));
}

// ---- mbarrier + bulk-copy primitives (sm_90+ PTX) ---------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Spin until the phase with the given parity has completed.  A wait that never ends (a protocol bug) traps instead of
// hanging the device.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
    const unsigned addr = smem_u32(bar);
    unsigned done = 0;
    for (unsigned spin = 0; !done; ++spin) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (spin > (1u << 26)) __trap();
    }
}
// One lane of the (converged) warp, the same for the whole warp: lets the compiler issue a warp-uniform instruction once.
__device__ __forceinline__ bool elect_one()
{
    unsigned pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
// A run of staged columns that are consecutive both in the tile's slot list and in X: what the producer walks.
struct GramRun {
    const double *src;      // column of the first slot
    int32_t slot0, len;
};
// global -> shared bulk copy (TMA engine, no tensor map), completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_g2s(void *smem, const void *gmem, unsigned bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(smem)),
                 "l"(gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// Consumer side of the mbarrier ring for a warp that owns NB work items (positions q = warp + 16 b): wait for a slab,
// issue its DMMAs, hand the stage back.  No CTA-wide barrier: warps drift up to stages - 1 slabs apart.
// FLEX: 0 = every block of the warp is a full regular 2 x 2 block (four operand loads per four DMMAs); 1 = the warp's first
// block is a loose / masked one (one operand pair per fragment, predicated DMMAs), the others are full regular blocks;
// 2 = every block takes the loose form.  The plan (gram_plan.h) puts at most one loose block on a warp whenever the
// tile has no more of them than busy warps, so the extra loads are spread evenly.
template <int WARPS, int NB, int FLEX>
__device__ __forceinline__ void gram_consume(const GramParams &P, const GramTileMeta &tm, const double *stages, size_t stage_doubles,
                                             int stride, uint64_t *full, uint64_t *empty, int nk, int lane, int warp, double *out)
{
    constexpr int kGramWarps = WARPS;
    constexpr int NF = FLEX == 2 ? NB : (FLEX == 1 ? 1 : 0);        // blocks 0 .. NF - 1: loose form
    constexpr int NFA = NF > 0 ? NF : 1, NR = NB - NF, NRA = NR > 0 ? NR : 1;
    int a_off[NRA], b_off[NRA];
    int la_off[NFA][4], lb_off[NFA][4];
    unsigned msk[NFA];
    const int frag_r = lane >> 2, frag_k = lane & 3;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const GramBlockMeta bm = P.blocks[tm.blk_off + warp + kGramWarps * b];
        if (b < NF) {
            msk[b] = bm.mask;
#pragma unroll
            for (int f = 0; f < 4; ++f) {
                la_off[b][f] = (bm.la[f] + frag_r) * stride + frag_k + 16 * bm.phase;     // this item's first 16-row chunk
                lb_off[b][f] = (bm.lb[f] + frag_r) * stride + frag_k + 16 * bm.phase;
            }
        } else {
            a_off[b - NF] = (bm.a_slot + frag_r) * stride + frag_k + 16 * bm.phase;
            b_off[b - NF] = (bm.b_slot + frag_r) * stride + frag_k + 16 * bm.phase;
        }
    }
    double acc[NB][4][2];
#pragma unroll
    for (int b = 0; b < NB; ++b)
#pragma unroll
        for (int f = 0; f < 4; ++f) acc[b][f][0] = acc[b][f][1] = 0.0;

    const int stages_n = P.stages;
    const int kstep = 16 * tm.ksplit;
    const int half = 8 * stride;                                   // second fragment row / column of a block
    int st = 0;
    unsigned ph = 0;
    for (int kt = 0; kt < nk; ++kt) {
        mbar_wait(full + st, ph);
        const double *S = stages + (size_t)st * stage_doubles;
        for (int k0 = 0; k0 < P.kb; k0 += kstep) {
#pragma unroll
            for (int kk = 0; kk < 16; kk += 4) {
                double a0[NRA], a1[NRA], b0[NRA], b1[NRA];
#pragma unroll
                for (int b = 0; b < NR; ++b) {
                    const double *pa = S + a_off[b] + k0 + kk, *pb = S + b_off[b] + k0 + kk;
                    a0[b] = pa[0]; a1[b] = pa[half]; b0[b] = pb[0]; b1[b] = pb[half];
                }
#pragma unroll
                for (int b = 0; b < NF; ++b) {
                    double av[4], bv[4];
#pragma unroll
                    for (int f = 0; f < 4; ++f) { av[f] = S[la_off[b][f] + k0 + kk]; bv[f] = S[lb_off[b][f] + k0 + kk]; }
                    dmma_m8n8k4_if<1u>(acc[b][0][0], acc[b][0][1], av[0], bv[0], msk[b]);
                    dmma_m8n8k4_if<2u>(acc[b][1][0], acc[b][1][1], av[1], bv[1], msk[b]);
                    dmma_m8n8k4_if<4u>(acc[b][2][0], acc[b][2][1], av[2], bv[2], msk[b]);
                    dmma_m8n8k4_if<8u>(acc[b][3][0], acc[b][3][1], av[3], bv[3], msk[b]);
                }
#pragma unroll
                for (int b = 0; b < NR; ++b) {
                    dmma_m8n8k4(acc[NF + b][0][0], acc[NF + b][0][1], a0[b], b0[b]);
                    dmma_m8n8k4(acc[NF + b][1][0], acc[NF + b][1][1], a0[b], b1[b]);
                    dmma_m8n8k4(acc[NF + b][2][0], acc[NF + b][2][1], a1[b], b0[b]);
                    dmma_m8n8k4(acc[NF + b][3][0], acc[NF + b][3][1], a1[b], b1[b]);
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + st);                    // this warp is done reading the stage
        if (++st == stages_n) { st = 0; ph ^= 1u; }
    }
    // accumulators in fragment order: lane l holds C[l >> 2][(l & 3) * 2 + {0, 1}] = row-major 8 x 8 at offset 2 l
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const int q = warp + kGramWarps * b;
#pragma unroll
        for (int f = 0; f < 4; ++f)
            *reinterpret_cast<double2 *>(out + (size_t)q * 256 + f * 64 + lane * 2) = make_double2(acc[b][f][0], acc[b][f][1]);
    }
}

// Producer warp of the mbarrier ring: one bulk copy per staged column and slab (KB rows = KB * 8 contiguous bytes),
// all completing on the stage's `full` barrier; a stage is refilled as soon as every consumer warp has released it.
// The whole warp walks the runs with warp-uniform operands and one elected lane issues each copy (per-lane operands
// would make the compiler serialise the warp lane by lane, ~55 cycles per copy: profiles/r01_gram_ksplit.txt).
__device__ __forceinline__ void gram_produce(const GramParams &P, double *stages, size_t stage_doubles, int stride,
                                             const GramRun *runs, int n_runs, int n_real, uint64_t *full, uint64_t *empty,
                                             int64_t n_lo, int64_t n_hi, int nk, int64_t ld, int lane)
{
    const unsigned slab_bytes = (unsigned)P.kb * 8u;
    const int stages_n = P.stages;
    int st = 0;
    unsigned ph = 0;
    for (int kt = 0; kt < nk; ++kt) {
        if (kt >= stages_n) mbar_wait(empty + st, ph ^ 1u);        // the previous use of this stage has been consumed
        double *dst = stages + (size_t)st * stage_doubles;
        const int64_t r0 = n_lo + (int64_t)kt * P.kb;
        const int64_t left = n_hi - r0;
        if (left >= P.kb) {
            if (elect_one()) mbar_arrive_expect_tx(full + st, (unsigned)n_real * slab_bytes);
            __syncwarp();
            for (int r = 0; r < n_runs; ++r) {
                const GramRun run = runs[r];
                const double *src = run.src + r0;
                double *d = dst + (size_t)run.slot0 * stride;
                for (int i = 0; i < run.len; ++i) {
                    if (elect_one()) bulk_g2s(d, src, slab_bytes, full + st);
                    src += ld;
                    d += stride;
                }
            }
        } else {
            // last, partial slab of the matrix: plain copies with zero fill (rows >= n never enter a product)
            for (int r = 0; r < n_runs; ++r) {
                const GramRun run = runs[r];
                for (int i = 0; i < run.len; ++i)
                    for (int k = lane; k < P.kb; k += 32)
                        dst[(size_t)(run.slot0 + i) * stride + k] = k < left ? run.src[(int64_t)i * ld + r0 + k] : 0.0;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(full + st);
        }
        if (++st == stages_n) { st = 0; ph ^= 1u; }
    }
}

// ---- 2-D tensor-map TMA ring (gram_kernel_tma) -------------------------------------------------------------------------
// Stage layout: [16-row chunk][slot][16 doubles], every 128-byte row written by the copy engine with the 128-byte
// swizzle (16-byte unit j of slot row s lands at unit j ^ (s & 7)).  A DMMA fragment load touches 8 slot rows x 4
// reduction indices; the reduction index is free to permute, so k-step t of a chunk uses the rows {2t, 2t+1, 2t+8, 2t+9}
// of the chunk: the two 16-byte units t and t + 4 of each slot row, which the swizzle spreads over all 32 banks for the
// 4 slot rows of a half warp (conflict-free, no padding).
__device__ __forceinline__ void tma_load_2d(void *smem, const CUtensorMap *map, int c0, int c1, uint64_t *bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::"r"(
                     smem_u32(smem)),
                 "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}

struct GramTmaMaps {
    CUtensorMap m[fokl::kGramBoxKinds];
};

template <int WARPS, int NB, int FLEX>
__device__ __forceinline__ void gram_consume_tma(const GramParams &P, const GramTileMeta &tm, const double *stages, size_t stage_doubles,
                                                 uint64_t *full, uint64_t *empty, int nk, int lane, int warp, double *out)
{
    constexpr int kGramWarps = WARPS;
    constexpr int NF = FLEX == 2 ? NB : (FLEX == 1 ? 1 : 0);        // blocks 0 .. NF - 1: loose form (see gram_consume)
    constexpr int NFA = NF > 0 ? NF : 1, NR = NB - NF, NRA = NR > 0 ? NR : 1;
    const int frag_r = lane >> 2, frag_k = lane & 3;
    // lane constants of the swizzled address: unit = (t + 4 h) ^ r with h = frag_k >> 1; element within the unit = frag_k & 1
    const int lane_off = 8 * ((frag_k >> 1) ^ (frag_r >> 2)) + (frag_k & 1);
    const int r3 = frag_r & 3;
    int a_off[NRA], b_off[NRA], ph0[NB];
    int la_off[NFA][4], lb_off[NFA][4];
    unsigned msk[NFA];
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const GramBlockMeta bm = P.blocks[tm.blk_off + warp + kGramWarps * b];
        ph0[b] = bm.phase;
        if (b < NF) {
            msk[b] = bm.mask;
#pragma unroll
            for (int f = 0; f < 4; ++f) {
                la_off[b][f] = (bm.la[f] + frag_r) * 16 + lane_off;
                lb_off[b][f] = (bm.lb[f] + frag_r) * 16 + lane_off;
            }
        } else {
            a_off[b - NF] = (bm.a_slot + frag_r) * 16 + lane_off;
            b_off[b - NF] = (bm.b_slot + frag_r) * 16 + lane_off;
        }
    }
    double acc[NB][4][2];
#pragma unroll
    for (int b = 0; b < NB; ++b)
#pragma unroll
        for (int f = 0; f < 4; ++f) acc[b][f][0] = acc[b][f][1] = 0.0;

    const int stages_n = P.stages;
    const int chunks = P.kb >> 4, ksplit = tm.ksplit;
    const int chunk_doubles = P.max_slots * 16;
    constexpr int half = 8 * 16;                                   // second fragment row / column of a block: 8 slot rows on
    int st = 0;
    unsigned ph = 0;
    for (int kt = 0; kt < nk; ++kt) {
        mbar_wait(full + st, ph);
        const double *S = stages + (size_t)st * stage_doubles;
        for (int c0 = 0; c0 < chunks; c0 += ksplit) {
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int toff = 2 * (t ^ r3);
                double a0[NRA], a1[NRA], b0[NRA], b1[NRA];
#pragma unroll
                for (int b = 0; b < NR; ++b) {
                    const double *base = S + (c0 + ph0[NF + b]) * chunk_doubles + toff;
                    const double *pa = base + a_off[b], *pb = base + b_off[b];
                    a0[b] = pa[0]; a1[b] = pa[half]; b0[b] = pb[0]; b1[b] = pb[half];
                }
#pragma unroll
                for (int b = 0; b < NF; ++b) {
                    const double *base = S + (c0 + ph0[b]) * chunk_doubles + toff;
                    double av[4], bv[4];
#pragma unroll
                    for (int f = 0; f < 4; ++f) { av[f] = base[la_off[b][f]]; bv[f] = base[lb_off[b][f]]; }
                    dmma_m8n8k4_if<1u>(acc[b][0][0], acc[b][0][1], av[0], bv[0], msk[b]);
                    dmma_m8n8k4_if<2u>(acc[b][1][0], acc[b][1][1], av[1], bv[1], msk[b]);
                    dmma_m8n8k4_if<4u>(acc[b][2][0], acc[b][2][1], av[2], bv[2], msk[b]);
                    dmma_m8n8k4_if<8u>(acc[b][3][0], acc[b][3][1], av[3], bv[3], msk[b]);
                }
#pragma unroll
                for (int b = 0; b < NR; ++b) {
                    dmma_m8n8k4(acc[NF + b][0][0], acc[NF + b][0][1], a0[b], b0[b]);
                    dmma_m8n8k4(acc[NF + b][1][0], acc[NF + b][1][1], a0[b], b1[b]);
                    dmma_m8n8k4(acc[NF + b][2][0], acc[NF + b][2][1], a1[b], b0[b]);
                    dmma_m8n8k4(acc[NF + b][3][0], acc[NF + b][3][1], a1[b], b1[b]);
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + st);                    // this warp is done reading the stage
        if (++st == stages_n) { st = 0; ph ^= 1u; }
    }
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const int q = warp + kGramWarps * b;
#pragma unroll
        for (int f = 0; f < 4; ++f)
            *reinterpret_cast<double2 *>(out + (size_t)q * 256 + f * 64 + lane * 2) = make_double2(acc[b][f][0], acc[b][f][1]);
    }
}

// K2 with the tensor-map ring: WARPS consumer warps + one producer warp per CTA; the producer issues one 2-D copy per box
// and 16-row chunk.  Rows >= n and columns >= 1 + p of [y | X] are outside the tensor map and arrive as zeros.
template <int WARPS>
__global__ void __launch_bounds__((WARPS + 1) * 32, 1)
gram_kernel_tma(const GramParams P, const __grid_constant__ GramTmaMaps maps, const fokl::GramBoxMeta *__restrict__ boxes)
{
    constexpr int kGramWarps = WARPS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const GramTileMeta tm = P.tiles[blockIdx.x];
    const size_t stage_doubles = (size_t)(P.kb >> 4) * P.max_slots * 16;
    // the swizzle pattern is a function of the shared-memory address: stages start on a 1024-byte boundary
    double *stages = reinterpret_cast<double *>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    uint64_t *full = reinterpret_cast<uint64_t *>(stages + P.stages * stage_doubles);
    uint64_t *empty = full + kMaxStagesTma;

    const int64_t n_lo = (int64_t)blockIdx.y * P.rows_per_split;
    const int64_t n_hi = (n_lo + P.rows_per_split < P.n) ? n_lo + P.rows_per_split : P.n;
    const int nk = n_hi > n_lo ? (int)((n_hi - n_lo + P.kb - 1) / P.kb) : 0;

    int nb = 0;
    int flex = 0;            // 0: all blocks full and regular, 1: the first one loose / masked, 2: any
    if (warp < kGramWarps) {
        for (int b = 0; b < kGramBlocksPerWarp; ++b) {
            const int q = warp + kGramWarps * b;
            if (q >= tm.n_blk) break;
            const GramBlockMeta bq = P.blocks[tm.blk_off + q];
            if (bq.mask == 0u) break;
            nb = b + 1;
            if (bq.loose != 0 || bq.mask != 15u) flex = b == 0 ? (flex > 1 ? flex : 1) : 2;     // see gram_consume
        }
    }
    const int active = __syncthreads_count(lane == 0 && nb > 0);   // consumer warps that own work (and release stages)
    if (tid == 0) {
        for (int s = 0; s < P.stages; ++s) {
            mbar_init(full + s, 1u);
            mbar_init(empty + s, (unsigned)active);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    __syncthreads();

    if (warp == kGramWarps) {
        if (active == 0) return;
        // bytes per stage: every box is written in full (zero fill included)
        int cols = 0;
        for (int b = 0; b < tm.n_box; ++b) cols += boxes[tm.box_off + b].ncols;
        const int chunks = P.kb >> 4;
        const unsigned stage_bytes = (unsigned)(cols * chunks) * 128u;
        const int stages_n = P.stages;
        int st = 0;
        unsigned ph = 0;
        for (int kt = 0; kt < nk; ++kt) {
            if (kt >= stages_n) mbar_wait(empty + st, ph ^ 1u);
            double *dst = stages + (size_t)st * stage_doubles;
            const int64_t r0 = n_lo + (int64_t)kt * P.kb;
            if (elect_one()) mbar_arrive_expect_tx(full + st, stage_bytes);
            __syncwarp();
            for (int b = 0; b < tm.n_box; ++b) {
                const fokl::GramBoxMeta bx = boxes[tm.box_off + b];
                const CUtensorMap *mp = &maps.m[bx.kind];
                for (int c = 0; c < chunks; ++c) {
                    if (elect_one())
                        tma_load_2d(dst + ((size_t)c * P.max_slots + bx.slot0) * 16, mp, (int)(r0 + 16 * c), bx.xcol0, full + st);
                }
            }
            if (++st == stages_n) { st = 0; ph ^= 1u; }
        }
        return;
    }
    double *out = P.part + ((size_t)blockIdx.y * P.n_tiles + blockIdx.x) * (size_t)(P.tile_blocks * 256);
#define FOKL_ROWS(NB)                                                                                                  \
    if (flex == 0) gram_consume_tma<WARPS, NB, 0>(P, tm, stages, stage_doubles, full, empty, nk, lane, warp, out);      \
    else if (flex == 1) gram_consume_tma<WARPS, NB, 1>(P, tm, stages, stage_doubles, full, empty, nk, lane, warp, out); \
    else gram_consume_tma<WARPS, NB, 2>(P, tm, stages, stage_doubles, full, empty, nk, lane, warp, out);                \
    break;
    switch (nb) {
    case 0: break;
    case 1: FOKL_ROWS(1)
    case 2: FOKL_ROWS(2)
    case 3: FOKL_ROWS(3)
    default: FOKL_ROWS(4)
    }
#undef FOKL_ROWS
}

// The row loop of one CTA for a warp that owns NB blocks (q = warp + 16 b, b < NB).  NB is a template parameter so
// the fragment loads of a k-step are all issued ahead of its DMMAs without per-block branches; MASKED selects the
// predicated DMMA form for warps that own a block with skipped fragments (diagonal / edge blocks).
template <int WARPS, int NB, bool MASKED>
__device__ __forceinline__ void gram_rows(const GramParams &P, const GramTileMeta &tm, double *stages,
                                          const double *const *s_ptr, size_t stage_doubles, int stride, int64_t n_lo,
                                          int64_t n_hi, int nk, int tid, int lane, int warp, double *out)
{
    constexpr int NBA = NB > 0 ? NB : 1;
    constexpr int kGramWarps = WARPS, kGramThreads = WARPS * 32;
    int a_off[NBA], b_off[NBA];
    unsigned msk[NBA];
    const int frag_r = lane >> 2, frag_k = lane & 3;
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const GramBlockMeta bm = P.blocks[tm.blk_off + warp + kGramWarps * b];
        a_off[b] = (bm.a_slot + frag_r) * stride + frag_k;
        b_off[b] = (bm.b_slot + frag_r) * stride + frag_k;
        msk[b] = bm.mask;
    }
    double acc[NBA][4][2];
#pragma unroll
    for (int b = 0; b < NB; ++b)
#pragma unroll
        for (int f = 0; f < 4; ++f) acc[b][f][0] = acc[b][f][1] = 0.0;

    const int segs = tm.n_slots << P.kb_shift;                     // 16-byte segments per stage
    const int seg_mask = (1 << P.kb_shift) - 1;
    auto load_stage = [&](int kt, int buf) {
        double *dst = stages + (size_t)buf * stage_doubles;
        const int64_t r0 = n_lo + (int64_t)kt * P.kb;
        for (int sg = tid; sg < segs; sg += kGramThreads) {
            const int slot = sg >> P.kb_shift, part = sg & seg_mask;
            const double *col = s_ptr[slot];
            if (col == nullptr) continue;
            const int64_t r = r0 + part * 2;
            const int64_t left = n_hi - r;
            const int bytes = left >= 2 ? 16 : (left == 1 ? 8 : 0);
            cp_async16(dst + slot * stride + part * 2, bytes ? col + r : col, bytes);
        }
    };

    const int stages_n = P.stages;
    for (int s = 0; s < stages_n - 1; ++s) {
        if (s < nk) load_stage(s, s);
        cp_async_commit();
    }
    const int half = 8 * stride;                                   // second fragment row / column of a block
    for (int kt = 0; kt < nk; ++kt) {
        if (stages_n == 4) cp_async_wait<2>();
        else cp_async_wait<1>();
        __syncthreads();
        // refill the ring one k-block into the stage (when the slab has more than one), so the DMMAs restart right after
        // the barrier instead of behind the cp.async issue: K2 94 -> 85 ms per cfg4 fit (profiles/r01_gram_variants.txt)
        const int load_at = (NB == 0 || P.kb < 32) ? 0 : 16;       // (tiles of this kernel are never k-split)
        const double *S = stages + (size_t)(kt % stages_n) * stage_doubles;
        for (int k0 = 0; k0 < P.kb; k0 += 16) {
            if (k0 == load_at) {
                const int nxt = kt + stages_n - 1;
                if (nxt < nk) load_stage(nxt, nxt % stages_n);
                cp_async_commit();
                if (NB == 0) break;
            }
#pragma unroll
            for (int kk = 0; kk < 16; kk += 4) {
                double a0[NBA], a1[NBA], b0[NBA], b1[NBA];
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    const double *pa = S + a_off[b] + k0 + kk, *pb = S + b_off[b] + k0 + kk;
                    a0[b] = pa[0]; a1[b] = pa[half]; b0[b] = pb[0]; b1[b] = pb[half];
                }
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    if (MASKED) {
                        dmma_m8n8k4_if<1u>(acc[b][0][0], acc[b][0][1], a0[b], b0[b], msk[b]);
                        dmma_m8n8k4_if<2u>(acc[b][1][0], acc[b][1][1], a0[b], b1[b], msk[b]);
                        dmma_m8n8k4_if<4u>(acc[b][2][0], acc[b][2][1], a1[b], b0[b], msk[b]);
                        dmma_m8n8k4_if<8u>(acc[b][3][0], acc[b][3][1], a1[b], b1[b], msk[b]);
                    } else {
                        dmma_m8n8k4(acc[b][0][0], acc[b][0][1], a0[b], b0[b]);
                        dmma_m8n8k4(acc[b][1][0], acc[b][1][1], a0[b], b1[b]);
                        dmma_m8n8k4(acc[b][2][0], acc[b][2][1], a1[b], b0[b]);
                        dmma_m8n8k4(acc[b][3][0], acc[b][3][1], a1[b], b1[b]);
                    }
                }
            }
        }
    }
    cp_async_wait<0>();

    // accumulators in fragment order: lane l holds C[l >> 2][(l & 3) * 2 + {0, 1}] = row-major 8 x 8 at offset 2 l
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const int q = warp + kGramWarps * b;
#pragma unroll
        for (int f = 0; f < 4; ++f)
            *reinterpret_cast<double2 *>(out + (size_t)q * 256 + f * 64 + lane * 2) = make_double2(acc[b][f][0], acc[b][f][1]);
    }
}

template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 16 / WARPS) gram_kernel(const GramParams P)
{
    constexpr int kGramWarps = WARPS, kGramThreads = WARPS * 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const GramTileMeta tm = P.tiles[blockIdx.x];
    const int stride = P.kb + kPad;
    const size_t stage_doubles = (size_t)P.max_slots * stride;
    double *stages = reinterpret_cast<double *>(smem_raw);
    const double **s_ptr = reinterpret_cast<const double **>(stages + P.stages * stage_doubles);

    const int64_t n_lo = (int64_t)blockIdx.y * P.rows_per_split;
    const int64_t n_hi = (n_lo + P.rows_per_split < P.n) ? n_lo + P.rows_per_split : P.n;
    const int nk = n_hi > n_lo ? (int)((n_hi - n_lo + P.kb - 1) / P.kb) : 0;

    // operand column pointers; padding slots stay zero in every stage (never written by cp.async)
    for (int s = tid; s < tm.n_slots; s += kGramThreads) {
        const int src = P.slot_src[tm.slot_off + s];
        s_ptr[s] = src < 0 ? nullptr : (src == P.p ? P.y : P.X + (int64_t)src * P.ld);
    }
    for (size_t e = tid; e < P.stages * stage_doubles; e += kGramThreads) stages[e] = 0.0;
    __syncthreads();

    double *out = P.part + ((size_t)blockIdx.y * P.n_tiles + blockIdx.x) * (size_t)(P.tile_blocks * 256);
    // work items of this warp: positions q = warp + 16 b < n_blk, filled from b = 0 (mask 0 = hole)
    int nb = 0;
    bool partial = false;
    for (int b = 0; b < kGramBlocksPerWarp; ++b) {
        const int q = warp + kGramWarps * b;
        if (q >= tm.n_blk) break;
        const unsigned mk = P.blocks[tm.blk_off + q].mask;
        if (mk == 0u) break;
        nb = b + 1;
        partial |= mk != 15u;
    }
#define FOKL_ROWS(NB)                                                                                                  \
    if (partial) gram_rows<WARPS, NB, true>(P, tm, stages, s_ptr, stage_doubles, stride, n_lo, n_hi, nk, tid, lane, warp, out); \
    else gram_rows<WARPS, NB, false>(P, tm, stages, s_ptr, stage_doubles, stride, n_lo, n_hi, nk, tid, lane, warp, out);        \
    break;
    switch (nb) {
    case 0: gram_rows<WARPS, 0, false>(P, tm, stages, s_ptr, stage_doubles, stride, n_lo, n_hi, nk, tid, lane, warp, out); break;
    case 1: FOKL_ROWS(1)
    case 2: FOKL_ROWS(2)
    case 3: FOKL_ROWS(3)
    default: FOKL_ROWS(4)
    }
#undef FOKL_ROWS
}

// K2 with the mbarrier ring: WARPS consumer warps + one producer warp per CTA.
template <int WARPS>
__global__ void __launch_bounds__((WARPS + 1) * 32, 1) gram_kernel_mb(const GramParams P)
{
    constexpr int kGramWarps = WARPS, kThreads = (WARPS + 1) * 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const GramTileMeta tm = P.tiles[blockIdx.x];
    const int stride = P.kb + kPad;
    const size_t stage_doubles = (size_t)P.max_slots * stride;
    double *stages = reinterpret_cast<double *>(smem_raw);
    // (same shared-memory carve-up as the cp.async kernel: the column-pointer area holds the run table, 16 bytes per run)
    GramRun *runs = reinterpret_cast<GramRun *>(stages + P.stages * stage_doubles);
    uint64_t *full = reinterpret_cast<uint64_t *>(reinterpret_cast<const double **>(runs) + P.max_slots);
    uint64_t *empty = full + kMaxStages;
    int *run_info = reinterpret_cast<int *>(empty + kMaxStages);      // [0] runs, [1] staged (non-padding) slots

    const int64_t n_lo = (int64_t)blockIdx.y * P.rows_per_split;
    const int64_t n_hi = (n_lo + P.rows_per_split < P.n) ? n_lo + P.rows_per_split : P.n;
    const int nk = n_hi > n_lo ? (int)((n_hi - n_lo + P.kb - 1) / P.kb) : 0;

    // work items of this warp: positions q = warp + 16 b < n_blk, filled from b = 0 (mask 0 = hole)
    int nb = 0;
    int flex = 0;            // 0: all blocks full and regular, 1: the first one loose / masked, 2: any
    if (warp < kGramWarps) {
        for (int b = 0; b < kGramBlocksPerWarp; ++b) {
            const int q = warp + kGramWarps * b;
            if (q >= tm.n_blk) break;
            const GramBlockMeta bq = P.blocks[tm.blk_off + q];
            if (bq.mask == 0u) break;
            nb = b + 1;
            if (bq.loose != 0 || bq.mask != 15u) flex = b == 0 ? (flex > 1 ? flex : 1) : 2;     // see gram_consume
        }
    }
    // runs of staged columns (at most n_slots / 2 of them fit the table: a run of one slot next to padding at worst);
    // padding slots stay zero in every stage (never written by a copy)
    if (tid == 0) {
        int n_runs = 0, n_real = 0, prev = -2;
        for (int sl = 0; sl < tm.n_slots; ++sl) {
            const int src = P.slot_src[tm.slot_off + sl];
            if (src < 0) { prev = -2; continue; }
            ++n_real;
            if (src == prev + 1 && src != P.p && n_runs > 0) {
                ++runs[n_runs - 1].len;
            } else {
                runs[n_runs].src = src == P.p ? P.y : P.X + (int64_t)src * P.ld;
                runs[n_runs].slot0 = sl;
                runs[n_runs].len = 1;
                ++n_runs;
            }
            prev = src;
        }
        run_info[0] = n_runs;
        run_info[1] = n_real;
    }
    for (size_t e = tid; e < P.stages * stage_doubles; e += kThreads) stages[e] = 0.0;
    const int active = __syncthreads_count(lane == 0 && nb > 0);   // consumer warps that own work (and release stages)
    if (tid == 0) {
        for (int s = 0; s < P.stages; ++s) {
            mbar_init(full + s, 1u);
            mbar_init(empty + s, (unsigned)active);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // the zero fill (generic proxy) precedes the bulk copies
    __syncthreads();

    if (warp == kGramWarps) {
        if (active > 0)
            gram_produce(P, stages, stage_doubles, stride, runs, run_info[0], run_info[1], full, empty, n_lo, n_hi, nk, P.ld, lane);
        return;
    }
    double *out = P.part + ((size_t)blockIdx.y * P.n_tiles + blockIdx.x) * (size_t)(P.tile_blocks * 256);
#define FOKL_ROWS(NB)                                                                                                          \
    if (flex == 0) gram_consume<WARPS, NB, 0>(P, tm, stages, stage_doubles, stride, full, empty, nk, lane, warp, out);          \
    else if (flex == 1) gram_consume<WARPS, NB, 1>(P, tm, stages, stage_doubles, stride, full, empty, nk, lane, warp, out);     \
    else gram_consume<WARPS, NB, 2>(P, tm, stages, stage_doubles, stride, full, empty, nk, lane, warp, out);                    \
    break;
    switch (nb) {
    case 0: break;
    case 1: FOKL_ROWS(1)
    case 2: FOKL_ROWS(2)
    case 3: FOKL_ROWS(3)
    default: FOKL_ROWS(4)
    }
#undef FOKL_ROWS
}

// Sum the row splits in a fixed order and scatter the fragments to the (p + 1) x c block.  One thread per
// accumulator element of every block of every tile.
__global__ void gram_reduce_kernel(const double *__restrict__ part, int nsplit, int n_tiles, const GramTileMeta *tiles,
                                   const GramBlockMeta *blocks, const int32_t *slot_arow, const int32_t *slot_bcol,
                                   int c, int tile_blocks, double *__restrict__ out)
{
    const int tile = blockIdx.y;
    const GramTileMeta tm = tiles[tile];
    const int total = tm.n_blk * 256;
    const size_t tile_stride = (size_t)tile_blocks * 256;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int q = e >> 8, f = (e >> 6) & 3, idx = e & 63;
        const GramBlockMeta bm = blocks[tm.blk_off + q];
        if (bm.phase != 0 || !(bm.mask >> f & 1u)) continue;   // not the head item of a block / fragment not computed
        const int arow = slot_arow[tm.slot_off + bm.la[f] + (idx >> 3)];
        const int bcol = slot_bcol[tm.slot_off + bm.lb[f] + (idx & 7)];
        if (arow < 0 || bcol < 0) continue;
        double s = 0.0;
        for (int qq = q; qq >= 0; qq = blocks[tm.blk_off + qq].next) {      // the block's items in phase order
            const double *src = part + (size_t)tile * tile_stride + (size_t)qq * 256 + (e & 255);
            // same ascending order (same bits), eight loads in flight instead of one dependent load per add
            const size_t kstride = (size_t)n_tiles * tile_stride;
            int k = 0;
            for (; k + 8 <= nsplit; k += 8) {
                double v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = __ldcg(src + (size_t)(k + j) * kstride);
#pragma unroll
                for (int j = 0; j < 8; ++j) s += v[j];
            }
            for (; k < nsplit; ++k) s += __ldcg(src + (size_t)k * kstride);
        }
        out[(size_t)arow * c + bcol] = s;
    }
}

}  // namespace

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn tensor_map_encoder()
{
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            return nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// [y | X] as a (cols x rows) float64 tensor, fetched in boxes of `box_cols` columns x 16 rows with the 128-byte swizzle;
// rows >= n and columns >= cols read as zeros.
bool encode_gram_map(CUtensorMap *map, const double *base, int64_t ld, int64_t n, int cols, int box_cols)
{
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)n, (cuuint64_t)cols};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(double)};
    const cuuint32_t box[2] = {16u, (cuuint32_t)box_cols};
    const cuuint32_t estr[2] = {1u, 1u};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(base), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

extern "C" int fokl_gram_last_config(fokl_ctx *ctx, int64_t out[9])
{
    FOKL_CHECK_CTX(ctx);
    if (!out) FOKL_FAIL(ctx, FOKL_EINVAL, "gram_last_config: bad argument");
    if (ctx->gram_cfg[0] < 0) FOKL_FAIL(ctx, FOKL_ESTATE, "gram_last_config: no Gram update on this context yet");
    memcpy(out, ctx->gram_cfg, sizeof ctx->gram_cfg);
    return FOKL_OK;
}

extern "C" int fokl_gram_update(fokl_ctx *ctx, const double *X, int64_t ld, int64_t n, int p_old, int c,
                                const double *y, double *block)
{
    return fokl_gram_update_ex(ctx, X, ld, n, p_old, c, p_old, 0, y, block);
}

extern "C" int fokl_gram_update_ex(fokl_ctx *ctx, const double *X, int64_t ld, int64_t n, int p_old, int c, int new_col0,
                                   int flags, const double *y, double *block)
{
    FOKL_CHECK_CTX(ctx);
    if (!X || !y || !block || n < 1 || p_old < 0 || c < 1 || ld < n || new_col0 < p_old)
        FOKL_FAIL(ctx, FOKL_EINVAL, "gram_update: bad argument");
    const int gap = new_col0 - p_old;
    const bool cross_only = (flags & FOKL_GRAM_CROSS_ONLY) != 0;
    if ((ld % 2) != 0 || ((uintptr_t)X % 16) != 0 || ((uintptr_t)y % 16) != 0)
        FOKL_FAIL(ctx, FOKL_EINVAL, "gram_update: X and y must be 16-byte aligned and ld even");
    if (p_old + c + 1 > 65000) FOKL_FAIL(ctx, FOKL_EINVAL, "gram_update: more than 65000 columns");
    if (cross_only && p_old < 1) FOKL_FAIL(ctx, FOKL_EINVAL, "gram_update: cross-only block without old columns");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    const int p = p_old + c;

    // CTA shape: one CTA of 16 warps per SM.  (Measured alternative, profiles/r01_gram_variants.txt: 8 warps with two
    // co-resident CTAs per SM and half the blocks each is 1.65x slower -- more duplicated operand traffic and
    // instruction-cache misses between the two CTAs' code paths.)
    // Two pipelines feed the DMMAs (profiles/r01_gram_ksplit.txt):
    //  * mbarrier ring (gram_kernel_mb): 15 consumer warps + 1 producer warp issuing one bulk copy per staged column and
    //    slab; no CTA-wide barrier.  A bulk copy costs the SM's copy engine ~60 cycles whatever its size, so this needs
    //    slabs of >= 64 rows (>= 512-byte copies): tiles of up to ~130 staged columns.  (A 17th warp would put five
    //    warps on one SM sub-partition and cap the kernel at 96 registers per thread.)
    //  * cp.async ring (gram_kernel): 16 warps, 16-byte cp.async by every thread and one __syncthreads per slab; the
    //    wide tiles of the three-way substages (~220 staged columns, 32-row slabs) run faster here.
    const int ctas_per_sm = 1;
    const size_t smem_total = ctx->smem_optin ? ctx->smem_optin : 48 * 1024;
    const size_t smem_cap = smem_total - 1024;
    auto smem_need = [&](int slots, int kb, int stages) {
        return (size_t)stages * slots * (kb + kPad) * sizeof(double) + (size_t)slots * sizeof(double *) +
               2 * kMaxStages * sizeof(uint64_t) + 16;
    };
    int cap = 32;
    while (smem_need(cap + 16, 16, kMaxStages) <= smem_cap) cap += 16;
    // tuning knobs (tools/gram_sweep.py): FOKL_GRAM_KERNEL = mb | cpasync, FOKL_GRAM_KB, FOKL_GRAM_STAGES
    const char *env_kernel = getenv("FOKL_GRAM_KERNEL");
    const int env_kb = getenv("FOKL_GRAM_KB") ? atoi(getenv("FOKL_GRAM_KB")) : 0;
    const int env_stages = getenv("FOKL_GRAM_STAGES") ? atoi(getenv("FOKL_GRAM_STAGES")) : 0;
    // * tensor-map ring (gram_kernel_tma): when y is stored in the row in front of X (the engine's [y | X] buffer) the
    //   operands of a tile are a handful of column runs of one 2-D tensor; one TMA copy moves a box of up to 128 columns
    //   x 16 rows, so the copy count no longer grows with the staged columns and the ring is 4 - 8 stages deep.
    //   A box is 16 rows deep (the swizzle span), so narrow tiles would move 1 KB per copy: they stay on the bulk-copy ring.
    const bool can_tma = (y + ld == X) && (ld % 16) == 0 && tensor_map_encoder() != nullptr;
    bool use_tma = can_tma && env_kernel && !strcmp(env_kernel, "tma");
    bool use_mb = !use_tma && !(env_kernel && !strcmp(env_kernel, "cpasync"));
    // FOKL_GRAM_WARPS = 12 / 15: force the consumer-warp count of the tensor-map kernel (tuning knob)
    const int env_warps = getenv("FOKL_GRAM_WARPS") ? atoi(getenv("FOKL_GRAM_WARPS")) : 0;
    int warps = 15, kb = 0, stages = 0;
    fokl::GramPlan plan;
    auto smem_need_tma = [&](int slots, int kb_, int st) {
        return (size_t)st * (kb_ / 16) * slots * 128 + 2 * kMaxStagesTma * sizeof(uint64_t) + 1024;
    };
    if (use_mb || use_tma) {
        plan = fokl::gram_make_plan(p_old, c, cap, warps, gap, cross_only);
        if (plan.tiles.empty() || plan.max_slots > cap) FOKL_FAIL(ctx, FOKL_ESTATE, "gram_update: empty or oversized plan");
    }
    if (use_mb) {
        // deepest slab that leaves a ring of >= 3 stages (>= 2 for slabs of >= 128 rows)
        for (int cand_kb = 256; cand_kb >= 64 && kb == 0; cand_kb /= 2) {
            if (n < (int64_t)cand_kb * 4) continue;
            for (int st = kMaxStages; st >= (cand_kb >= 128 ? 2 : 3); --st)
                if (smem_need(plan.max_slots, cand_kb, st) <= smem_cap) { kb = cand_kb; stages = st; break; }
        }
        if (kb == 0 && !env_kernel) { use_mb = false; use_tma = can_tma; }       // wide tile: tensor-map ring, else cp.async
    }
    if (use_tma && env_warps == 12) {
        // 12 consumer warps (three per sub-partition next to the producer): a tuning knob since the placement deals the
        // work items evenly over the sub-partitions (gram_plan.h, mode 2) -- 15 warps are then as fast or faster on every
        // shape of the cfg4 fit (profiles/r02_gram_round2.txt)
        fokl::GramPlan p12 = fokl::gram_make_plan(p_old, c, cap, 12, gap, cross_only);
        if (!p12.tiles.empty() && p12.max_slots <= cap) {
            warps = 12;
            plan = p12;
        }
    }
    if (use_tma) {
        // deepest slab that leaves a ring of >= 4 stages
        kb = 0;
        for (int cand_kb = 256; cand_kb >= 16 && kb == 0; cand_kb /= 2) {
            if (cand_kb > 16 && n < (int64_t)cand_kb * 4) continue;
            for (int st = kMaxStagesTma; st >= (cand_kb > 16 ? 4 : 2); --st)
                if (smem_need_tma(plan.max_slots, cand_kb, st) <= smem_cap) { kb = cand_kb; stages = st; break; }
        }
        if (kb == 0) use_tma = false;
    }
    if (!use_mb && !use_tma) {
        warps = 16;
        plan = fokl::gram_make_plan(p_old, c, cap, warps, gap, cross_only, -1, false);    // (this kernel has no loose-block form)
        if (plan.tiles.empty() || plan.max_slots > cap) FOKL_FAIL(ctx, FOKL_ESTATE, "gram_update: empty or oversized plan");
        // deepest slab that fits (fewer CTA-wide barriers per row), giving up one ring stage for it if necessary
        kb = 0;
        for (int cand_kb = 256; cand_kb >= 32; cand_kb /= 2) {
            if (cand_kb > 64 && plan.max_slots * (cand_kb + kPad) * (int)sizeof(double) > 40 * 1024) continue;   // <= 40 KB per stage
            if (n < (int64_t)cand_kb * 4) continue;
            if (smem_need(plan.max_slots, cand_kb, 4) <= smem_cap) { kb = cand_kb; stages = 4; break; }
            if (smem_need(plan.max_slots, cand_kb, 3) <= smem_cap) { kb = cand_kb; stages = 3; break; }
        }
    }
    if (kb == 0) { kb = 16; stages = kMaxStages; }
    if (env_kb >= 16 && env_kb <= 256 && (env_kb & (env_kb - 1)) == 0) kb = env_kb;
    if (env_stages >= 2 && env_stages <= (use_tma ? kMaxStagesTma : kMaxStages)) stages = env_stages;
    if (!use_mb && !use_tma && stages < 3) stages = 3;            // the cp.async ring waits on groups of a 3- or 4-deep ring
    if ((use_tma ? smem_need_tma(plan.max_slots, kb, stages) : smem_need(plan.max_slots, kb, stages)) > smem_cap)
        FOKL_FAIL(ctx, FOKL_EINVAL, "gram_update: slab does not fit in shared memory");
    const int n_tiles = (int)plan.tiles.size();
    const int kTileBlocks = fokl::gram_tile_blocks(warps);
    int kb_shift = 0;
    while ((2 << kb_shift) < kb) ++kb_shift;
    // placement (gram_plan.h): 2 = even deal over the SM sub-partitions with at most one loose block per warp (the
    // default), 1 = sequential deal, 0 = balanced by needed fragments
    const int place_mode = getenv("FOKL_GRAM_PLACE") ? atoi(getenv("FOKL_GRAM_PLACE")) : 2;
    // k-split of tiles with few blocks (gram_plan.h); the cp.async kernel works whole slabs per item
    // FOKL_GRAM_KSPLIT: force the k-split (largest admissible power of two <= the value; tuning knob)
    const int force_r = getenv("FOKL_GRAM_KSPLIT") ? atoi(getenv("FOKL_GRAM_KSPLIT")) : 0;
    fokl::gram_plan_place(plan, warps, (use_mb || use_tma) ? kb / 16 : 1, place_mode, force_r);

    // row splits: about one resident CTA slot each
    const int64_t chunks = (n + kb - 1) / kb;
    // a context with an SM budget (fokl_ctx_set_sm_budget) leaves the other SMs to the latency-bound kernels of the
    // candidate stage it runs next to
    const int sms_use = (ctx->sm_budget > 0 && ctx->sm_budget < ctx->num_sms) ? ctx->sm_budget : ctx->num_sms;
    const int slots_total = sms_use * ctas_per_sm;
    int64_t want = std::max<int64_t>(1, slots_total / n_tiles);
    if (n_tiles > slots_total) want = 1;
    int nsplit = (int)std::max<int64_t>(1, std::min<int64_t>(want, chunks));
    int64_t rows_per_split = ((chunks + nsplit - 1) / nsplit) * kb;
    nsplit = (int)((n + rows_per_split - 1) / rows_per_split);

    // upload the plan (one buffer)
    const size_t n_slots = plan.slot_src.size(), n_blocks = plan.blocks.size();
    size_t off_tiles = 0;
    size_t off_src = off_tiles + (size_t)n_tiles * sizeof(GramTileMeta);
    size_t off_arow = off_src + n_slots * sizeof(int32_t);
    size_t off_bcol = off_arow + n_slots * sizeof(int32_t);
    size_t off_blk = off_bcol + n_slots * sizeof(int32_t);
    size_t off_box = (off_blk + n_blocks * sizeof(GramBlockMeta) + 15) & ~(size_t)15;
    size_t meta_bytes = off_box + plan.boxes.size() * sizeof(fokl::GramBoxMeta);
    std::vector<unsigned char> host(meta_bytes);
    memcpy(host.data() + off_tiles, plan.tiles.data(), (size_t)n_tiles * sizeof(GramTileMeta));
    memcpy(host.data() + off_src, plan.slot_src.data(), n_slots * sizeof(int32_t));
    memcpy(host.data() + off_arow, plan.slot_arow.data(), n_slots * sizeof(int32_t));
    memcpy(host.data() + off_bcol, plan.slot_bcol.data(), n_slots * sizeof(int32_t));
    memcpy(host.data() + off_blk, plan.blocks.data(), n_blocks * sizeof(GramBlockMeta));
    memcpy(host.data() + off_box, plan.boxes.data(), plan.boxes.size() * sizeof(fokl::GramBoxMeta));
    const size_t part_bytes = (size_t)nsplit * n_tiles * kTileBlocks * 256 * sizeof(double);
    const size_t part_off = (meta_bytes + 255) & ~(size_t)255;
    unsigned char *buf = (unsigned char *)fokl_scratch(ctx, fokl_ctx::B_GRAM, part_off + part_bytes);
    if (!buf) return FOKL_ENOMEM;
    // stream-ordered behind any kernel still reading the previous plan; pageable source = staged before return
    FOKL_CUDA(ctx, cudaMemcpyAsync(buf, host.data(), meta_bytes, cudaMemcpyHostToDevice, ctx->stream));
    FOKL_CUDA(ctx, cudaMemsetAsync(block, 0, (size_t)(p + 1) * c * sizeof(double), ctx->stream));

    GramParams P;
    P.X = X; P.y = y; P.ld = ld; P.n = n; P.p = p + gap;      // slot source P.p marks y (physical indices, gram_plan.h)
    P.kb = kb; P.kb_shift = kb_shift; P.stages = stages; P.max_slots = plan.max_slots;
    P.rows_per_split = rows_per_split;
    P.tiles = reinterpret_cast<const GramTileMeta *>(buf + off_tiles);
    P.slot_src = reinterpret_cast<const int32_t *>(buf + off_src);
    P.blocks = reinterpret_cast<const GramBlockMeta *>(buf + off_blk);
    P.part = reinterpret_cast<double *>(buf + part_off);
    P.n_tiles = n_tiles;
    P.tile_blocks = kTileBlocks;
    const int64_t cfg[9] = {use_tma ? 2 : (use_mb ? 1 : 0), warps, kb, stages, n_tiles, nsplit, rows_per_split,
                            plan.max_slots, cap};
    memcpy(ctx->gram_cfg, cfg, sizeof cfg);
    const size_t smem = use_tma ? smem_need_tma(plan.max_slots, kb, stages) : smem_need(plan.max_slots, kb, stages);
    if (use_tma) {
        GramTmaMaps maps;
        for (int k = 0; k < fokl::kGramBoxKinds; ++k)
            if (!encode_gram_map(&maps.m[k], y, ld, n, p + gap + 1, fokl::kGramBoxCols[k]))
                FOKL_FAIL(ctx, FOKL_ECUDA, "gram_update: cuTensorMapEncodeTiled failed");
        if (warps == 12) {
            FOKL_CUDA(ctx, cudaFuncSetAttribute(gram_kernel_tma<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));
            gram_kernel_tma<12><<<dim3(n_tiles, nsplit), 13 * 32, smem, ctx->stream>>>(
                P, maps, reinterpret_cast<const fokl::GramBoxMeta *>(buf + off_box));
        } else {
            FOKL_CUDA(ctx, cudaFuncSetAttribute(gram_kernel_tma<15>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));
            gram_kernel_tma<15><<<dim3(n_tiles, nsplit), 16 * 32, smem, ctx->stream>>>(
                P, maps, reinterpret_cast<const fokl::GramBoxMeta *>(buf + off_box));
        }
    } else if (!use_mb) {
        FOKL_CUDA(ctx, cudaFuncSetAttribute(gram_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));
        gram_kernel<16><<<dim3(n_tiles, nsplit), 512, smem, ctx->stream>>>(P);
    } else {
        FOKL_CUDA(ctx, cudaFuncSetAttribute(gram_kernel_mb<15>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));
        gram_kernel_mb<15><<<dim3(n_tiles, nsplit), 16 * 32, smem, ctx->stream>>>(P);
    }
    FOKL_LAUNCH_CHECK(ctx);
    gram_reduce_kernel<<<dim3(kTileBlocks, n_tiles), 256, 0, ctx->stream>>>(
        P.part, nsplit, n_tiles, P.tiles, P.blocks, reinterpret_cast<const int32_t *>(buf + off_arow),
        reinterpret_cast<const int32_t *>(buf + off_bcol), c, kTileBlocks, block);
    FOKL_LAUNCH_CHECK(ctx);
    return FOKL_OK;
}
