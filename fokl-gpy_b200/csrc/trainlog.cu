// trainlog.cu -- `generate_trainlog` (FR:509-530) in HBM, bit for bit with numpy's legacy RandomState: the keep-mask
// and the MT19937 state after the last word numpy would have consumed (fokl_trainlog, include/fokl_b200.h).
//
// The rounds of the reference loop, with the rules of csrc/trainlog_math.cuh:
//   * trainlog_mt_gen: one CTA streams MT19937 blocks (twist in three dependent phases of <= 227 words) into a window of
//     raw key words; windows follow one another as the parse uses them up, so the ~70 M words of a 10^7-row split
//     never exist at once;
//   * trainlog_parse: one CTA walks the window in tiles of kParseTile words.  A step's bound is n - 1 (randint) or
//     U - 1 - s (shuffle step s), so every word of a tile is tested against the tile's bound range at once
//     (interval_classify); the few words whose verdict depends on the exact step are decided in order by one thread,
//     and a block scan gives every accepted word its step.  randint steps set bits of an n-bit bitmap (the set, not its
//     order, is what np.unique keeps); shuffle steps of the last round record j_i for the positions i >= l_log;
//   * trainlog_popcount / trainlog_scan: U = bits set; trainlog_unique: the sorted unique indices u;
//   * trainlog_link / trainlog_exclude: the values that end up at positions >= l_log (shuffle_final_value, pointer
//     chains over the recorded j_i instead of ~10^6 dependent swaps) are cleared from the mask trainlog_keep wrote.
#include "fokl_ctx.cuh"
#include "trainlog_math.cuh"

using namespace fokl;

namespace {

constexpr int kGenThreads = 256;
constexpr int kParseThreads = 1024;
constexpr int kParsePer = 4;                                  // consecutive words per thread and tile
constexpr int kParseTile = kParseThreads * kParsePer;         // 4096 words
constexpr int kPopThreads = 256;
constexpr int kPopPer = 16;
constexpr int kPopTile = kPopThreads * kPopPer;               // bitmap words per popcount / unique block
constexpr int64_t kWindowBlocks = 16384;                      // MT blocks per window: 10.2 M words, 41 MB (L2-resident)

struct ParseState {
    int64_t off;      // next word of the window
    int64_t s;        // steps done
};

}  // namespace

__global__ void __launch_bounds__(kGenThreads) trainlog_mt_gen(uint32_t *__restrict__ key, int copy_first,
                                                               int64_t blocks, uint32_t *__restrict__ out)
{
    __shared__ uint32_t buf[2][kMtN];
    int t = threadIdx.x;
    for (int k = t; k < kMtN; k += kGenThreads) buf[0][k] = key[k];
    __syncthreads();
    int c = 0;
    for (int64_t b = 0; b < blocks; ++b) {
        if (b > 0 || !copy_first) {
            const uint32_t *o = buf[c];
            uint32_t *w = buf[c ^ 1];
            if (t < 227) w[t] = mt_twist(o[t], o[t + 1], o[t + kMtM]);
            __syncthreads();
            if (t < 227) w[227 + t] = mt_twist(o[227 + t], o[228 + t], w[t]);
            __syncthreads();
            if (t < 170) w[454 + t] = mt_twist(o[454 + t], t < 169 ? o[455 + t] : w[0], w[227 + t]);
            __syncthreads();
            c ^= 1;
        }
        uint32_t *dst = out + b * kMtN;
        for (int k = t; k < kMtN; k += kGenThreads) dst[k] = buf[c][k];
        __syncthreads();      // the next twist overwrites the other buffer only; this one is read above
    }
    for (int k = t; k < kMtN; k += kGenThreads) key[k] = buf[c][k];
}

// exclusive scan of one 64-bit value per thread over the block; *total (shared) = the block's sum
static __device__ __forceinline__ uint64_t block_excl_scan(uint64_t v, uint64_t *warp_s, uint64_t &total)
{
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint64_t s = v;
    for (int o = 1; o < 32; o <<= 1) {
        uint64_t u = __shfl_up_sync(0xffffffffu, s, o);
        if (lane >= o) s += u;
    }
    if (lane == 31) warp_s[warp] = s;
    __syncthreads();
    if (warp == 0) {
        uint64_t w = lane < nw ? warp_s[lane] : 0;
        for (int o = 1; o < 32; o <<= 1) {
            uint64_t u = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += u;
        }
        warp_s[lane] = w;
    }
    __syncthreads();
    total = warp_s[nw - 1];
    uint64_t r = s - v + (warp > 0 ? warp_s[warp - 1] : 0);
    __syncthreads();      // warp_s is reused by the next scan
    return r;
}

// Steps st->s .. R - 1 from word st->off of the window words[0, W).  fixed >= 0: randint (bound fixed, set bitmap
// bits); else shuffle (bound U - 1 - s; jrec != nullptr records j_i for i >= l_log).  Stops at the R-th step or at the
// end of the window, and writes the state back.
__global__ void __launch_bounds__(kParseThreads) trainlog_parse(const uint32_t *__restrict__ words, int64_t W,
                                                                ParseState *st, int64_t R, int64_t fixed, int64_t U,
                                                                int64_t l_log, uint32_t *__restrict__ bitmap,
                                                                int32_t *__restrict__ jrec)
{
    __shared__ uint64_t warp_s[32];
    __shared__ uint32_t dep_word[kParseTile];
    __shared__ uint16_t dep_before[kParseTile];      // accepted-for-sure words of the tile before it
    __shared__ uint8_t dep_ok[kParseTile];
    __shared__ int64_t cut_end;
    const int tid = threadIdx.x;
    int64_t off = st->off, s = st->s;
    const uint32_t mask_fixed = fixed >= 0 ? interval_mask((uint32_t)fixed) : 0u;
    uint32_t cur[kParsePer], nxt[kParsePer];
#pragma unroll
    for (int r = 0; r < kParsePer; ++r) {
        int64_t i = off + tid * kParsePer + r;
        cur[r] = i < W ? words[i] : 0u;
    }
    while (s < R && off < W) {
#pragma unroll
        for (int r = 0; r < kParsePer; ++r) {          // the next tile's words, while this one is decided
            int64_t i = off + kParseTile + tid * kParsePer + r;
            nxt[r] = i < W ? words[i] : 0u;
        }
        uint32_t hi = fixed >= 0 ? (uint32_t)fixed : (uint32_t)(U - 1 - s);
        uint32_t lo = fixed >= 0 ? hi : (hi >= (uint32_t)kParseTile ? hi - (uint32_t)(kParseTile - 1) : 1u);
        uint32_t w[kParsePer];
        unsigned acc = 0, dep = 0;
#pragma unroll
        for (int r = 0; r < kParsePer; ++r) {
            w[r] = mt_temper(cur[r]);
            int64_t i = off + tid * kParsePer + r;
            int c = i < W ? interval_classify(w[r], lo, hi) : kReject;
            acc |= (c == kAccept ? 1u : 0u) << r;
            dep |= (c == kDepends ? 1u : 0u) << r;
        }
        uint64_t tot;
        uint64_t pre = block_excl_scan((uint64_t)__popc(acc) | ((uint64_t)__popc(dep) << 32), warp_s, tot);
        uint32_t n_dep = (uint32_t)(tot >> 32);
        uint32_t before = (uint32_t)pre;
        uint64_t total = tot & 0xffffffffu;
        if (n_dep) {
            uint32_t e = (uint32_t)(pre >> 32), b = before;
#pragma unroll
            for (int r = 0; r < kParsePer; ++r) {
                if (dep >> r & 1u) {
                    dep_word[e] = w[r];
                    dep_before[e] = (uint16_t)b;
                    ++e;
                }
                b += acc >> r & 1u;
            }
            __syncthreads();
            if (tid == 0) {
                uint32_t extra = 0;
                for (uint32_t k = 0; k < n_dep; ++k) {
                    int64_t step = s + dep_before[k] + extra;
                    bool ok = false;
                    if (step < R) {
                        uint32_t bound = fixed >= 0 ? (uint32_t)fixed : (uint32_t)(U - 1 - step);
                        ok = interval_accepts(dep_word[k], bound);
                    }
                    dep_ok[k] = ok;
                    extra += ok;
                }
            }
            __syncthreads();
            e = (uint32_t)(pre >> 32);
#pragma unroll
            for (int r = 0; r < kParsePer; ++r)
                if (dep >> r & 1u) acc |= (unsigned)dep_ok[e++] << r;
            before = (uint32_t)block_excl_scan((uint64_t)__popc(acc), warp_s, total);
        }
        int64_t step = s + before;
#pragma unroll
        for (int r = 0; r < kParsePer; ++r) {
            if (!(acc >> r & 1u) || step >= R) continue;
            if (fixed >= 0) {
                uint32_t v = w[r] & mask_fixed;
                atomicOr(&bitmap[v >> 5], 1u << (v & 31));
            } else if (jrec) {
                int64_t i = U - 1 - step;
                if (i >= l_log) jrec[i - l_log] = (int32_t)(w[r] & interval_mask((uint32_t)i));
            }
            if (step == R - 1) cut_end = off + tid * kParsePer + r + 1;
            ++step;
        }
        __syncthreads();
        if (s + (int64_t)total >= R) {
            s = R;
            off = cut_end;
        } else {
            s += (int64_t)total;
            off = off + kParseTile < W ? off + kParseTile : W;
        }
#pragma unroll
        for (int r = 0; r < kParsePer; ++r) cur[r] = nxt[r];
    }
    if (tid == 0) {
        st->off = off;
        st->s = s;
    }
}

__global__ void __launch_bounds__(kPopThreads) trainlog_popcount(const uint32_t *__restrict__ bitmap, int64_t nw,
                                                                 int64_t *__restrict__ tile_count)
{
    int64_t base = (int64_t)blockIdx.x * kPopTile;
    int c = 0;
    for (int r = 0; r < kPopPer; ++r) {
        int64_t i = base + r * kPopThreads + threadIdx.x;
        c += i < nw ? __popc(bitmap[i]) : 0;
    }
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    __shared__ int warp_c[kPopThreads / 32];
    if ((threadIdx.x & 31) == 0) warp_c[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < kPopThreads / 32; ++w) t += warp_c[w];
        tile_count[blockIdx.x] = t;
    }
}

// exclusive scan of the tile counts in place (one block); total -> *total
__global__ void __launch_bounds__(1024) trainlog_scan(int64_t *__restrict__ tile_off, int64_t tiles,
                                                      int64_t *__restrict__ total)
{
    __shared__ uint64_t warp_s[32];
    int64_t carry = 0;
    for (int64_t b0 = 0; b0 < tiles; b0 += 1024) {
        int64_t i = b0 + threadIdx.x;
        uint64_t v = i < tiles ? (uint64_t)tile_off[i] : 0, all;
        uint64_t pre = block_excl_scan(v, warp_s, all);
        if (i < tiles) tile_off[i] = carry + (int64_t)pre;
        carry += (int64_t)all;
    }
    if (threadIdx.x == 0) *total = carry;
}

// u: the set bits of the bitmap in ascending order.  Thread k of a block owns bitmap words base + k * kPopPer ..
__global__ void __launch_bounds__(kPopThreads) trainlog_unique(const uint32_t *__restrict__ bitmap, int64_t nw,
                                                               const int64_t *__restrict__ tile_off,
                                                               int32_t *__restrict__ u)
{
    __shared__ uint64_t warp_s[32];
    int64_t base = (int64_t)blockIdx.x * kPopTile + (int64_t)threadIdx.x * kPopPer;
    int c = 0;
    for (int r = 0; r < kPopPer; ++r) c += base + r < nw ? __popc(bitmap[base + r]) : 0;
    uint64_t all;
    int64_t o = tile_off[blockIdx.x] + (int64_t)block_excl_scan((uint64_t)c, warp_s, all);
    for (int r = 0; r < kPopPer; ++r) {
        if (base + r >= nw) break;
        uint32_t bits = bitmap[base + r];
        while (bits) {
            int b = __ffs(bits) - 1;
            bits &= bits - 1;
            u[o++] = (int32_t)((base + r) * 32 + b);
        }
    }
}

// next[i - l_log] / head[p]: the steps i >= l_log with j_i = p, as singly linked lists (order irrelevant)
__global__ void trainlog_link(const int32_t *__restrict__ j, int64_t l_log, int64_t U, int32_t *__restrict__ head,
                              int32_t *__restrict__ next)
{
    for (int64_t i = l_log + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < U; i += (int64_t)gridDim.x * blockDim.x)
        next[i - l_log] = atomicExch(&head[j[i - l_log]], (int32_t)i);
}

__global__ void trainlog_keep(const uint32_t *__restrict__ bitmap, int64_t n, uint8_t *__restrict__ keep)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x)
        keep[r] = (uint8_t)(bitmap[r >> 5] >> (r & 31) & 1u);
}

__global__ void trainlog_exclude(const int32_t *__restrict__ j, const int32_t *__restrict__ head,
                                 const int32_t *__restrict__ next, const int32_t *__restrict__ u, int64_t l_log,
                                 int64_t U, uint8_t *__restrict__ keep)
{
    for (int64_t i = l_log + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < U; i += (int64_t)gridDim.x * blockDim.x)
        keep[shuffle_final_value(i, j, head, next, u, l_log)] = 0;
}

namespace {

// device buffers of one call, stream-ordered: freed (and the stream drained) on every return path
struct Scratch {
    fokl_ctx *ctx;
    std::vector<void *> ptrs;
    explicit Scratch(fokl_ctx *c) : ctx(c) {}
    void *get(size_t bytes)
    {
        void *p = nullptr;
        if (cudaMallocAsync(&p, bytes ? bytes : 16, ctx->stream) != cudaSuccess) {
            cudaGetLastError();
            char m[160];
            snprintf(m, sizeof m, "trainlog: workspace allocation of %zu bytes failed", bytes);
            ctx->err = m;
            return nullptr;
        }
        ptrs.push_back(p);
        return p;
    }
    ~Scratch()
    {
        for (void *p : ptrs) cudaFreeAsync(p, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
    }
};

int grid_for(fokl_ctx *ctx, int64_t items, int threads, int per_sm)
{
    int64_t b = (items + threads - 1) / threads;
    int64_t cap = (int64_t)ctx->num_sms * per_sm;
    return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

extern "C" int fokl_trainlog(fokl_ctx *ctx, const uint32_t *key, int pos, int64_t n, int64_t l_log, uint8_t *keep,
                             uint32_t *key_out, int *pos_out, int64_t *words_out)
{
    FOKL_CHECK_CTX(ctx);
    if (!key || !keep || !key_out || !pos_out || !words_out || pos < 0 || pos > kMtN || l_log < 2 || l_log > n ||
        n >= (int64_t(1) << 31))
        FOKL_FAIL(ctx, FOKL_EINVAL, "trainlog: bad argument");
    int rc = fokl_bind_device(ctx);
    if (rc) return rc;
    cudaStream_t sm = ctx->stream;
    Scratch scr(ctx);

    // a window holds about what one round needs (<= 2 words per randint step, <= 2 per shuffle step), at least 2 blocks
    int64_t wblocks = (4 * (n + l_log) + kMtN - 1) / kMtN + 2;
    if (wblocks > kWindowBlocks) wblocks = kWindowBlocks;
    const int64_t W = wblocks * kMtN;
    const int64_t nw = (n + 31) / 32;
    const int64_t pop_tiles = (nw + kPopTile - 1) / kPopTile;
    uint32_t *d_key = (uint32_t *)scr.get(kMtN * sizeof(uint32_t));
    uint32_t *window = (uint32_t *)scr.get((size_t)W * sizeof(uint32_t));
    uint32_t *bitmap = (uint32_t *)scr.get((size_t)nw * sizeof(uint32_t));
    int64_t *tiles = (int64_t *)scr.get((size_t)(pop_tiles + 1) * sizeof(int64_t));
    ParseState *d_st = (ParseState *)scr.get(sizeof(ParseState));
    if (!d_key || !window || !bitmap || !tiles || !d_st) return FOKL_ENOMEM;
    FOKL_CUDA(ctx, cudaMemcpyAsync(d_key, key, kMtN * sizeof(uint32_t), cudaMemcpyHostToDevice, sm));
    FOKL_CUDA(ctx, cudaMemsetAsync(bitmap, 0, (size_t)nw * sizeof(uint32_t), sm));
    trainlog_mt_gen<<<1, kGenThreads, 0, sm>>>(d_key, 1, wblocks, window);    // block 0 is the current key itself
    FOKL_LAUNCH_CHECK(ctx);
    int64_t win_base = 0;       // stream position of window[0]
    int64_t off = pos;          // next word

    // steps 0 .. R - 1 of one parse, generating windows as it runs out of words
    auto parse = [&](int64_t R, int64_t fixed, int64_t U, int32_t *jrec) -> int {
        ParseState h = {off, 0};
        while (true) {
            FOKL_CUDA(ctx, cudaMemcpyAsync(d_st, &h, sizeof h, cudaMemcpyHostToDevice, sm));
            trainlog_parse<<<1, kParseThreads, 0, sm>>>(window, W, d_st, R, fixed, U, l_log, bitmap, jrec);
            FOKL_LAUNCH_CHECK(ctx);
            FOKL_CUDA(ctx, cudaMemcpyAsync(&h, d_st, sizeof h, cudaMemcpyDeviceToHost, sm));
            FOKL_CUDA(ctx, cudaStreamSynchronize(sm));
            if (h.s >= R) break;
            trainlog_mt_gen<<<1, kGenThreads, 0, sm>>>(d_key, 0, wblocks, window);
            FOKL_LAUNCH_CHECK(ctx);
            win_base += W;
            h.off = 0;
        }
        off = h.off;
        return FOKL_OK;
    };

    int64_t U = 0;
    int32_t *u = nullptr, *j = nullptr, *head = nullptr, *next = nullptr;
    while (U < l_log) {
        if ((rc = parse(l_log, n - 1, 0, nullptr))) return rc;
        trainlog_popcount<<<(unsigned)pop_tiles, kPopThreads, 0, sm>>>(bitmap, nw, tiles);
        FOKL_LAUNCH_CHECK(ctx);
        trainlog_scan<<<1, 1024, 0, sm>>>(tiles, pop_tiles, tiles + pop_tiles);
        FOKL_LAUNCH_CHECK(ctx);
        FOKL_CUDA(ctx, cudaMemcpyAsync(&U, tiles + pop_tiles, sizeof U, cudaMemcpyDeviceToHost, sm));
        FOKL_CUDA(ctx, cudaStreamSynchronize(sm));
        bool last = U >= l_log;
        if (last) {
            int64_t H = U - l_log;
            u = (int32_t *)scr.get((size_t)U * sizeof(int32_t));
            j = (int32_t *)scr.get((size_t)H * sizeof(int32_t));
            head = (int32_t *)scr.get((size_t)U * sizeof(int32_t));
            next = (int32_t *)scr.get((size_t)H * sizeof(int32_t));
            if (!u || !j || !head || !next) return FOKL_ENOMEM;
            trainlog_unique<<<(unsigned)pop_tiles, kPopThreads, 0, sm>>>(bitmap, nw, tiles, u);
            FOKL_LAUNCH_CHECK(ctx);
        }
        if (U > 1 && (rc = parse(U - 1, -1, U, last ? j : nullptr))) return rc;
    }

    // keep-mask: bitmap minus the values the shuffle moved to positions >= l_log
    trainlog_keep<<<grid_for(ctx, n, 256, 8), 256, 0, sm>>>(bitmap, n, keep);
    FOKL_LAUNCH_CHECK(ctx);
    if (U > l_log) {
        FOKL_CUDA(ctx, cudaMemsetAsync(head, 0xff, (size_t)U * sizeof(int32_t), sm));
        trainlog_link<<<grid_for(ctx, U - l_log, 256, 8), 256, 0, sm>>>(j, l_log, U, head, next);
        FOKL_LAUNCH_CHECK(ctx);
        trainlog_exclude<<<grid_for(ctx, U - l_log, 256, 8), 256, 0, sm>>>(j, head, next, u, l_log, U, keep);
        FOKL_LAUNCH_CHECK(ctx);
    }
    // the state after the last consumed word (off - 1 of this window; off >= 1, the window holds that word)
    int64_t last_blk = (off - 1) / kMtN;
    FOKL_CUDA(ctx, cudaMemcpyAsync(key_out, window + last_blk * kMtN, kMtN * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                                   sm));
    FOKL_CUDA(ctx, cudaStreamSynchronize(sm));
    *pos_out = (int)((off - 1) % kMtN + 1);
    *words_out = win_base + off - pos;
    return FOKL_OK;
}
