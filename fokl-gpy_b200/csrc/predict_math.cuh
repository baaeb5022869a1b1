// predict_math.cuh -- per-row summary of the prediction draws, shared by the sm_100a kernels (csrc/predict.cu) and the
// host emulation build (tests/host_emu/predict_emu.cpp).
//
// For one row v[0..n) of X @ betas' the summary is numpy's `np.mean(v)` and `np.sort(v)[k]`, bit for bit:
//   * the mean is numpy's pairwise sum (loops_utils.h.src, PW_BLOCKSIZE 128) added to the reduction identity 0.0 and
//     divided by n.  Leaves of at most 128 elements are summed with 8 strided accumulators (plain loop below 8);
//     longer runs split at n2 = n/2 - (n/2) % 8.  The device sums the leaves on different lanes, then combines them in
//     the tree's order (pw_tree), which is the recursion's order of additions;
//   * ranks are selected on an order-preserving integer key of each double: NaN (any sign or payload) sorts last, as
//     in numpy, and -0.0 gets the key of +0.0 (numpy's sort treats them as equal and is not stable, so only the sign
//     of a zero result may differ from numpy's).  The selection is an MSD radix select, 8 bits a pass, starting at the
//     highest bit in which the row's smallest and largest keys differ, and stopping as soon as one key is left.
#pragma once
#include "fokl_math.cuh"
#include <string.h>

namespace fokl {

constexpr int kPwBlock = 128;      // numpy PW_BLOCKSIZE

FOKL_HD int pw_split(int n) { return n / 2 - (n / 2) % 8; }

// numpy's pairwise sum of a run of at most 128 elements
FOKL_HD double pw_leaf(const double *a, int n)
{
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; ++i) res = FOKL_ADD(res, a[i]);
        return res;
    }
    double r[8];
    for (int k = 0; k < 8; ++k) r[k] = a[k];
    int i = 8;
    for (; i < n - (n % 8); i += 8)
        for (int k = 0; k < 8; ++k) r[k] = FOKL_ADD(r[k], a[i + k]);
    double res = FOKL_ADD(FOKL_ADD(FOKL_ADD(r[0], r[1]), FOKL_ADD(r[2], r[3])),
                          FOKL_ADD(FOKL_ADD(r[4], r[5]), FOKL_ADD(r[6], r[7])));
    for (; i < n; ++i) res = FOKL_ADD(res, a[i]);
    return res;
}

// Leaves of the pairwise recursion over n elements, in order: f(index, offset, length) for each; returns their count.
template <class F>
FOKL_HD int pw_leaves(int n, F &&f)
{
    int off[40], len[40], sp = 0, count = 0;
    off[0] = 0;
    len[0] = n;
    sp = 1;
    while (sp > 0) {
        --sp;
        int o = off[sp], l = len[sp];
        if (l <= kPwBlock) {
            f(count++, o, l);
            continue;
        }
        int n2 = pw_split(l);
        off[sp] = o + n2; len[sp] = l - n2; ++sp;      // right half, visited after the left one
        off[sp] = o;      len[sp] = n2;     ++sp;
    }
    return count;
}

FOKL_HD int pw_leaf_count(int n)
{
    return pw_leaves(n, [](int, int, int) {});
}

// Sum of n elements from their leaf sums (pw_leaves order), added as numpy's recursion adds them.
FOKL_HD double pw_tree(int n, const double *leaf)
{
    int len[40], state[40], sp = 1, next = 0;
    double left[40], ret = 0.0;
    len[0] = n;
    state[0] = 0;
    while (true) {
        int l = len[sp - 1];
        if (l <= kPwBlock) {
            ret = leaf[next++];
            --sp;
        } else if (state[sp - 1] == 0) {
            state[sp - 1] = 1;
            len[sp] = pw_split(l); state[sp] = 0; ++sp;
            continue;
        } else if (state[sp - 1] == 1) {
            left[sp - 1] = ret;
            state[sp - 1] = 2;
            len[sp] = l - pw_split(l); state[sp] = 0; ++sp;
            continue;
        } else {
            ret = FOKL_ADD(left[sp - 1], ret);
            --sp;
        }
        if (sp == 0) return ret;
    }
}

// np.mean of a row: (0.0 + pairwise sum) / n
FOKL_HD double pw_mean(double sum, int n)
{
#if defined(__CUDA_ARCH__)
    return __ddiv_rn(__dadd_rn(0.0, sum), (double)n);
#else
    return (0.0 + sum) / (double)n;
#endif
}

FOKL_HD uint64_t dbits(double v)
{
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(v);
#else
    uint64_t u;
    memcpy(&u, &v, sizeof u);
    return u;
#endif
}

FOKL_HD double bits_to_double(uint64_t u)
{
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)u);
#else
    double v;
    memcpy(&v, &u, sizeof v);
    return v;
#endif
}

constexpr uint64_t kSignBit = 0x8000000000000000ull;

// ascending order of doubles as numpy sorts them -> ascending unsigned keys
FOKL_HD uint64_t order_key(double v)
{
    if (v != v) return ~0ull;
    uint64_t u = v == 0.0 ? 0ull : dbits(v);
    return (u & kSignBit) ? ~u : (u | kSignBit);
}

FOKL_HD double key_value(uint64_t k) { return bits_to_double((k & kSignBit) ? (k & ~kSignBit) : ~k); }

FOKL_HD uint64_t shr64(uint64_t x, int s) { return s >= 64 ? 0ull : x >> s; }

// Key of ascending rank k (0-based) among keys[0..n), kmin / kmax their smallest and largest.  Run by a team of nlane
// lanes (one warp on the device, one thread on the host) sharing the 256 counters `hist`.
FOKL_HD uint64_t select_key(const uint64_t *keys, int n, int k, uint32_t *hist, int lane, int nlane, uint64_t kmin,
                            uint64_t kmax)
{
    uint64_t diff = kmin ^ kmax;
    if (diff == 0) return kmin;
#if defined(__CUDA_ARCH__)
    int hi = 64 - __clzll((long long)diff);       // bits [hi, 64) are the same in every key
#else
    int hi = 64 - __builtin_clzll(diff);
#endif
    uint64_t prefix = shr64(kmin, hi) << (hi & 63);
    while (true) {
        const int lo = hi > 8 ? hi - 8 : 0;
        const uint32_t dmask = (1u << (hi - lo)) - 1u;
        const uint64_t want = shr64(prefix, hi);
        for (int b = lane; b < 256; b += nlane) hist[b] = 0;
#if defined(__CUDA_ARCH__)
        __syncwarp();
#endif
        for (int i = lane; i < n; i += nlane) {
            uint64_t key = keys[i];
            if (shr64(key, hi) == want) {
#if defined(__CUDA_ARCH__)
                atomicAdd(&hist[(uint32_t)(key >> lo) & dmask], 1u);
#else
                ++hist[(uint32_t)(key >> lo) & dmask];
#endif
            }
        }
        uint32_t digit = 0, below = 0, cnt = 0;
#if defined(__CUDA_ARCH__)
        __syncwarp();
        {   // each lane owns 8 consecutive digits; an inclusive scan over the lanes finds the one holding rank k
            uint32_t c[8], s = 0;
            for (int t = 0; t < 8; ++t) { c[t] = hist[lane * 8 + t]; s += c[t]; }
            uint32_t incl = s;
            for (int o = 1; o < 32; o <<= 1) {
                uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += y;
            }
            uint32_t excl = incl - s;
            unsigned owner = __ballot_sync(0xffffffffu, excl <= (uint32_t)k && (uint32_t)k < incl);
            int src = __ffs(owner) - 1;
            uint32_t d = 0, bl = excl, ct = 0;
            for (int t = 0; t < 8; ++t) {
                if ((uint32_t)k < bl + c[t]) { d = lane * 8 + t; ct = c[t]; break; }
                bl += c[t];
            }
            digit = __shfl_sync(0xffffffffu, d, src);
            below = __shfl_sync(0xffffffffu, bl, src);
            cnt = __shfl_sync(0xffffffffu, ct, src);
        }
        __syncwarp();
#else
        for (uint32_t b = 0; b < 256; ++b) {
            if ((uint32_t)k < below + hist[b]) { digit = b; cnt = hist[b]; break; }
            below += hist[b];
        }
#endif
        k -= (int)below;
        prefix |= (uint64_t)digit << lo;
        if (lo == 0) return prefix;
        if (cnt == 1) {    // one key left under this prefix: it is the answer
            const uint64_t w = prefix >> lo;
#if defined(__CUDA_ARCH__)
            for (int i0 = 0; i0 < n; i0 += 32) {
                int i = i0 + lane;
                uint64_t key = i < n ? keys[i] : 0ull;
                unsigned hit = __ballot_sync(0xffffffffu, i < n && (key >> lo) == w);
                if (hit) return __shfl_sync(0xffffffffu, key, __ffs(hit) - 1);
            }
#else
            for (int i = 0; i < n; ++i)
                if ((keys[i] >> lo) == w) return keys[i];
#endif
        }
        hi = lo;
    }
}

}  // namespace fokl
