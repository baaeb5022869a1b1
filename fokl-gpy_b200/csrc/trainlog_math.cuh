// trainlog_math.cuh -- per-word rules of the train split (FR:509-530 `generate_trainlog`), shared by the sm_100a kernels
// (csrc/trainlog.cu) and the host emulation build (tests/host_emu/trainlog_emu.cpp).
//
// numpy's legacy RandomState draws from MT19937 (key[624], pos).  A word is temper(key[pos++]); at pos == 624 the whole
// key is first replaced by its twist (mt19937_gen).  Both calls of the split consume one word per trial:
//   * randint(1, n + 1, size=l_log): masked rejection, value = w & mask(n - 1), retried while value > n - 1;
//   * shuffle of the sorted unique indices (length U), Fisher-Yates: for i = U - 1 .. 1, j = w & mask(i), retried while
//     j > i (random_interval), then swap(a[i], a[j]).
// Step s of a parse has the bound n - 1 (randint) or U - 1 - s (shuffle).
#pragma once
#include "fokl_math.cuh"
#include <stdint.h>

namespace fokl {

constexpr int kMtN = 624;
constexpr int kMtM = 397;

FOKL_HD uint32_t mt_temper(uint32_t y)
{
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

// one word of the twist: new key[k] from key[k], key[k + 1] and key[k + 397] as mt19937_gen reads them in place --
// the old key[k + 1] (the new key[0] for k = 623) and the old key[k + 397] for k < 227, the new key[k - 227] after
FOKL_HD uint32_t mt_twist(uint32_t cur, uint32_t next, uint32_t far)
{
    uint32_t y = (cur & 0x80000000u) | (next & 0x7fffffffu);
    return far ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}

FOKL_HD void mt_next_block(uint32_t *key)
{
    for (int k = 0; k < kMtN; ++k)
        key[k] = mt_twist(key[k], key[(k + 1) % kMtN], key[(k + kMtM) % kMtN]);
}

// smallest 2^b - 1 >= v (numpy's gen_mask / random_interval mask)
FOKL_HD uint32_t interval_mask(uint32_t v)
{
    v |= v >> 1;
    v |= v >> 2;
    v |= v >> 4;
    v |= v >> 8;
    v |= v >> 16;
    return v;
}

FOKL_HD bool interval_accepts(uint32_t w, uint32_t bound) { return (w & interval_mask(bound)) <= bound; }

enum { kReject = 0, kAccept = 1, kDepends = 2 };

// The word w (tempered) tested at every bound in [lo, hi] (1 <= lo <= hi): kAccept if every bound accepts it, kReject
// if none does, else kDepends.  Within one mask the accepted bounds are those >= (w & mask), so each power-of-two piece
// of the range is decided by its ends.  A parse tile whose steps can only have bounds in [lo, hi] decides its words
// with this in parallel and leaves only the kDepends ones to a sequential pass.
FOKL_HD int interval_classify(uint32_t w, uint32_t lo, uint32_t hi)
{
    bool acc = false, rej = false;
    uint32_t b = hi;
    while (true) {
        uint32_t m = interval_mask(b);
        uint32_t piece_lo = (m >> 1) + 1 > lo ? (m >> 1) + 1 : lo;
        uint32_t v = w & m;
        if (v <= piece_lo)
            acc = true;
        else if (v > b)
            rej = true;
        else
            return kDepends;
        if (piece_lo == lo) break;
        b = piece_lo - 1;
    }
    return acc && rej ? kDepends : (acc ? kAccept : kReject);
}

// The last round's shuffle keeps the set of a[0 .. l_log) -- the unique indices u minus the values that end up at the
// positions i >= l_log, each final after step i.  With j_i known for every such step, the value at position p just
// before step t (p <= t) is u[p] unless an earlier step (a k > t with j_k = p; the latest is the smallest such k) wrote
// it, in which case it is the value at position k just before step k.  head[p] / next[k - l_log] list the steps k with
// j_k = p (any order).  Returns the value at position i after the shuffle, for l_log <= i < U.
FOKL_HD int32_t shuffle_final_value(int64_t i, const int32_t *j, const int32_t *head, const int32_t *next,
                                    const int32_t *u, int64_t l_log)
{
    int64_t p = j[i - l_log], t = i;
    while (true) {
        int64_t best = -1;
        for (int64_t k = head[p]; k >= 0; k = next[k - l_log])
            if (k > t && (best < 0 || k < best)) best = k;
        if (best < 0) return u[p];
        p = best;
        t = best;
    }
}

}  // namespace fokl
