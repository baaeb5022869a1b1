// trainlog_emu.cpp -- host build of the device train split (csrc/trainlog_math.cuh, csrc/trainlog.cu) (TEST
// INFRASTRUCTURE).  The same rounds as fokl_trainlog: randint words set bits of an n-bit bitmap, the shuffle words are
// parsed tile by tile (words decided by interval_classify against the tile's bound range, the kDepends ones in order),
// and the last round's kept set is the bitmap minus shuffle_final_value of every position >= l_log.
// Build: g++ -O2 -std=c++17 -shared -fPIC.
#include <cstdint>
#include <cstring>
#include <vector>
#include "../../fokl-gpy_b200/csrc/trainlog_math.cuh"

using namespace fokl;

namespace {

struct Stream {
    uint32_t key[kMtN];
    int pos;
    uint32_t next()
    {
        if (pos == kMtN) {
            mt_next_block(key);
            pos = 0;
        }
        return mt_temper(key[pos++]);
    }
};

// the words from the start state, generated on demand
struct Words {
    Stream st;
    std::vector<uint32_t> w;
    uint32_t at(int64_t i)
    {
        while ((int64_t)w.size() <= i) w.push_back(st.next());
        return w[i];
    }
};

// Consumes words from *off until R steps have accepted one; step s has bound `fixed` (>= 0: randint) or U - 1 - s.
// on_step(s, word).  Returns -1 if a word decided by classification disagrees with its actual bound.
template <class F>
int parse(Words &wd, int64_t &off, int64_t R, int64_t fixed, int64_t U, int tile, F on_step)
{
    auto bound = [&](int64_t s) { return (uint32_t)(fixed >= 0 ? fixed : U - 1 - s); };
    int64_t s = 0;
    std::vector<int> cls(tile);
    while (s < R) {
        uint32_t hi = bound(s);
        uint32_t lo = fixed >= 0 ? hi : (hi >= (uint32_t)tile ? hi - (uint32_t)(tile - 1) : 1u);
        for (int t = 0; t < tile; ++t) cls[t] = interval_classify(wd.at(off + t), lo, hi);
        int t = 0;
        for (; t < tile && s < R; ++t) {
            uint32_t w = wd.at(off + t), b = bound(s);
            bool acc = interval_accepts(w, b);
            if (cls[t] != kDepends && (cls[t] == kAccept) != acc) return -1;
            if (acc) on_step(s++, w);
        }
        off += t;
    }
    return 0;
}

}  // namespace

extern "C" {

// count tempered words from (key, pos); the state after them -> key_out, pos_out
void emu_mt_words(const uint32_t *key, int pos, int64_t count, uint32_t *out, uint32_t *key_out, int *pos_out)
{
    Stream st;
    memcpy(st.key, key, sizeof st.key);
    st.pos = pos;
    for (int64_t i = 0; i < count; ++i) out[i] = st.next();
    memcpy(key_out, st.key, sizeof st.key);
    *pos_out = st.pos;
}

// fokl_trainlog's contract on the host: keep[n] (0/1), the state after the last consumed word, the words consumed,
// rounds.  tile = words per parse tile.  Returns 0, -1 on bad arguments, -2 on a misclassified word.
int emu_trainlog(const uint32_t *key, int pos, int64_t n, int64_t l_log, int tile, uint8_t *keep, uint32_t *key_out,
                 int *pos_out, int64_t *words_out, int *rounds_out)
{
    if (!key || !keep || !key_out || !pos_out || !words_out || pos < 0 || pos > kMtN || l_log < 2 || l_log > n ||
        n >= (int64_t(1) << 31) || tile < 1)
        return -1;
    Words wd;
    memcpy(wd.st.key, key, sizeof wd.st.key);
    wd.st.pos = pos;
    int64_t off = 0;
    std::vector<uint32_t> bitmap((n + 31) / 32, 0u);
    int64_t U = 0;
    int rounds = 0;
    const uint32_t mask_n = interval_mask((uint32_t)(n - 1));
    std::vector<int32_t> j;
    while (U < l_log) {
        ++rounds;
        if (parse(wd, off, l_log, n - 1, 0, tile, [&](int64_t, uint32_t w) {
                uint32_t v = w & mask_n;
                bitmap[v >> 5] |= 1u << (v & 31);
            }))
            return -2;
        U = 0;
        for (uint32_t b : bitmap) U += __builtin_popcount(b);
        bool last = U >= l_log;
        if (last) j.assign(U - l_log, 0);
        if (parse(wd, off, U - 1, -1, U, tile, [&](int64_t s, uint32_t w) {
                int64_t i = U - 1 - s;
                if (last && i >= l_log) j[i - l_log] = (int32_t)(w & interval_mask((uint32_t)i));
            }))
            return -2;
    }
    std::vector<int32_t> u;
    u.reserve(U);
    for (int64_t r = 0; r < n; ++r)
        if (bitmap[r >> 5] >> (r & 31) & 1u) u.push_back((int32_t)r);
    std::vector<int32_t> head(U, -1), next(U - l_log, -1);
    for (int64_t i = l_log; i < U; ++i) {
        next[i - l_log] = head[j[i - l_log]];
        head[j[i - l_log]] = (int32_t)i;
    }
    for (int64_t r = 0; r < n; ++r) keep[r] = bitmap[r >> 5] >> (r & 31) & 1u;
    for (int64_t i = l_log; i < U; ++i) keep[shuffle_final_value(i, j.data(), head.data(), next.data(), u.data(), l_log)] = 0;
    // the state after word `off` - 1 of the stream
    Stream st;
    memcpy(st.key, key, sizeof st.key);
    st.pos = pos;
    for (int64_t i = 0; i < off; ++i) st.next();
    memcpy(key_out, st.key, sizeof st.key);
    *pos_out = st.pos;
    *words_out = off;
    if (rounds_out) *rounds_out = rounds;
    return 0;
}

}
