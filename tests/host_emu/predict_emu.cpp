// predict_emu.cpp -- host build of the per-row prediction summary (csrc/predict_math.cuh) (TEST INFRASTRUCTURE).
// The same functions the summary kernel calls, run by a single-lane team: pw_leaves / pw_leaf / pw_tree for the mean,
// order_key / select_key / key_value for the ranks.  Build: g++ -O2 -ffp-contract=off -shared -fPIC.
#include <cstdint>
#include <vector>
#include "../../fokl-gpy_b200/csrc/predict_math.cuh"

using namespace fokl;

extern "C" {

// a: n x d row-major; mean[n]; when rank_lo >= 0 also lo[n], hi[n] = the values at ascending ranks rank_lo, rank_hi
void emu_predict_summary(const double *a, int64_t n, int d, int rank_lo, int rank_hi, double *mean, double *lo,
                         double *hi)
{
    std::vector<double> leaf(pw_leaf_count(d));
    std::vector<uint64_t> keys(d);
    uint32_t hist[256];
    for (int64_t i = 0; i < n; ++i) {
        const double *v = a + i * d;
        pw_leaves(d, [&](int t, int off, int len) { leaf[t] = pw_leaf(v + off, len); });
        mean[i] = pw_mean(pw_tree(d, leaf.data()), d);
        if (rank_lo < 0) continue;
        uint64_t kmin = ~0ull, kmax = 0ull;
        for (int j = 0; j < d; ++j) {
            keys[j] = order_key(v[j]);
            kmin = keys[j] < kmin ? keys[j] : kmin;
            kmax = keys[j] > kmax ? keys[j] : kmax;
        }
        lo[i] = key_value(select_key(keys.data(), d, rank_lo, hist, 0, 1, kmin, kmax));
        hi[i] = key_value(select_key(keys.data(), d, rank_hi, hist, 0, 1, kmin, kmax));
    }
}

int emu_pw_leaf_count(int d) { return pw_leaf_count(d); }

}
