// dgreduce.h — TEST INFRASTRUCTURE ONLY.  Steps 2 and 3 of the deterministic per-key sums (DESIGN.md §4.9) for one
// window on the host, shared by the gradient simulators: the window's pairs (key[e], e) sorted with std::stable_sort in
// place of the onesweep sort (a stable sort of the same keys yields the same permutation), the run starts, level 0
// with contrib(e, out) the contribution of pair e, and the further levels, all with the RT_HD functions of
// rt_distgrad.cuh.  Each key below n_keys adds its sum to acc[key].
#pragma once
#include <algorithm>
#include <numeric>
#include <vector>
#include "../../trimesh-ray-optix_b200/csrc/rt_distgrad.cuh"

template <class Contrib>
void dg_reduce_host(const std::vector<uint64_t>& key, uint64_t n_keys, const Contrib& contrib, float* acc) {
    using namespace rt;
    const int64_t m = (int64_t)key.size();
    std::vector<uint32_t> vals(m);
    std::iota(vals.begin(), vals.end(), 0u);
    std::stable_sort(vals.begin(), vals.end(), [&](uint32_t a, uint32_t b) { return key[a] < key[b]; });
    std::vector<uint64_t> keys(m);
    for (int64_t j = 0; j < m; ++j) keys[j] = key[vals[j]];
    std::vector<uint32_t> start(n_keys);
    for (int64_t j = 0; j < m; ++j) dg_run_start(j, keys.data(), n_keys, start.data());
    const uint64_t slots = dg_next_size(m);
    std::vector<uint32_t> lk[2], li[2];
    std::vector<float> lv[2];
    for (int b = 0; b < 2; ++b) { lk[b].assign(slots, kDgEmpty); li[b].assign(slots, 0); lv[b].assign(3 * slots, 0.0f); }
    DgLevel lev[2] = {{lk[0].data(), li[0].data(), lv[0].data()}, {lk[1].data(), li[1].data(), lv[1].data()}};
    for (int64_t j = 0; j < m; ++j) dg_level0_with(j, m, keys.data(), vals.data(), start.data(), n_keys, contrib, acc, lev[0]);
    uint64_t size = m, len = m;
    int cur = 0;
    while (len > kDgGroup) {
        size = dg_next_size(size);
        len = (len + kDgGroup - 1) / kDgGroup;
        std::fill(lk[cur ^ 1].begin(), lk[cur ^ 1].end(), kDgEmpty);
        for (uint64_t j = 0; j < size; ++j) dg_level_at(j, size, lev[cur], acc, lev[cur ^ 1]);
        cur ^= 1;
    }
}
