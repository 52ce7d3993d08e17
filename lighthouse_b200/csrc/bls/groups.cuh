// groups.cuh — host-side plan of a grouped verification (lhb200_verify_signature_set_groups): the chunk tables of the
// segmented reductions, whose chunks never cross a group boundary.  Plain C++ (also compiled into tests/hostsim).
//
// The inputs of a segmented reduction are stored group after group: group g owns cnt[g] consecutive values.  One level
// cuts group g into max(1, ceil(cnt[g] / chunk)) chunks; chunk t of the level covers inputs [seg[t], seg[t + 1]) and
// yields one output, the outputs again stored group after group.  An empty group gets one empty chunk, whose output is
// the neutral element (the infinity point, Fp12 one), so after the first level every group holds at least one value.
#pragma once
#include <stdint.h>
#include <algorithm>
#include <vector>

namespace lhb200 {
namespace groups {

constexpr uint32_t SUM_CHUNK = 4;       // points per warp and level of the segmented G2 sum (as k_g2_sum_warp's latency mode)
constexpr uint32_t FOLD_CHUNK = 8;      // Miller values per thread and level of the segmented product (k_fp12_reduce_seg)
constexpr uint32_t FOLD_MAX = 16;       // values k_final_groups_warp folds per group itself (~7 us each)

struct Levels {
    std::vector<uint32_t> at, n_out;    // per level: position of its table in the plan's words, number of outputs
    uint64_t max_out = 0;
};

// Append one level's table (n_out + 1 chunk starts) to `words`; cnt becomes the per-group output counts.
inline uint32_t add_level(std::vector<uint32_t>& words, std::vector<uint32_t>& cnt, uint32_t chunk) {
    uint32_t in = 0, n_out = 0;
    for (uint32_t& c : cnt) {
        const uint32_t k = c ? (c + chunk - 1) / chunk : 1;
        for (uint32_t j = 0; j < k; j++) words.push_back(in + j * chunk);
        in += c;
        n_out += k;
        c = k;
    }
    words.push_back(in);
    return n_out;
}

// Levels until every group holds at most `max_per_group` values and, if `at_least_one`, no group is empty.
inline Levels plan_levels(std::vector<uint32_t>& words, std::vector<uint32_t>& cnt, uint32_t chunk, uint32_t max_per_group,
                          bool at_least_one) {
    Levels L;
    for (;;) {
        bool done = true;
        for (uint32_t c : cnt) done = done && c <= max_per_group && (c > 0 || !at_least_one);
        if (done) return L;
        L.at.push_back((uint32_t)words.size());
        L.n_out.push_back(add_level(words, cnt, chunk));
        L.max_out = std::max<uint64_t>(L.max_out, L.n_out.back());
    }
}

// The whole plan of one call, uploaded as one array of words:
//   [group offsets (n_groups + 1) | sum tables | product tables | value offsets (n_groups + 1)]
// The sum levels leave exactly one point per group (group g's sum at index g; no level at all when every group has
// one set: the sets' own points are the sums).  The product levels run only while some group has more than FOLD_MAX
// Miller values; the value offsets then index the last level's outputs, otherwise they are the group offsets.
struct Plan {
    uint32_t n_groups = 0;
    std::vector<uint32_t> words;
    Levels sum, fold;
    uint32_t val_off_at = 0;
};

inline void build_plan(Plan& p, const uint32_t* group_offsets, uint32_t n_groups) {
    p.n_groups = n_groups;
    p.words.assign(group_offsets, group_offsets + n_groups + 1);
    std::vector<uint32_t> cnt(n_groups);
    for (uint32_t g = 0; g < n_groups; g++) cnt[g] = group_offsets[g + 1] - group_offsets[g];
    std::vector<uint32_t> c = cnt;
    p.sum = plan_levels(p.words, c, SUM_CHUNK, 1, true);
    c = cnt;
    p.fold = plan_levels(p.words, c, FOLD_CHUNK, FOLD_MAX, false);
    p.val_off_at = (uint32_t)p.words.size();
    uint32_t acc = 0;
    p.words.push_back(0);
    for (uint32_t g = 0; g < n_groups; g++) p.words.push_back(acc += c[g]);
}

}  // namespace groups
}  // namespace lhb200
