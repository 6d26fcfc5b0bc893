// fm_shard.h -- how image pairs are split over GPUs, shared by bin/match -gpus (match_main.cpp) and fm_group_match
// (fm_api.cu).  Host-only, no CUDA.
#pragma once
#include <algorithm>
#include <cstddef>
#include <numeric>
#include <vector>

namespace fm {

// Longest-processing-time-first sharding of independent image pairs (match.cpp:638-652).  weight[p] is pair p's
// N_first * N_second.  Pairs are taken by descending weight (stable: equal weights keep submission order), each goes to
// the first of the G shards with the least load so far, and every shard comes back in ascending pair order
// (consecutive pairs share their first image).  With fewer pairs than shards, the last shards stay empty.
inline std::vector<std::vector<size_t>> shard_pairs(const std::vector<double>& weight, int G) {
  std::vector<std::vector<size_t>> shard(G);
  std::vector<size_t> order(weight.size());
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return weight[a] > weight[b]; });
  std::vector<double> load(G, 0.0);
  for (size_t id : order) {
    const int g = (int)(std::min_element(load.begin(), load.end()) - load.begin());
    shard[g].push_back(id);
    load[g] += weight[id];
  }
  for (auto& s : shard) std::sort(s.begin(), s.end());
  return shard;
}

}  // namespace fm
