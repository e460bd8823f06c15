// Stateless minibatch sampling — device twin of nn_distributed_training_b200/data/sampler.py.
// A batch is a pure function of (seed, node, call index): the epoch permutation is a
// keyed 4-round Feistel network with cycle walking, evaluated in registers, so the whole
// training round is CUDA-graph capturable and no index list is ever stored or copied.
#pragma once
#include "common.cuh"

namespace nndt {

NNDT_DEVINL uint32_t mix_key(uint32_t seed, uint32_t node, uint32_t epoch) {
  uint32_t x = seed * 0x9E3779B1u + node * 0x85EBCA77u + epoch * 0xC2B2AE3Du + 0x27D4EB2Fu;
  x ^= x >> 16; x *= 0x7FEB352Du; x ^= x >> 15; x *= 0x846CA68Bu; x ^= x >> 16;
  return x;
}

NNDT_DEVINL uint32_t feistel_round(uint32_t x, uint32_t k, uint32_t mask) {
  x = (x ^ k) * 0x9E3779B1u;
  x ^= x >> 15;
  x *= 0x85EBCA6Bu;
  x ^= x >> 13;
  return x & mask;
}

// bijection of [0, m); pos < m
NNDT_DEVINL uint32_t feistel_permute(uint32_t pos, uint32_t m, uint32_t key) {
  if (m <= 1) return 0;
  int bits = 32 - __clz(m - 1);
  if (bits < 2) bits = 2;
  const int h = (bits + 1) >> 1;
  const uint32_t mask = (1u << h) - 1u;
  uint32_t x = pos;
  do {
    uint32_t l = x >> h, r = x & mask;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t rk = (i == 0) ? 0xA511E9B3u : (i == 1) ? 0x63D83595u : (i == 2) ? 0x1B873593u : 0xCC9E2D51u;
      const uint32_t t = l ^ feistel_round(r, key + rk, mask);
      l = r; r = t;
    }
    x = (l << h) | r;
  } while (x >= m);
  return x;
}

// DataLoader-equivalent batch geometry of the c-th draw over m samples (batch B).
struct BatchLoc { uint32_t epoch, start, size; };
NNDT_DEVINL BatchLoc locate_batch(uint32_t call, uint32_t m, uint32_t B) {
  const uint32_t bpe = (m + B - 1) / B;
  BatchLoc o;
  o.epoch = call / bpe;
  o.start = (call % bpe) * B;
  o.size = min(B, m - o.start);
  return o;
}

// Online sliding-window stream (floorplans/lidar/lidar.py:397-424 as index arithmetic).  One period of a node's
// stream is described by the table [K, P, cum[0..kWinMax], lb[kWinMax], ub[kWinMax]] (ops/mlp_fused.py:
// FusedMLP._window_table): K windows of rows [lb, ub), P draws per period, window w starting at draw cum[w].
constexpr int kWinMax = 64;
constexpr int kWinTableLen = 2 + (kWinMax + 1) + 2 * kWinMax;

// shard row of draw d (counted from the start of the stream) of node `node`
NNDT_DEVINL int window_draw(const long long* wt, long long d, uint32_t seed, uint32_t node) {
  const long long K = wt[0], P = wt[1];
  const long long q = d / P, r = d - q * P;
  int w = 0;
  while (w + 1 < K && wt[2 + w + 1] <= r) ++w;
  const long long lb = wt[2 + kWinMax + 1 + w], ub = wt[2 + kWinMax + 1 + kWinMax + w];
  const uint32_t wkey = mix_key(seed, node, (uint32_t)(q * K + w));
  return (int)lb + (int)feistel_permute((uint32_t)(r - wt[2 + w]), (uint32_t)(ub - lb), wkey);
}

}  // namespace nndt
