// tcgen05 / TMEM implementation of the implicit-density MLPs (FourierNet and ReLU nets).
//
// One CTA processes tiles of 128 batch rows.  Per tile the hidden GEMMs run on the 5th-gen
// tensor cores: activations live in shared memory as bf16 128B-swizzled slabs that are written
// by the previous layer's epilogue, weights are staged once per CTA as bf16 slabs, accumulators
// are fp32 in TMEM (M = 128: TMEM lane == batch row) and are read back with tcgen05.ld for the
// fused bias+activation epilogue.  The K=2 Fourier/SIREN input layer (sin on the SFU) and the
// 64->1 output layer (+sigmoid, +loss) stay on CUDA cores inside the same kernel.
// Reference op chain: models/fourier_nn.py:33-35,48-57 driven by
// problems/dist_online_dense_problem.py:117-127 (5 eager GEMMs + elementwise kernels per pass).
#include "common.cuh"
#include "mlp.h"
#include "sampler.cuh"
#include "umma.cuh"

namespace nndt {
namespace mlp {

using namespace umma;

constexpr int NT = 256;         // 8 warps: two warpgroups share the 128 TMEM lanes (32 columns each per pass)
constexpr int TILE = 128;
constexpr int HID = 64;
constexpr int MAX_DIN = 4;
constexpr int ACT_SLAB = TILE * kSlabRowBytes;   // 16 KB: 128 rows x 64 bf16
constexpr int W_SLAB = HID * kSlabRowBytes;      // 8 KB: 64 rows x 64 bf16

template <int H1>
struct FwdSmem {
  alignas(1024) uint8_t w1[(H1 / 64) * W_SLAB];
  alignas(1024) uint8_t w2[W_SLAB];
  alignas(1024) uint8_t w3[W_SLAB];
  alignas(1024) uint8_t h1[(H1 / 64) * ACT_SLAB];
  alignas(1024) uint8_t ha[ACT_SLAB];
  alignas(1024) uint8_t hb[ACT_SLAB];
  float w0[H1 * MAX_DIN];
  float b0[H1];
  float b1[HID], b2[HID], b3[HID], w4[HID];
  float b4;
  float xs[TILE * MAX_DIN];
  float part[TILE];
  alignas(8) uint64_t bar;
  uint32_t tmem_base;
};

// stage a [64 x K] fp32 weight matrix (row-major, K multiple of 64) as K/64 bf16 swizzled slabs
template <int TN>
NNDT_DEVINL void stage_weight(uint8_t* dst, const float* w, int K, int tid) {
  const int chunks = HID * (K / 8);            // 16-byte chunks
  for (int o = tid; o < chunks; o += TN) {
    const int n = o / (K / 8), c = o - n * (K / 8);
    const float4 lo = *reinterpret_cast<const float4*>(w + (size_t)n * K + 8 * c);
    const float4 hi = *reinterpret_cast<const float4*>(w + (size_t)n * K + 8 * c + 4);
    const float v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    const int slab = c >> 3, cc = c & 7;
    *reinterpret_cast<uint4*>(dst + slab * W_SLAB + swz_chunk_off(n, cc)) = pack_bf16x8(v);
  }
}

template <int H1, int TN, class S>
NNDT_DEVINL void stage_all_weights(S& sm, const Args& a, const float* th, int tid) {
  stage_weight<TN>(sm.w1, th + a.off[2], H1, tid);
  stage_weight<TN>(sm.w2, th + a.off[4], HID, tid);
  stage_weight<TN>(sm.w3, th + a.off[6], HID, tid);
  for (int o = tid; o < H1 * a.d_in; o += TN) sm.w0[o] = th[a.off[0] + o];
  for (int o = tid; o < H1; o += TN) sm.b0[o] = th[a.off[1] + o];
  if (tid < HID) {
    sm.b1[tid] = th[a.off[3] + tid];
    sm.b2[tid] = th[a.off[5] + tid];
    sm.b3[tid] = th[a.off[7] + tid];
    sm.w4[tid] = th[a.off[8] + tid];
  }
  if (tid == 0) sm.b4 = th[a.off[9]];
}

// first layer on CUDA cores: h1[r][f] = relu(sin(scale * z)) or relu(z), z = x[r] . W0[f] + b0[f]
template <int H1, int DIN, int TN, class S>
NNDT_DEVINL void first_layer(S& sm, const Args& a, int tid) {
  const int r = tid & (TILE - 1);
  const int half = tid >> 7;                       // TN/128 thread groups split the features
  float x[DIN];
#pragma unroll
  for (int d = 0; d < DIN; ++d) x[d] = sm.xs[r * MAX_DIN + d];
  constexpr int CH = H1 / 8 / (TN / TILE);         // 16-byte chunks per thread
  for (int c = 0; c < CH; ++c) {
    const int chunk = half * CH + c;               // global chunk index along the H1 features
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int f = chunk * 8 + e;
      float z = sm.b0[f];
#pragma unroll
      for (int d = 0; d < DIN; ++d) z = fmaf(x[d], sm.w0[f * DIN + d], z);
      if (a.first_act == kFirstSinRelu) z = __sinf(a.scale * z);
      v[e] = fmaxf(z, 0.f);
    }
    const int slab = chunk >> 3, cc = chunk & 7;
    *reinterpret_cast<uint4*>(sm.h1 + slab * ACT_SLAB + swz_chunk_off(r, cc)) = pack_bf16x8(v);
  }
}

// D[128 x 64] (+)= A[128 x K] . B[64 x K]^T, both K-major; issued by one thread
NNDT_DEVINL void gemm_kmajor(uint32_t tmem_d, const uint8_t* a_slabs, const uint8_t* b_slabs, int k_slabs,
                             bool accumulate_first) {
  constexpr uint32_t idesc = make_idesc(128, 64, false, false);
  const uint32_t a0 = smem_u32(a_slabs), b0 = smem_u32(b_slabs);
  for (int s = 0; s < k_slabs; ++s)
#pragma unroll
    for (int k = 0; k < 4; ++k)
      mma_bf16(tmem_d, desc_kmajor(a0 + s * ACT_SLAB, k), desc_kmajor(b0 + s * W_SLAB, k), idesc,
               accumulate_first || (s | k) != 0);
}

// epilogue of a 64-wide hidden layer: h = relu(acc + bias) -> bf16 slab; returns the fp32 values
NNDT_DEVINL void hidden_epilogue(uint32_t tmem_d, const float* bias, uint8_t* dst, int warp, int lane, float (&v)[32]) {
  const int row = (warp & 3) * 32 + lane;
  const int colhalf = warp >> 2;
  tmem_ld32(tmem_d + ((uint32_t)((warp & 3) * 32) << 16) + colhalf * 32, v);
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i] + bias[colhalf * 32 + i], 0.f);
  if (dst != nullptr) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
      *reinterpret_cast<uint4*>(dst + swz_chunk_off(row, colhalf * 4 + c)) = pack_bf16x8(v + 8 * c);
  }
}

template <int H1, int DIN>
__global__ void __launch_bounds__(NT, 1) mlp_forward_kernel(const Args a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  FwdSmem<H1>& sm = *reinterpret_cast<FwdSmem<H1>*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int l = blockIdx.y;
  const float* th = a.theta + (size_t)l * a.n_pad;

  if (warp == 0) tmem_alloc(&sm.tmem_base, 64);
  if (tid == 32) { mbar_init(&sm.bar, 1); mbar_init_fence(); }
  stage_all_weights<H1, NT>(sm, a, th, tid);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_d = sm.tmem_base;
  uint32_t phase = 0;

  const int ntiles = (a.n_rows + TILE - 1) / TILE;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int row0 = tile * TILE;
    for (int o = tid; o < TILE * a.d_in; o += NT) {
      const int r = o / a.d_in, d = o - r * a.d_in;
      sm.xs[r * MAX_DIN + d] = (row0 + r < a.n_rows) ? a.x[(size_t)(row0 + r) * a.d_in + d] : 0.f;
    }
    __syncthreads();
    first_layer<H1, DIN, NT>(sm, a, tid);
    fence_async_smem();
    __syncthreads();

    float v[32];
    // ---- layer 2: [128 x H1] . W1^T ------------------------------------------------------------
    if (tid == 0) { fence_after_sync(); gemm_kmajor(tmem_d, sm.h1, sm.w1, H1 / 64, false); commit(&sm.bar); }
    mbar_wait(&sm.bar, phase); phase ^= 1;
    fence_after_sync();
    hidden_epilogue(tmem_d, sm.b1, sm.ha, warp, lane, v);
    fence_before_sync(); fence_async_smem();
    __syncthreads();
    // ---- layer 3 --------------------------------------------------------------------------------
    if (tid == 0) { fence_after_sync(); gemm_kmajor(tmem_d, sm.ha, sm.w2, 1, false); commit(&sm.bar); }
    mbar_wait(&sm.bar, phase); phase ^= 1;
    fence_after_sync();
    hidden_epilogue(tmem_d, sm.b2, sm.hb, warp, lane, v);
    fence_before_sync(); fence_async_smem();
    __syncthreads();
    // ---- layer 4 + output layer -------------------------------------------------------------------
    if (tid == 0) { fence_after_sync(); gemm_kmajor(tmem_d, sm.hb, sm.w3, 1, false); commit(&sm.bar); }
    mbar_wait(&sm.bar, phase); phase ^= 1;
    fence_after_sync();
    hidden_epilogue(tmem_d, sm.b3, nullptr, warp, lane, v);
    fence_before_sync();
    const int colhalf = warp >> 2, row = (warp & 3) * 32 + lane;
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) dot = fmaf(v[i], sm.w4[colhalf * 32 + i], dot);
    if (colhalf == 1) sm.part[row] = dot;
    __syncthreads();
    if (colhalf == 0 && row0 + row < a.n_rows) {
      float z = dot + sm.part[row] + sm.b4;
      if (a.last_act == kLastSigmoid) z = 1.f / (1.f + __expf(-z));
      a.out[(size_t)l * a.n_rows + row0 + row] = z;
    }
    __syncthreads();
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_d, 64);
}

template <int H1>
static cudaError_t launch_forward_t(const Args& a, int ctas, cudaStream_t st) {
  const int smem = (int)sizeof(FwdSmem<H1>);
  static cudaError_t attr = cudaFuncSetAttribute(mlp_forward_kernel<H1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (attr != cudaSuccess) return attr;
  if (a.d_in != 2) return cudaErrorInvalidValue;
  mlp_forward_kernel<H1, 2><<<dim3(ctas, a.L), NT, smem, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_forward(const Args& a, int ctas_per_node, cudaStream_t st) {
  if (a.d_in > MAX_DIN) return cudaErrorInvalidValue;
  switch (a.h1) {
    case 64: return launch_forward_t<64>(a, ctas_per_node, st);
    case 128: return launch_forward_t<128>(a, ctas_per_node, st);
    case 256: return launch_forward_t<256>(a, ctas_per_node, st);
    default: return cudaErrorInvalidValue;
  }
}

// =====================================================================================
// Training: forward + backward of one minibatch per node, gradients to per-CTA partial rows.
//
// Backward GEMMs reuse the forward operand tiles through MN-major descriptors:
//   dH_{l-1}[128 x K_in] = dZ_l[128 x 64] (K-major A, K = out features) . W_l (MN-major B: N = in features,
//                          K = the 64 weight rows)
//   dW_l accumulators    = dZ_l^T . H_{l-1}: both operands MN-major with K = the 128 batch rows; fp32
//                          accumulation stays in TMEM across all tiles of a node and is flushed once.
//   bias / first-layer grads = dZ^T . [x, 1]: the same trick against a 16-column slab holding the tile's
//                          inputs and a ones column, so no cross-lane shuffle reductions are needed.
// TMEM map (columns): [0,128) scratch (forward D / dH) | [128,192) dW3 | [192,256) dW2 |
//   [256,384) dW1^T (2 blocks of 128 input features x 64) | [384,416) [dW0 | db0] (2 blocks x 16) |
//   [416,432) db3 | [432,448) db2 | [448,464) db1   (bias sums live in column DIN of their block)
// =====================================================================================
template <int H1>
struct TrainSmem {
  alignas(1024) uint8_t w1[(H1 / 64) * W_SLAB];
  alignas(1024) uint8_t w2[W_SLAB];
  alignas(1024) uint8_t w3[W_SLAB];
  alignas(1024) uint8_t h1[(H1 < 128 ? 2 : H1 / 64) * ACT_SLAB];   // h1, later dZ1 (>= 2 slabs: M = 128 A operand)
  alignas(1024) uint8_t dz[ACT_SLAB];       // dZ of the layer being back-propagated (the slab after it is the
  alignas(1024) uint8_t h2[ACT_SLAB];       //  don't-care second M atom of the dW GEMMs)
  alignas(1024) uint8_t h3[ACT_SLAB];
  alignas(1024) uint8_t xa[ACT_SLAB];       // [x_0..x_{DIN-1}, 1, 0...] per row, 16 valid columns
  float w0[H1 * MAX_DIN];
  float b0[H1];
  float b1[HID], b2[HID], b3[HID], w4[HID];
  float b4;
  float g_w4[HID];
  float g_b4;
  float loss_acc;
  float xs[TILE * MAX_DIN];
  float ys[TILE];
  float part[4 * TILE];
  float dz5[TILE];
  int ridx[TILE];
  alignas(8) uint64_t bar;
  uint32_t tmem_base;
};

// column sums over the 32 lanes of a warp of 32 per-lane values: 31 shuffles; lane j returns column j
NNDT_DEVINL float colsum32(float (&v)[32], int lane) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    const bool hi = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < o; ++i) {
      const float send = hi ? v[i] : v[i + o];
      const float keep = hi ? v[i + o] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  return v[0];
}

// dH[128 x N] = dZ[128 x 64] . W  (A K-major; B MN-major: N/64 atoms W_SLAB apart starting at `w`)
template <int N>
NNDT_DEVINL void gemm_dh(uint32_t tmem_d, const uint8_t* dz, const uint8_t* w) {
  constexpr uint32_t idesc = make_idesc(128, N, false, true);
  const uint32_t a0 = smem_u32(dz), b0 = smem_u32(w);
#pragma unroll
  for (int k = 0; k < 4; ++k)
    mma_bf16(tmem_d, desc_kmajor(a0, k), desc_mnmajor(b0, k, W_SLAB), idesc, k != 0);
}
// acc[128 x N] (+)= A^T . B over the 128 tile rows; A, B MN-major slabs (A: 2 atoms ACT_SLAB apart)
template <int N>
NNDT_DEVINL void gemm_dw(uint32_t tmem_d, const uint8_t* a_slab, const uint8_t* b_slab, bool accumulate) {
  constexpr uint32_t idesc = make_idesc(128, N, true, true);
  const uint32_t a0 = smem_u32(a_slab), b0 = smem_u32(b_slab);
#pragma unroll
  for (int k = 0; k < 8; ++k)
    mma_bf16(tmem_d, desc_mnmajor(a0, k, ACT_SLAB), desc_mnmajor(b0, k, ACT_SLAB), idesc, accumulate || k != 0);
}

constexpr int NTT = 512;       // training CTA: 16 warps = 4 TMEM lane quarters x 4 column groups of 16

// column sums over the 32 lanes of a warp of 16 per-lane values: lane j (and j+16) returns column j
NNDT_DEVINL float colsum16(float (&v)[16], int lane) {
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], 16);
#pragma unroll
  for (int o = 8; o >= 1; o >>= 1) {
    const bool hi = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < o; ++i) {
      const float send = hi ? v[i] : v[i + o];
      const float keep = hi ? v[i + o] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  return v[0];
}

// hidden-layer epilogue for a 16-column slice: h = relu(acc + bias) -> two 16-byte chunks of the bf16 slab
NNDT_DEVINL void hidden_epilogue16(uint32_t tmem_d, uint32_t lane_addr, int cg, int row, const float* bias, uint8_t* dst,
                                   float (&v)[16]) {
  tmem_ld16(tmem_d + lane_addr + cg * 16, v);
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i] + bias[cg * 16 + i], 0.f);
  if (dst != nullptr) {
#pragma unroll
    for (int c = 0; c < 2; ++c)
      *reinterpret_cast<uint4*>(dst + swz_chunk_off(row, cg * 2 + c)) = pack_bf16x8(v + 8 * c);
  }
}

template <int H1, int DIN>
__global__ void __launch_bounds__(NTT, 1) mlp_train_kernel(const Args a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  TrainSmem<H1>& sm = *reinterpret_cast<TrainSmem<H1>*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cg = warp >> 2, row = (warp & 3) * 32 + lane;      // column group 0..3, batch row of the tile
  const uint32_t lane_addr = (uint32_t)((warp & 3) * 32) << 16;
  constexpr int NBLK1 = (H1 + 127) / 128;       // 128-feature blocks of the first hidden layer
  constexpr int NH = H1 > 128 ? 128 : H1;        // dH1 is produced NH columns at a time

  if (warp == 0) tmem_alloc(&sm.tmem_base, 512);
  if (tid == 32) { mbar_init(&sm.bar, 1); mbar_init_fence(); }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tm = sm.tmem_base;
  const uint32_t T_SCR = tm, T_DW3 = tm + 128, T_DW2 = tm + 192, T_DW1 = tm + 256, T_DW0 = tm + 384,
                 T_B3 = tm + 416, T_B2 = tm + 432, T_B1 = tm + 448;
  uint32_t phase = 0;
  bool pending = false;        // MMAs of the previous tile still in flight (committed, not yet waited)

  // ---- static work partition: items (node, tile) in node-major order -------------------------
  const int Tmax = (a.batch + TILE - 1) / TILE;
  const int I = a.L * Tmax, G = gridDim.x, c = blockIdx.x;
  const int it0 = (int)(((long long)c * I) / G), it1 = (int)(((long long)(c + 1) * I) / G);

  int cur = -1;          // node whose weights / accumulators are live
  bool have_acc = false;
  uint32_t bs = 0, start = 0, key = 0, m = 0;
  int shard_off = 0;
  long long first_draw = 0;            // online sliding-window mode: index of the batch's first draw
  const long long* wt = nullptr;       // [K, P, cum[0..KMAX], lb[KMAX], ub[KMAX]] of the current node

  for (int it = it0; it <= it1; ++it) {
    const int l = (it < it1) ? it / Tmax : -1;
    if (l != cur) {
      if (pending) { mbar_wait(&sm.bar, phase); phase ^= 1; pending = false; }
      // ---------------- flush the finished node segment ---------------------------------------
      if (cur >= 0) {
        const long long first_item = (long long)cur * Tmax;
        int cf = (int)((first_item * G) / I);
        while ((long long)(cf + 1) * I / G <= first_item) ++cf;
        while ((long long)cf * I / G > first_item) --cf;
        const int slot = c - cf;       // this CTA's slot among the CTAs that cover node `cur`
        float* gp = a.grad_part + ((size_t)cur * a.S + slot) * a.n_pad;
        fence_after_sync();
        float w[16];
        // dW3, dW2: lanes 0..63 = output feature n, columns = input feature k
        for (int q = 0; q < 2; ++q) {
          tmem_ld16((q == 0 ? T_DW3 : T_DW2) + lane_addr + cg * 16, w);
          if (row < HID) {
            float4* dst = reinterpret_cast<float4*>(gp + (q == 0 ? a.off[6] : a.off[4]) + row * HID + cg * 16);
#pragma unroll
            for (int i = 0; i < 4; ++i)
              dst[i] = have_acc ? make_float4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
        // dW1^T blocks: lane = input feature k (within the 128-block), column = output feature n
        for (int blk = 0; blk < NBLK1; ++blk) {
          tmem_ld16(T_DW1 + blk * 64 + lane_addr + cg * 16, w);
          const int k = blk * 128 + row;
          if (k < H1) {
#pragma unroll
            for (int i = 0; i < 16; ++i) gp[a.off[2] + (cg * 16 + i) * H1 + k] = have_acc ? w[i] : 0.f;
          }
        }
        // 16-column blocks: [dW0 | db0] (lane = first-layer feature) and the hidden bias sums (lane = feature)
        if (cg == 0) {
          for (int blk = 0; blk < NBLK1; ++blk) {
            tmem_ld16(T_DW0 + blk * 16 + lane_addr, w);
            const int f = blk * 128 + row;
            if (f < H1) {
#pragma unroll
              for (int d = 0; d < DIN; ++d) gp[a.off[0] + f * DIN + d] = have_acc ? w[d] : 0.f;
              gp[a.off[1] + f] = have_acc ? w[DIN] : 0.f;
            }
          }
          for (int q = 0; q < 3; ++q) {
            tmem_ld16((q == 0 ? T_B3 : q == 1 ? T_B2 : T_B1) + lane_addr, w);
            if (row < HID) gp[a.off[q == 0 ? 7 : q == 1 ? 5 : 3] + row] = have_acc ? w[DIN] : 0.f;
          }
        }
        fence_before_sync();
        if (tid < HID) gp[a.off[8] + tid] = sm.g_w4[tid];
        if (tid == 0) { gp[a.off[9]] = sm.g_b4; a.loss_part[cur * a.S + slot] = sm.loss_acc; }
        __syncthreads();
      }
      if (l < 0) break;
      // ---------------- set up the next node ----------------------------------------------------
      cur = l;
      have_acc = false;
      const float* th = a.theta + (size_t)l * a.n_pad;
      stage_all_weights<H1, NTT>(sm, a, th, tid);
      if (tid < HID) sm.g_w4[tid] = 0.f;
      if (tid == 0) { sm.g_b4 = 0.f; sm.loss_acc = 0.f; }
      if (a.direct) {
        bs = (uint32_t)a.batch;
      } else {
        m = (uint32_t)a.shard_len[l];
        shard_off = a.shard_off[l];
        const BatchLoc loc = locate_batch((uint32_t)a.calls[l], m, (uint32_t)a.batch);
        bs = loc.size; start = loc.start;
        key = mix_key((uint32_t)a.seed, (uint32_t)(a.node0 + l), loc.epoch);
        if (a.win_table != nullptr) {
          wt = reinterpret_cast<const long long*>(a.win_table) + (size_t)l * kWinTableLen;
          first_draw = (long long)loc.epoch * m + loc.start;
        }
      }
      fence_async_smem();
      __syncthreads();
    }
    const int tile = it - l * Tmax;
    const uint32_t t0 = (uint32_t)tile * TILE;
    if (t0 >= bs) continue;                              // partial batch: nothing in this tile
    const float inv_bs = 1.f / (float)bs;

    // ---- gather the tile's rows (overlaps the previous tile's last MMAs) ---------------------------
    int my_idx = -1;
    float my_x[DIN];
    float my_y = 0.f;
    if (tid < TILE) {
      const uint32_t t = t0 + tid;
      if (t < bs) {
        if (a.direct) {
          my_idx = (int)(l * a.batch + t);
        } else if (wt != nullptr) {
          my_idx = shard_off + window_draw(wt, first_draw + t, (uint32_t)a.seed, (uint32_t)(a.node0 + l));
        } else {
          my_idx = shard_off + (int)feistel_permute(start + t, m, key);
        }
      }
#pragma unroll
      for (int d = 0; d < DIN; ++d) my_x[d] = my_idx >= 0 ? a.x[(size_t)my_idx * DIN + d] : 0.f;
      my_y = my_idx >= 0 ? a.y[my_idx] : 0.f;
    }
    if (pending) { mbar_wait(&sm.bar, phase); phase ^= 1; pending = false; }   // xa / h1 are free again
    if (tid < TILE) {
      sm.ridx[tid] = my_idx;
      sm.ys[tid] = my_y;
      float xv[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) xv[e] = 0.f;
#pragma unroll
      for (int d = 0; d < DIN; ++d) { sm.xs[tid * MAX_DIN + d] = my_x[d]; xv[d] = my_x[d]; }
      xv[DIN] = my_idx >= 0 ? 1.f : 0.f;
      *reinterpret_cast<uint4*>(sm.xa + swz_chunk_off(tid, 0)) = pack_bf16x8(xv);
      *reinterpret_cast<uint4*>(sm.xa + swz_chunk_off(tid, 1)) = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    first_layer<H1, DIN, NTT>(sm, a, tid);
    fence_async_smem();
    __syncthreads();

    float v[16];
    // ======================= forward ===============================================================
    if (warp == 0 && lane == 0) { fence_after_sync(); gemm_kmajor(T_SCR, sm.h1, sm.w1, H1 / 64, false); commit(&sm.bar); }
    mbar_wait(&sm.bar, phase); phase ^= 1;
    fence_after_sync();
    hidden_epilogue16(T_SCR, lane_addr, cg, row, sm.b1, sm.h2, v);
    fence_before_sync(); fence_async_smem();
    __syncthreads();
    if (warp == 0 && lane == 0) { fence_after_sync(); gemm_kmajor(T_SCR, sm.h2, sm.w2, 1, false); commit(&sm.bar); }
    mbar_wait(&sm.bar, phase); phase ^= 1;
    fence_after_sync();
    hidden_epilogue16(T_SCR, lane_addr, cg, row, sm.b2, sm.h3, v);
    fence_before_sync(); fence_async_smem();
    __syncthreads();
    if (warp == 0 && lane == 0) { fence_after_sync(); gemm_kmajor(T_SCR, sm.h3, sm.w3, 1, false); commit(&sm.bar); }
    mbar_wait(&sm.bar, phase); phase ^= 1;
    fence_after_sync();
    hidden_epilogue16(T_SCR, lane_addr, cg, row, sm.b3, nullptr, v);     // v = h4[row][cg*16 ..]
    fence_before_sync();
    // ---- output layer, loss, dL/dz5 --------------------------------------------------------------------
    {
      float dot = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) dot = fmaf(v[i], sm.w4[cg * 16 + i], dot);
      sm.part[cg * TILE + row] = dot;
      __syncthreads();
      if (cg == 0) {
        const bool valid = sm.ridx[row] >= 0;
        const float z = sm.part[row] + sm.part[TILE + row] + sm.part[2 * TILE + row] + sm.part[3 * TILE + row] + sm.b4;
        const float y = sm.ys[row];
        float p = z, dpdz = 1.f;
        if (a.last_act == kLastSigmoid) { p = 1.f / (1.f + __expf(-z)); dpdz = p * (1.f - p); }
        float loss, g;
        if (a.loss == kLossBCE) {
          loss = -(y * fmaxf(__logf(p), -100.f) + (1.f - y) * fmaxf(__logf(1.f - p), -100.f));
          g = (a.last_act == kLastSigmoid) ? (p - y) : (p - y) / fmaxf(p * (1.f - p), 1e-12f);
        } else if (a.loss == kLossMSE) {
          loss = (p - y) * (p - y); g = 2.f * (p - y) * dpdz;
        } else {
          loss = fabsf(p - y); g = (p > y ? 1.f : (p < y ? -1.f : 0.f)) * dpdz;
        }
        sm.dz5[row] = valid ? g * inv_bs : 0.f;
        const float lsum = warp_sum(valid ? loss * inv_bs : 0.f);
        const float gsum = warp_sum(valid ? g * inv_bs : 0.f);
        if (lane == 0) { atomicAdd(&sm.loss_acc, lsum); atomicAdd(&sm.g_b4, gsum); }
      }
      __syncthreads();
    }
    // ======================= backward ================================================================
    {
      // layer 5 -> dz4 = dz5 * w4 * relu'(h4);  dW4 += dz5 * h4 (the one remaining shuffle reduction)
      const float d5 = sm.dz5[row];
      float t1[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        t1[i] = d5 * v[i];
        v[i] = v[i] > 0.f ? d5 * sm.w4[cg * 16 + i] : 0.f;
      }
#pragma unroll
      for (int cch = 0; cch < 2; ++cch)
        *reinterpret_cast<uint4*>(sm.dz + swz_chunk_off(row, cg * 2 + cch)) = pack_bf16x8(v + 8 * cch);
      const float s4 = colsum16(t1, lane);
      if (lane < 16) atomicAdd(&sm.g_w4[cg * 16 + lane], s4);
    }
    fence_async_smem();
    __syncthreads();
    // dh3 = dz4 . W3 ; dW3 += dz4^T . h3 ; db3 += dz4^T . [x,1]
    if (warp == 0 && lane == 0) {
      fence_after_sync();
      gemm_dh<64>(T_SCR, sm.dz, sm.w3);
      gemm_dw<64>(T_DW3, sm.dz, sm.h3, have_acc);
      gemm_dw<16>(T_B3, sm.dz, sm.xa, have_acc);
      commit(&sm.bar);
    }
    mbar_wait(&sm.bar, phase); phase ^= 1;
    fence_after_sync();
#pragma unroll 1
    for (int layer = 3; layer >= 2; --layer) {
      // dz_{layer} = dh_{layer} * relu'(h_{layer})
      const uint8_t* hs = layer == 3 ? sm.h3 : sm.h2;
      tmem_ld16(T_SCR + lane_addr + cg * 16, v);
      fence_before_sync();
#pragma unroll
      for (int cch = 0; cch < 2; ++cch) {
        const uint4 hv = *reinterpret_cast<const uint4*>(hs + swz_chunk_off(row, cg * 2 + cch));
        const __nv_bfloat16* hb = reinterpret_cast<const __nv_bfloat16*>(&hv);
#pragma unroll
        for (int e = 0; e < 8; ++e) v[cch * 8 + e] = __bfloat162float(hb[e]) > 0.f ? v[cch * 8 + e] : 0.f;
      }
#pragma unroll
      for (int cch = 0; cch < 2; ++cch)
        *reinterpret_cast<uint4*>(sm.dz + swz_chunk_off(row, cg * 2 + cch)) = pack_bf16x8(v + 8 * cch);
      fence_async_smem();
      __syncthreads();
      if (warp == 0 && lane == 0) {
        fence_after_sync();
        if (layer == 3) {
          gemm_dh<64>(T_SCR, sm.dz, sm.w2);
          gemm_dw<64>(T_DW2, sm.dz, sm.h2, have_acc);
          gemm_dw<16>(T_B2, sm.dz, sm.xa, have_acc);
        } else {
          gemm_dh<NH>(T_SCR, sm.dz, sm.w1);
          // dW1^T[k][n] = h1^T . dz2 : A = h1 (M = 128 input features per MMA), B = dz2
          for (int blk = 0; blk < NBLK1; ++blk)
            gemm_dw<64>(T_DW1 + blk * 64, sm.h1 + blk * 2 * ACT_SLAB, sm.dz, have_acc);
          gemm_dw<16>(T_B1, sm.dz, sm.xa, have_acc);
        }
        commit(&sm.bar);
      }
      mbar_wait(&sm.bar, phase); phase ^= 1;
      fence_after_sync();
    }
    // ---- first layer: dz1 = dh1 * act'(z1) -> bf16 slabs over the dead h1 tile;  [dW0|db0] += dz1^T [x,1] ----
    {
      float x[DIN];
#pragma unroll
      for (int d = 0; d < DIN; ++d) x[d] = sm.xs[row * MAX_DIN + d];
      constexpr int CPT = NH / 4;              // columns per thread per half (4 column groups)
#pragma unroll 1
      for (int half = 0; half < (H1 + NH - 1) / NH; ++half) {
        if (half > 0) {
          fence_before_sync();
          __syncthreads();
          if (warp == 0 && lane == 0) {
            fence_after_sync(); gemm_dh<NH>(T_SCR, sm.dz, sm.w1 + half * (NH / 64) * W_SLAB); commit(&sm.bar);
          }
          mbar_wait(&sm.bar, phase); phase ^= 1;
          fence_after_sync();
        }
#pragma unroll 1
        for (int q = 0; q < CPT / 16; ++q) {
          const int col = cg * CPT + q * 16;           // column inside the NH-wide scratch
          const int f0 = half * NH + col;              // first-layer feature of v[0]
          tmem_ld16(T_SCR + lane_addr + col, v);
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int f = f0 + i;
            float z = sm.b0[f];
#pragma unroll
            for (int d = 0; d < DIN; ++d) z = fmaf(x[d], sm.w0[f * DIN + d], z);
            float dact;
            if (a.first_act == kFirstSinRelu) {
              float sn, cs;
              __sincosf(a.scale * z, &sn, &cs);
              dact = sn > 0.f ? cs * a.scale : 0.f;
            } else {
              dact = z > 0.f ? 1.f : 0.f;
            }
            v[i] *= dact;
          }
          const int chunk0 = (f0 & 63) >> 3;
          uint8_t* slab = sm.h1 + (f0 >> 6) * ACT_SLAB;
#pragma unroll
          for (int cch = 0; cch < 2; ++cch)
            *reinterpret_cast<uint4*>(slab + swz_chunk_off(row, chunk0 + cch)) = pack_bf16x8(v + 8 * cch);
        }
      }
      fence_before_sync();
      fence_async_smem();
      __syncthreads();
      if (warp == 0 && lane == 0) {
        fence_after_sync();
        for (int blk = 0; blk < NBLK1; ++blk)
          gemm_dw<16>(T_DW0 + blk * 16, sm.h1 + blk * 2 * ACT_SLAB, sm.xa, have_acc);
        commit(&sm.bar);
      }
      pending = true;      // waited for at the top of the next tile / before the flush
    }
    have_acc = true;
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tm, 512);
}

template <int H1>
static cudaError_t launch_train_t(const Args& a, int ctas, cudaStream_t st) {
  const int smem = (int)sizeof(TrainSmem<H1>);
  static cudaError_t attr = cudaFuncSetAttribute(mlp_train_kernel<H1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (attr != cudaSuccess) return attr;
  if (a.d_in != 2) return cudaErrorInvalidValue;
  mlp_train_kernel<H1, 2><<<dim3(ctas), NTT, smem, st>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_train(const Args& a, int ctas, cudaStream_t st) {
  if (a.d_in > MAX_DIN) return cudaErrorInvalidValue;
  switch (a.h1) {
    case 64: return launch_train_t<64>(a, ctas, st);
    case 128: return launch_train_t<128>(a, ctas, st);
    case 256: return launch_train_t<256>(a, ctas, st);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace mlp
}  // namespace nndt
