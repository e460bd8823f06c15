// fp64 CUDA-core implementation of the implicit-density MLPs (FourierNet and ReLU nets), the float64 arm of
// mlp_tc.cu: same network family, same launch contract (one launch for all local nodes, rows read from the
// arena through the slot offsets, minibatches drawn in the kernel by the stateless samplers of sampler.cuh),
// all arithmetic in double.
//
// A CTA processes tiles of R = 64 batch rows with 256 threads; thread (tr, tc) = (tid / 16, tid % 16) owns the
// outputs at rows tr + 16 i and columns tc + 16 j of every 64-row contraction (DFMA register tiles, operands in
// shared memory with odd row strides, so neither operand read has a bank conflict).  The first hidden layer is
// never stored whole: its 256 features are produced 32 at a time straight from x (2 MACs + one sin each), and
// each chunk is contracted against the matching 32 columns of W1, which are staged from L2.  The backward pass
// recomputes the chunk.
//
// Training: CTA (s, l) handles tiles s, s + S, ... of node l's minibatch and owns grad_part[l, s] and
// loss_part[l, s]; every gradient element is accumulated by one fixed thread in tile order, and every cross-thread
// sum runs in a fixed order, so two launches on the same inputs give bitwise-equal partials.
//
// The loss chain follows ATen's float64 kernels rather than the fused sigmoid-BCE form `p - y`: BCE clamps the
// logs at -100 and divides dL/dp by max(p (1 - p), 1e-12), then the sigmoid backward multiplies by (1 - p) p.
// The two differ once p (1 - p) < 1e-12 (|z| > 27.6).
#include "common.cuh"
#include "mlp.h"
#include "sampler.cuh"

namespace nndt {
namespace mlp {
namespace {

constexpr int NT = 256;
constexpr int R = 64;          // batch rows per tile
constexpr int HID = 64;
constexpr int KC = 32;         // first-layer features per chunk
constexpr int MAX_DIN = 4;
constexpr int MAX_H1 = 256;
constexpr int LD = HID + 1;    // row stride of the 64-wide shared matrices
constexpr int LDC = KC + 1;    // row stride of the 32-wide chunk matrices

struct Smem {
  double h2[R * LD], h3[R * LD], h4[R * LD];   // activations [r][k]; the backward pass overwrites them with dz2..dz4
  double w[HID * LD];                          // W2 or W3 [n][k], or a W1 chunk [n][kc] (stride LDC)
  double h1[R * LDC];                          // first-layer chunk [r][kc]
  double red[2][16 * HID];                     // per-thread-row partial sums, reduced in a fixed order
  double w0[MAX_H1 * MAX_DIN], b0[MAX_H1];
  double b1[HID], b2[HID], b3[HID], w4[HID];
  double b4;
  double xs[R * MAX_DIN];
  double ys[R];
  double dz5[R];
  double lrow[R];
  int valid[R];
};

// acc[i][j] += sum_k A(tr + 16 i, k) B(k, tc + 16 j) with A(m, k) = A[m * ar + k * ak], B(k, n) = B[k * bk + n * bn]
template <int MI, int MJ, int K>
NNDT_DEVINL void mm(double (&acc)[MI][MJ], const double* A, int ar, int ak, const double* B, int bk, int bn, int tr, int tc) {
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    double av[MI], bv[MJ];
#pragma unroll
    for (int i = 0; i < MI; ++i) av[i] = A[(tr + 16 * i) * ar + k * ak];
#pragma unroll
    for (int j = 0; j < MJ; ++j) bv[j] = B[k * bk + (tc + 16 * j) * bn];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
      for (int j = 0; j < MJ; ++j) acc[i][j] = fma(av[i], bv[j], acc[i][j]);
  }
}

template <int MI, int MJ>
NNDT_DEVINL void zero(double (&acc)[MI][MJ]) {
#pragma unroll
  for (int i = 0; i < MI; ++i)
#pragma unroll
    for (int j = 0; j < MJ; ++j) acc[i][j] = 0.0;
}

// stage a [64 x 64] weight matrix (row-major in theta) as [n][k] with stride LD
NNDT_DEVINL void stage_w64(double* dst, const double* w, int tid) {
  for (int o = tid; o < HID * HID; o += NT) dst[(o >> 6) * LD + (o & 63)] = w[o];
}

// stage columns [c * KC, c * KC + KC) of W1 [64 x H1] as [n][kc] with stride LDC
template <int H1>
NNDT_DEVINL void stage_w1_chunk(double* dst, const double* w1, int c, int tid) {
  for (int o = tid; o < HID * KC; o += NT) {
    const int n = o / KC, kc = o - n * KC;
    dst[n * LDC + kc] = w1[n * H1 + c * KC + kc];
  }
}

template <int DIN>
NNDT_DEVINL double z1(const Smem& sm, int r, int f) {
  double z = sm.b0[f];
#pragma unroll
  for (int d = 0; d < DIN; ++d) z = fma(sm.xs[r * MAX_DIN + d], sm.w0[f * DIN + d], z);
  return z;
}

// first-layer chunk c: h1[r][kc] = relu(sin(scale * z)) or relu(z), z = x[r] . W0[f] + b0[f], f = c * KC + kc
template <int DIN>
NNDT_DEVINL void first_layer_chunk(Smem& sm, const ArgsF64& a, int c, int tid) {
  for (int o = tid; o < R * KC; o += NT) {
    const int r = o / KC, kc = o - r * KC;
    double z = z1<DIN>(sm, r, c * KC + kc);
    if (a.first_act == kFirstSinRelu) z = sin(a.scale * z);
    sm.h1[r * LDC + kc] = fmax(z, 0.0);
  }
}

// h_out[r][n] = relu(acc + b[n]) for the thread's micro-tile
NNDT_DEVINL void store_relu(double* h, const double (&acc)[4][4], const double* b, int tr, int tc) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) h[(tr + 16 * i) * LD + tc + 16 * j] = fmax(acc[i][j] + b[tc + 16 * j], 0.0);
}

// Forward pass of the tile whose inputs are in sm.xs.  Leaves h2, h3, h4 in shared memory and W3 in sm.w; returns
// the output-layer pre-activation z5 of row tid / 4 (identical in the 4 threads of the row).
template <int H1, int DIN>
NNDT_DEVINL double forward_tile(Smem& sm, const ArgsF64& a, const double* th, int tid) {
  const int tr = tid >> 4, tc = tid & 15;
  double acc[4][4];
  zero(acc);
#pragma unroll 1
  for (int c = 0; c < H1 / KC; ++c) {
    __syncthreads();                                  // previous chunk consumed; xs written
    stage_w1_chunk<H1>(sm.w, th + a.off[2], c, tid);
    first_layer_chunk<DIN>(sm, a, c, tid);
    __syncthreads();
    mm<4, 4, KC>(acc, sm.h1, LDC, 1, sm.w, 1, LDC, tr, tc);
  }
  store_relu(sm.h2, acc, sm.b1, tr, tc);
  __syncthreads();
  stage_w64(sm.w, th + a.off[4], tid);
  __syncthreads();
  zero(acc);
  mm<4, 4, HID>(acc, sm.h2, LD, 1, sm.w, 1, LD, tr, tc);
  store_relu(sm.h3, acc, sm.b2, tr, tc);
  __syncthreads();
  stage_w64(sm.w, th + a.off[6], tid);
  __syncthreads();
  zero(acc);
  mm<4, 4, HID>(acc, sm.h3, LD, 1, sm.w, 1, LD, tr, tc);
  store_relu(sm.h4, acc, sm.b3, tr, tc);
  __syncthreads();
  // output layer: 4 threads per row, interleaved features, fixed butterfly
  const int r = tid >> 2, q = tid & 3;
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < HID / 4; ++i) s = fma(sm.h4[r * LD + q + 4 * i], sm.w4[q + 4 * i], s);
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  return s + sm.b4;
}

NNDT_DEVINL void stage_small(Smem& sm, const ArgsF64& a, const double* th, int tid) {
  for (int o = tid; o < a.h1 * a.d_in; o += NT) sm.w0[o] = th[a.off[0] + o];
  for (int o = tid; o < a.h1; o += NT) sm.b0[o] = th[a.off[1] + o];
  if (tid < HID) {
    sm.b1[tid] = th[a.off[3] + tid];
    sm.b2[tid] = th[a.off[5] + tid];
    sm.b3[tid] = th[a.off[7] + tid];
    sm.w4[tid] = th[a.off[8] + tid];
  }
  if (tid == 0) sm.b4 = th[a.off[9]];
}

template <int H1, int DIN>
__global__ void __launch_bounds__(NT, 1) mlp_f64_forward_kernel(const ArgsF64 a) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  const int tid = threadIdx.x, l = blockIdx.y;
  const double* th = a.theta + (size_t)l * a.n_pad;
  stage_small(sm, a, th, tid);
  const int ntiles = (a.n_rows + R - 1) / R;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int row0 = tile * R;
    __syncthreads();                                  // the previous tile's h4 reads are done
    for (int o = tid; o < R * DIN; o += NT) {
      const int r = o / DIN, d = o - r * DIN;
      sm.xs[r * MAX_DIN + d] = (row0 + r < a.n_rows) ? a.x[(size_t)(row0 + r) * DIN + d] : 0.0;
    }
    const double z = forward_tile<H1, DIN>(sm, a, th, tid);
    const int r = tid >> 2;
    if ((tid & 3) == 0 && row0 + r < a.n_rows)
      a.out[(size_t)l * a.n_rows + row0 + r] = a.last_act == kLastSigmoid ? 1.0 / (1.0 + exp(-z)) : z;
  }
}

// column sums over the 64 tile rows of per-thread values v[i][j] (row tr + 16 i, column tc + 16 j): partials to red,
// reduced after the caller's __syncthreads by colsum_finish
NNDT_DEVINL void colsum_part(double* red, const double (&v)[4][4], int tr, int tc) {
#pragma unroll
  for (int j = 0; j < 4; ++j) red[tr * HID + tc + 16 * j] = ((v[0][j] + v[1][j]) + v[2][j]) + v[3][j];
}
NNDT_DEVINL double colsum_finish(const double* red, int col) {
  double s = 0.0;
#pragma unroll
  for (int t = 0; t < 16; ++t) s += red[t * HID + col];
  return s;
}

// grad[n][k] += acc (64 x 64 weight gradient of the thread's micro-tile)
NNDT_DEVINL void add_w64(double* g, const double (&acc)[4][4], int tr, int tc) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) g[(tr + 16 * i) * HID + tc + 16 * j] += acc[i][j];
}

// hidden layer backward: dh = dz . W (W in sm.w), dW += dz^T . h_in; then dz_in = dh * relu'(h_in) overwrites
// h_in, and the bias gradient of the layer below (column sums of dz_in) is added to gb_in
NNDT_DEVINL void hidden_backward(Smem& sm, const double* dz, double* h_in, double* gw, double* gb_in, const double* w_next,
                                 int tid) {
  const int tr = tid >> 4, tc = tid & 15;
  double dh[4][4], dw[4][4];
  zero(dh); zero(dw);
  mm<4, 4, HID>(dh, dz, LD, 1, sm.w, LD, 1, tr, tc);
  mm<4, 4, HID>(dw, dz, 1, LD, h_in, LD, 1, tr, tc);
  add_w64(gw, dw, tr, tc);
  __syncthreads();                                    // sm.w and h_in are read by every thread above
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      double& h = h_in[(tr + 16 * i) * LD + tc + 16 * j];
      dh[i][j] = h > 0.0 ? dh[i][j] : 0.0;
      h = dh[i][j];
    }
  colsum_part(sm.red[0], dh, tr, tc);
  if (w_next != nullptr) stage_w64(sm.w, w_next, tid);
  __syncthreads();
  if (tid < HID) gb_in[tid] += colsum_finish(sm.red[0], tid);
}

template <int H1, int DIN>
__global__ void __launch_bounds__(NT, 1) mlp_f64_train_kernel(const ArgsF64 a) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  const int tid = threadIdx.x, tr = tid >> 4, tc = tid & 15;
  const int s = blockIdx.x, l = blockIdx.y;
  const double* th = a.theta + (size_t)l * a.n_pad;
  double* gp = a.grad_part + ((size_t)l * a.S + s) * a.n_pad;
  for (int o = tid; o < a.n_pad; o += NT) gp[o] = 0.0;
  stage_small(sm, a, th, tid);

  const uint32_t m = (uint32_t)a.shard_len[l];
  const int shard_off = a.shard_off[l];
  const BatchLoc loc = locate_batch((uint32_t)a.calls[l], m, (uint32_t)a.batch);
  const uint32_t bs = loc.size;
  const uint32_t key = mix_key((uint32_t)a.seed, (uint32_t)(a.node0 + l), loc.epoch);
  const long long* wt = a.win_table == nullptr ? nullptr
                        : reinterpret_cast<const long long*>(a.win_table) + (size_t)l * kWinTableLen;
  const long long first_draw = (long long)loc.epoch * m + loc.start;
  const double inv_bs = 1.0 / (double)bs;
  double loss_sum = 0.0, gb4 = 0.0;             // thread 0
  const int ntiles = (int)((bs + R - 1) / R);

#pragma unroll 1
  for (int tile = s; tile < ntiles; tile += a.S) {
    const uint32_t t0 = (uint32_t)tile * R;
    __syncthreads();                                  // previous tile done with xs / ys / valid; gp zeroed
    if (tid < R) {
      const uint32_t t = t0 + tid;
      int idx = -1;
      if (t < bs)
        idx = shard_off + (wt != nullptr ? window_draw(wt, first_draw + t, (uint32_t)a.seed, (uint32_t)(a.node0 + l))
                                         : (int)feistel_permute(loc.start + t, m, key));
#pragma unroll
      for (int d = 0; d < DIN; ++d) sm.xs[tid * MAX_DIN + d] = idx >= 0 ? a.x[(size_t)idx * DIN + d] : 0.0;
      sm.ys[tid] = idx >= 0 ? a.y[idx] : 0.0;
      sm.valid[tid] = idx >= 0;
    }
    const double z = forward_tile<H1, DIN>(sm, a, th, tid);

    // ---- output activation, loss and dL/dz5 (ATen's float64 chain) ------------------------------------------------
    if ((tid & 3) == 0) {
      const int r = tid >> 2;
      const double y = sm.ys[r];
      const double p = a.last_act == kLastSigmoid ? 1.0 / (1.0 + exp(-z)) : z;
      double loss, g;
      if (a.loss == kLossBCE) {
        loss = (y - 1.0) * fmax(log1p(-p), -100.0) - y * fmax(log(p), -100.0);
        g = (inv_bs * (p - y)) / fmax((1.0 - p) * p, 1e-12);
      } else if (a.loss == kLossMSE) {
        loss = (p - y) * (p - y);
        g = (2.0 * inv_bs) * (p - y);
      } else {
        loss = fabs(p - y);
        g = (p > y ? 1.0 : (p < y ? -1.0 : 0.0)) * inv_bs;
      }
      if (a.last_act == kLastSigmoid) g = (g * (1.0 - p)) * p;
      const bool v = sm.valid[r] != 0;
      sm.dz5[r] = v ? g : 0.0;
      sm.lrow[r] = v ? loss : 0.0;
    }
    __syncthreads();
    if (tid < 32) {
      double ls = sm.lrow[tid] + sm.lrow[tid + 32], gs = sm.dz5[tid] + sm.dz5[tid + 32];
      ls = warp_sum(ls);
      gs = warp_sum(gs);
      if (tid == 0) { loss_sum += ls; gb4 += gs; }
    }

    // ---- output layer backward: dW4 = dz5^T h4, dz4 = dz5 w4 relu'(h4) over h4 --------------------------------
    {
      double gw[4][4], dz[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = tr + 16 * i;
        const double d5 = sm.dz5[r];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = tc + 16 * j;
          double& h = sm.h4[r * LD + k];
          gw[i][j] = d5 * h;
          dz[i][j] = h > 0.0 ? d5 * sm.w4[k] : 0.0;
          h = dz[i][j];
        }
      }
      colsum_part(sm.red[0], gw, tr, tc);
      colsum_part(sm.red[1], dz, tr, tc);
      __syncthreads();
      if (tid < HID) {
        gp[a.off[8] + tid] += colsum_finish(sm.red[0], tid);
        gp[a.off[7] + tid] += colsum_finish(sm.red[1], tid);
      }
    }
    // ---- hidden layers (sm.w holds W3 from the forward pass) ----------------------------------------------------
    hidden_backward(sm, sm.h4, sm.h3, gp + a.off[6], gp + a.off[5], th + a.off[4], tid);   // dz3 over h3, W2 staged
    hidden_backward(sm, sm.h3, sm.h2, gp + a.off[4], gp + a.off[3], nullptr, tid);         // dz2 over h2

    // ---- first hidden layer, chunk by chunk: dW1 += dz2^T h1, dz1 = (dz2 W1) act'(z1), [dW0 | db0] += dz1^T [x, 1]
#pragma unroll 1
    for (int c = 0; c < H1 / KC; ++c) {
      __syncthreads();
      stage_w1_chunk<H1>(sm.w, th + a.off[2], c, tid);
      first_layer_chunk<DIN>(sm, a, c, tid);
      __syncthreads();
      double dw[4][2], dh[4][2];
      zero(dw); zero(dh);
      mm<4, 2, R>(dw, sm.h2, 1, LD, sm.h1, LDC, 1, tr, tc);
      mm<4, 2, HID>(dh, sm.h2, LD, 1, sm.w, LDC, 1, tr, tc);
      double* g1 = gp + a.off[2] + c * KC;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) g1[(tr + 16 * i) * H1 + tc + 16 * j] += dw[i][j];
      double part[2][DIN + 1];
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int d = 0; d <= DIN; ++d) part[j][d] = 0.0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = tr + 16 * i;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const double z = z1<DIN>(sm, r, c * KC + tc + 16 * j);
          double dz;
          if (a.first_act == kFirstSinRelu) {
            double sn, cs;
            sincos(a.scale * z, &sn, &cs);
            dz = sn > 0.0 ? (dh[i][j] * cs) * a.scale : 0.0;
          } else {
            dz = z > 0.0 ? dh[i][j] : 0.0;
          }
#pragma unroll
          for (int d = 0; d < DIN; ++d) part[j][d] = fma(dz, sm.xs[r * MAX_DIN + d], part[j][d]);
          part[j][DIN] += dz;
        }
      }
      double* red = sm.red[0];                        // [tr][kc][DIN + 1]
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int d = 0; d <= DIN; ++d) red[(tr * KC + tc + 16 * j) * (DIN + 1) + d] = part[j][d];
      __syncthreads();
      if (tid < KC * (DIN + 1)) {
        const int kc = tid / (DIN + 1), d = tid - kc * (DIN + 1), f = c * KC + kc;
        double sum = 0.0;
#pragma unroll
        for (int t = 0; t < 16; ++t) sum += red[(t * KC + kc) * (DIN + 1) + d];
        gp[d < DIN ? a.off[0] + f * DIN + d : a.off[1] + f] += sum;
      }
    }
  }
  __syncthreads();                                    // orders the zero fill of gp when this CTA had no tile
  if (tid == 0) {
    gp[a.off[9]] += gb4;
    a.loss_part[(size_t)l * a.S + s] = loss_sum * inv_bs;
  }
}

template <class K>
cudaError_t set_smem(K kernel) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
}

template <int H1>
cudaError_t forward_t(const ArgsF64& a, int ctas, cudaStream_t st) {
  static cudaError_t attr = set_smem(mlp_f64_forward_kernel<H1, 2>);
  if (attr != cudaSuccess) return attr;
  mlp_f64_forward_kernel<H1, 2><<<dim3(ctas, a.L), NT, sizeof(Smem), st>>>(a);
  return cudaGetLastError();
}

template <int H1>
cudaError_t train_t(const ArgsF64& a, cudaStream_t st) {
  static cudaError_t attr = set_smem(mlp_f64_train_kernel<H1, 2>);
  if (attr != cudaSuccess) return attr;
  mlp_f64_train_kernel<H1, 2><<<dim3(a.S, a.L), NT, sizeof(Smem), st>>>(a);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_forward(const ArgsF64& a, int ctas_per_node, cudaStream_t st) {
  if (a.d_in != 2 || ctas_per_node < 1) return cudaErrorInvalidValue;
  switch (a.h1) {
    case 64: return forward_t<64>(a, ctas_per_node, st);
    case 128: return forward_t<128>(a, ctas_per_node, st);
    case 256: return forward_t<256>(a, ctas_per_node, st);
    default: return cudaErrorInvalidValue;
  }
}

cudaError_t launch_train(const ArgsF64& a, int, cudaStream_t st) {
  if (a.d_in != 2 || a.direct || a.S < 1 || a.batch < 1) return cudaErrorInvalidValue;
  switch (a.h1) {
    case 64: return train_t<64>(a, st);
    case 128: return train_t<128>(a, st);
    case 256: return train_t<256>(a, st);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace mlp
}  // namespace nndt
