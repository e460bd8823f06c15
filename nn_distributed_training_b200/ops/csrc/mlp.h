// Launch interface of the implicit-density MLP kernels: networks of the form
//   d_in (<= 4) -> H1 (64|128|256) -> 64 -> 64 -> 64 -> 1
// i.e. the reference's FourierNet [2,256,64,64,64,1] (models/fourier_nn.py:43-59) and ReLU MLPs
// of the same shape family (models/relu_nn.py:4-41).
//   float:  tcgen05 kernels, bf16 operands with fp32 accumulation (mlp_tc.cu)
//   double: CUDA-core fp64 kernels (mlp_f64.cu)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace nndt {
namespace mlp {

enum FirstAct : int { kFirstRelu = 0, kFirstSinRelu = 1 };
enum LastAct : int { kLastNone = 0, kLastSigmoid = 1 };
enum Loss : int { kLossBCE = 0, kLossMSE = 1, kLossL1 = 2 };

// T is the arena dtype: parameters, data, outputs, partials and `scale` are all T.
template <typename T>
struct ArgsT {
  const T* theta;       // [L, n_pad]
  int n_pad, L;
  int off[10];          // slot offsets: W0,b0,W1,b1,W2,b2,W3,b3,W4,b4
  int d_in, h1;
  int first_act, last_act, loss;
  T scale;
  // data: x [M, d_in], y [M]
  const T* x;
  const T* y;
  // forward-only
  int n_rows;           // rows evaluated per node (same inputs for every node)
  T* out;               // [L, n_rows] network output
  // training (see mlp_tc.cu / mlp_f64.cu)
  int direct, batch, seed, node0;
  const int* shard_off; const int* shard_len; const int* calls;
  const int64_t* win_table;  // online sliding-window tables (nullptr: plain epoch sampling)
  T* grad_part;         // [L, S, n_pad]
  T* loss_part;         // [L, S]
  int S;
};
using Args = ArgsT<float>;
using ArgsF64 = ArgsT<double>;

// float: `ctas` is the total grid of the training kernel (static partition of (node, tile) items, S >= G/L + 1 slots)
cudaError_t launch_forward(const Args& a, int ctas_per_node, cudaStream_t st);
cudaError_t launch_train(const Args& a, int ctas, cudaStream_t st);
// double: the training grid is (S, L); CTA s of node l owns grad_part[l, s] and loss_part[l, s] (`ctas` is unused)
cudaError_t launch_forward(const ArgsF64& a, int ctas_per_node, cudaStream_t st);
cudaError_t launch_train(const ArgsF64& a, int ctas, cudaStream_t st);

}  // namespace mlp
}  // namespace nndt
