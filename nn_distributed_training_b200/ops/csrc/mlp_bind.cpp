// Bindings of the implicit-density MLP kernels (mlp_tc.cu: float, mlp_f64.cu: double), the lidar kernels and the generic MLP kernels.
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "mlp.h"
#include "lidar.h"
#include "mlp_generic.h"

namespace py = pybind11;
using namespace nndt;

namespace {
template <typename P> P* ptr(const py::dict& d, const char* k) {
  if (!d.contains(k) || d[k].is_none()) return nullptr;
  return reinterpret_cast<P*>(d[k].cast<uint64_t>());
}
int geti(const py::dict& d, const char* k, int dflt = 0) { return d.contains(k) ? d[k].cast<int>() : dflt; }
double getf(const py::dict& d, const char* k, double dflt = 0) { return d.contains(k) ? d[k].cast<double>() : dflt; }
void check(cudaError_t e, const char* what) {
  if (e != cudaSuccess) throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}

// T = float: tcgen05 kernels (mlp_tc.cu); T = double: fp64 kernels (mlp_f64.cu).  Every pointer, and `scale`, is T.
template <typename T>
struct MlpOpT {
  mlp::ArgsT<T> a{};
  int fwd_ctas = 1, train_ctas = 1;
  explicit MlpOpT(const py::dict& d) { update(d); }
  void update(const py::dict& d) {
    a.theta = ptr<const T>(d, "theta"); a.n_pad = geti(d, "n_pad"); a.L = geti(d, "L");
    auto off = d["off"].cast<std::vector<int>>();
    for (int i = 0; i < 10; ++i) a.off[i] = off.at(i);
    a.d_in = geti(d, "d_in"); a.h1 = geti(d, "h1");
    a.first_act = geti(d, "first_act"); a.last_act = geti(d, "last_act"); a.loss = geti(d, "loss");
    a.scale = (T)getf(d, "scale", 1.0);
    a.x = ptr<const T>(d, "x"); a.y = ptr<const T>(d, "y");
    a.n_rows = geti(d, "n_rows"); a.out = ptr<T>(d, "out");
    a.direct = geti(d, "direct"); a.batch = geti(d, "batch"); a.seed = geti(d, "seed"); a.node0 = geti(d, "node0");
    a.shard_off = ptr<const int>(d, "shard_off"); a.shard_len = ptr<const int>(d, "shard_len");
    a.calls = ptr<const int>(d, "calls"); a.win_table = ptr<const int64_t>(d, "win_table");
    a.grad_part = ptr<T>(d, "grad_part"); a.loss_part = ptr<T>(d, "loss_part"); a.S = geti(d, "S", 1);
    fwd_ctas = geti(d, "fwd_ctas", 1); train_ctas = geti(d, "train_ctas", 1);
  }
  void forward() { check(mlp::launch_forward(a, fwd_ctas, at::cuda::getCurrentCUDAStream().stream()), "mlp_forward"); }
  void train() { check(mlp::launch_train(a, train_ctas, at::cuda::getCurrentCUDAStream().stream()), "mlp_train"); }
};

template <typename T>
void bind_op(py::module& m, const char* name) {
  py::class_<MlpOpT<T>>(m, name)
      .def(py::init<const py::dict&>())
      .def("update", &MlpOpT<T>::update)
      .def("forward", &MlpOpT<T>::forward)
      .def("train", &MlpOpT<T>::train);
}
}  // namespace

static lidar::Args lidar_args(const py::dict& d) {
  lidar::Args a{};
  a.tx = ptr<const double>(d, "tx"); a.ty = ptr<const double>(d, "ty"); a.coef = ptr<const double>(d, "coef");
  a.ntx = geti(d, "ntx"); a.nty = geti(d, "nty");
  a.poses = ptr<const double>(d, "poses"); a.n_poses = geti(d, "n_poses");
  a.num_beams = geti(d, "num_beams"); a.beam_samps = geti(d, "beam_samps");
  a.collision_samps = geti(d, "collision_samps"); a.fine_samps = geti(d, "fine_samps");
  a.beam_len = getf(d, "beam_len"); a.samp_df = getf(d, "samp_df", 1.0);
  a.out = ptr<double>(d, "out");
  return a;
}

static mlpg::Args generic_args(const py::dict& d) {
  mlpg::Args a{};
  a.x = ptr<const void>(d, "x"); a.params = ptr<const void>(d, "params");
  a.M = geti(d, "M"); a.dtype64 = geti(d, "dtype64");
  auto dims = d["dims"].cast<std::vector<int>>();
  auto act = d["act"].cast<std::vector<int>>();
  auto w_off = d["w_off"].cast<std::vector<int>>();
  auto b_off = d["b_off"].cast<std::vector<int>>();
  a.nl = (int)dims.size() - 1;
  if (a.nl < 1 || a.nl > mlpg::kMaxLayers || (int)act.size() != a.nl || (int)w_off.size() != a.nl || (int)b_off.size() != a.nl)
    throw std::runtime_error("mlp_generic: bad layer description");
  int off = 0;
  for (int l = 0; l <= a.nl; ++l) a.dims[l] = dims[l];
  for (int l = 0; l < a.nl; ++l) {
    a.act[l] = act[l]; a.w_off[l] = w_off[l]; a.b_off[l] = b_off[l];
    a.act_off[l] = off; off += dims[l + 1];
  }
  a.act_stride = off;
  a.acts = ptr<void>(d, "acts"); a.gout = ptr<const void>(d, "gout"); a.gparams = ptr<void>(d, "gparams"); a.gx = ptr<void>(d, "gx");
  return a;
}

void bind_mlp(py::module& m) {
  m.def("mlp_generic_forward", [](const py::dict& d) {
    check(mlpg::launch_forward(generic_args(d), at::cuda::getCurrentCUDAStream().stream()), "mlp_generic_forward");
  });
  m.def("mlp_generic_backward", [](const py::dict& d) {
    check(mlpg::launch_backward(generic_args(d), at::cuda::getCurrentCUDAStream().stream()), "mlp_generic_backward");
  });
  m.def("lidar_scan", [](const py::dict& d) {
    check(lidar::launch_scan(lidar_args(d), at::cuda::getCurrentCUDAStream().stream()), "lidar_scan");
  });
  m.def("lidar_density", [](const py::dict& d, uint64_t xy, int n, uint64_t out) {
    check(lidar::launch_density(lidar_args(d), reinterpret_cast<const double*>(xy), n, reinterpret_cast<double*>(out),
                                at::cuda::getCurrentCUDAStream().stream()), "lidar_density");
  });
  bind_op<float>(m, "MlpOp");
  bind_op<double>(m, "MlpOpF64");
}
