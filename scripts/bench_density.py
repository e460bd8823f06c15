"""Secondary benchmark: dist_online_dense_PAPER-shaped DiNNO (FourierNet [2,256,64,64,64,1],
7 robots, batch 12 500, 5 primal steps/round) on a procedural floor plan.
Prints one JSON line with rounds/s for the fused path and the PyTorch-eager path.

DTYPE=float32 (default): the tcgen05 kernels (bf16 operands).  DTYPE=float64: the fp64 kernels (csrc/mlp_f64.cu)
against float64 autograd; the line also carries the GPU's name and power limit and the time of the training kernel
alone over many launches, with its fp64 rate computed from the shapes."""
import glob, json, os, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from nn_distributed_training_b200.floorplans.lidar import Lidar2D, OnlineTrajectoryLidarDataset, RandomPoseLidarDataset
from nn_distributed_training_b200.floorplans.synthetic import write_dataset
from nn_distributed_training_b200.models import FourierNet
from nn_distributed_training_b200.optimizers import DiNNO
from nn_distributed_training_b200.problems import DistOnlineDensityProblem

N = int(os.environ.get("NODES", 7)); B = int(os.environ.get("BATCH", 12500)); PITS = 5
K = int(sys.argv[1]) if len(sys.argv) > 1 else 50
DTYPE = {"float32": torch.float32, "float64": torch.float64}[os.environ.get("DTYPE", "float32")]
tmp = tempfile.mkdtemp()
write_dataset(tmp, n_paths=N, seed=0)
lidar = Lidar2D(os.path.join(tmp, "floor_img.png"), 20, 0.2, 25, 1.0, 50, 3, border_width=8)
paths = sorted(glob.glob(os.path.join(tmp, "tight_paths", "*.npy")))
np.random.seed(0)
train = [OnlineTrajectoryLidarDataset(lidar, np.load(p), 30, 200, seed=0, node=i) for i, p in enumerate(paths)]
val = RandomPoseLidarDataset(lidar, 100)
print("points/node", [len(t) for t in train], file=sys.stderr)
out = {}
for backend in ("fused", "torch"):
    oc = {"alg_name": "dinno", "rho_init": 0.3, "rho_scaling": 1.0004, "outer_iterations": 4000, "primal_iterations": PITS,
          "primal_optimizer": "adam", "persistant_primal_opt": False, "primal_lr_start": 0.001, "primal_lr_finish": 0.0001,
          "lr_decay_type": "log", "profile": False}
    conf = {"problem_name": "o", "train_batch_size": B, "val_batch_size": 10000, "comm_radius": 350.0, "dynamic_graph": True,
            "save_models": False, "metrics": ["validation_loss", "train_loss_moving_average"],
            "metrics_config": {"evaluate_frequency": 10 ** 9, "tloss_decay": 0.2, "mesh_only_at_end": True}, "optimizer_config": oc}
    torch.manual_seed(0)
    pr = DistOnlineDensityProblem(FourierNet([2, 256, 64, 64, 64, 1], 0.05, dtype=DTYPE), torch.nn.BCELoss(), train, val,
                                  "cuda:0", conf, backend=backend, seed=0)
    opt = DiNNO(pr, "cuda:0", dict(oc, consensus_backend="auto" if backend == "fused" else "torch"))
    k = K if backend == "fused" else max(3, K // 10)
    opt.run_rounds(5); opt.run_rounds(k)       # warm-up incl. graph capture of this chunk size
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); opt.run_rounds(k); e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / k
    pr.evaluate_metrics()
    flop = N * PITS * B * 150e3
    out[backend] = {"ms_per_round": ms, "rounds_per_s": 1e3 / ms, "val_loss": pr.metrics["validation_loss"][-1].mean().item(),
                    "model_tflops": flop / (ms * 1e-3) / 1e12}
    if backend == "fused" and DTYPE == torch.float64:
        # the training kernel alone: one launch = one primal step of every node (forward + backward of N x B rows)
        n = 200
        e0.record()
        for _ in range(n):
            pr.fused.train_op.train()
        e1.record(); torch.cuda.synchronize()
        kms = e0.elapsed_time(e1) / n
        out[backend].update(train_kernel_ms=kms, train_kernel_tflops=N * B * 150e3 / (kms * 1e-3) / 1e12)
extra = {}
if DTYPE == torch.float64:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    extra = {"dtype": "float64", "gpu": torch.cuda.get_device_name(0), "nvidia_smi": q}
print(json.dumps({"workload": "dist_online_dense DiNNO", "nodes": N, "batch": B, "primal_iterations": PITS, **extra, **out}))
