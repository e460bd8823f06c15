"""Precision parity study (VERDICT r1 next-round #2): dist_mnist_PAPER (N = 10 cycle, hetero split, 2000 rounds) on the
NON-separable synthetic set, identical data / seeds / sampler:

  * ours fp64 fused  vs  ours fp32 fused: parameter-trajectory distance ||theta32 - theta64|| / ||theta64|| per evaluation
    point, validation accuracy / loss curves of both;
  * the unmodified reference (oracle/_ref, float64, its own DataLoader shuffling) on the same shards: accuracy / loss
    curve next to ours (different minibatch order, so curves agree statistically, not point-wise).

    python scripts/precision_parity.py [--rounds 2000] [--algs dinno,dsgt,dsgd] [--ref-algs dinno] [--out profiles/precision_parity.md]
"""
import argparse
import contextlib
import copy
import json
import os
import sys
import time

import networkx as nx
import torch

ROOT = os.path.join(os.path.dirname(__file__), "..")
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from nn_distributed_training_b200.data.mnist import MNIST_MEAN, MNIST_STD, synthetic_mnist_hard  # noqa: E402
from nn_distributed_training_b200.models import MNISTConvNet  # noqa: E402
from nn_distributed_training_b200.optimizers import build_optimizer  # noqa: E402
from nn_distributed_training_b200.problems.dist_mnist_problem import DistMNISTProblem  # noqa: E402

N = 10
# difficulty presets of data/mnist.py: synthetic_mnist_hard
PRESETS = {"hard": dict(),                                                        # + 2 % label noise
           "hard_clean": dict(label_noise=0.0, dropout=0.25, shift=3, noise=0.55),   # same images, clean labels
           "medium": dict(label_noise=0.0, dropout=0.1, shift=2, noise=0.45)}
METRICS = ["forward_pass_count", "validation_loss", "consensus_error", "top1_accuracy", "current_epoch"]


def shards(train):
    out = []
    for i in range(N):      # hetero split: one class per node (experiments/dist_mnist_ex.py:113-127 of the reference)
        out.append(train.select((train.y == i).nonzero().reshape(-1)))
    return out


def conf_for(alg, rounds, every):
    oc = bench.opt_conf(rounds, alg)
    return {"problem_name": alg, "train_batch_size": 64, "val_batch_size": 128, "metrics": METRICS,
            "metrics_config": {"evaluate_frequency": every}, "optimizer_config": oc}, oc


def run_ours(alg, dtype, train_shards, val, rounds, every):
    pc, oc = conf_for(alg, rounds, every)
    torch.manual_seed(0)
    base = MNISTConvNet(3, 5, 64)
    if dtype == torch.float64:
        base = base.double()
    pr = DistMNISTProblem(nx.cycle_graph(N), base, torch.nn.NLLLoss(), train_shards, val, "cuda:0", pc, backend="fused", seed=0)
    opt = build_optimizer(pr, torch.device("cuda:0"), copy.deepcopy(oc))
    thetas = []
    orig = pr.evaluate_metrics

    def hooked(at_end=False):
        thetas.append(pr.arena.compact(pr.arena.theta).double().cpu().clone())
        return orig(at_end=at_end)
    pr.evaluate_metrics = hooked
    t0 = time.time()
    opt.train()
    torch.cuda.synchronize()
    return {"acc": [float(a.mean()) for a in pr.metrics["top1_accuracy"]],
            "loss": [float(v.mean()) for v in pr.metrics["validation_loss"]],
            "cons": [float(c[1].mean()) for c in pr.metrics["consensus_error"]],
            "theta": thetas, "seconds": time.time() - t0, "kernel": pr.fused.kernel_name}


def run_reference(alg, train_shards, val, rounds, every):
    ref = bench.ensure_reference()
    if ref is None:
        return None
    if ref not in sys.path:
        sys.path.insert(0, ref)
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        from models.mnist_conv_nn import MNISTConvNet as RefNet
        from optimizers.dinno import DiNNO
        from optimizers.dsgd import DSGD
        from optimizers.dsgt import DSGT
        from problems.dist_mnist_problem import DistMNISTProblem as RefProblem

        class U8(torch.utils.data.Dataset):
            def __init__(self, s):
                self.x, self.y = s.x, s.y

            def __len__(self):
                return self.x.shape[0]

            def __getitem__(self, i):
                return ((self.x[i].to(torch.float64) / 255.0) - MNIST_MEAN) / MNIST_STD, int(self.y[i])
        pc, oc = conf_for(alg, rounds, every)
        torch.manual_seed(0)
        base = RefNet(3, 5, 64)
        t0 = time.time()
        with contextlib.redirect_stdout(sys.stderr):
            prob = RefProblem(nx.cycle_graph(N), base, torch.nn.NLLLoss(), [U8(s) for s in train_shards], U8(val), torch.device("cuda:0"), pc)
            {"dinno": DiNNO, "dsgd": DSGD, "dsgt": DSGT}[alg](prob, torch.device("cuda:0"), oc).train()
        return {"acc": [float(a.mean()) for a in prob.metrics["top1_accuracy"]],
                "loss": [float(v.mean()) for v in prob.metrics["validation_loss"]], "seconds": time.time() - t0}
    finally:
        torch.set_default_dtype(old)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2000)
    ap.add_argument("--every", type=int, default=100)
    ap.add_argument("--algs", default="dinno,dsgt,dsgd")
    ap.add_argument("--ref-algs", default="dinno")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "precision_parity.md"))
    ap.add_argument("--preset", default="hard", choices=sorted(PRESETS))
    args = ap.parse_args()
    kw = PRESETS[args.preset]
    train, val = synthetic_mnist_hard(60000, seed=0, **kw), synthetic_mnist_hard(10000, seed=1, **kw)
    sh = shards(train)
    lines = ["# Precision parity: fp32 fused vs fp64 fused vs the fp64 reference", "",
             f"dist_mnist_PAPER hyper-parameters, N = {N} cycle, hetero split (one class per node), batch 64, {args.rounds} rounds, "
             f"`synthetic_mnist_hard` preset `{args.preset}` {PRESETS[args.preset] or '(defaults: stroke dropout 0.25, +-3 px shifts, noise 0.55, 2 % label noise)'} "
             "(classes share strokes; samples drop strokes at random, are shifted and buried in noise).",
             "Same shards, same initial weights; ours fp32 / fp64 also share the minibatch sequence (stateless sampler), the reference "
             "draws its own DataLoader order.  `traj` = ||theta_fp32 - theta_fp64|| / ||theta_fp64|| over all nodes.", ""]
    results = {}
    for alg in args.algs.split(","):
        r64 = run_ours(alg, torch.float64, sh, val, args.rounds, args.every)
        r32 = run_ours(alg, torch.float32, sh, val, args.rounds, args.every)
        ref = run_reference(alg, sh, val, args.rounds, args.every) if alg in args.ref_algs.split(",") else None
        results[alg] = {"fp64": {k: v for k, v in r64.items() if k != "theta"}, "fp32": {k: v for k, v in r32.items() if k != "theta"},
                        "reference": ref}
        lines += [f"## {alg}", "", f"ours fp64: `{r64['kernel']}` {r64['seconds']:.1f} s; ours fp32: `{r32['kernel']}` {r32['seconds']:.1f} s"
                  + (f"; reference fp64: {ref['seconds']:.1f} s" if ref else ""), "",
                  "| round | top-1 ref fp64 | top-1 ours fp64 | top-1 ours fp32 | val-loss ref | val-loss ours fp64 | val-loss ours fp32 | traj fp32 vs fp64 |",
                  "|---|---|---|---|---|---|---|---|"]
        rounds = list(range(0, args.rounds, args.every)) + [args.rounds - 1]
        for i, k in enumerate(rounds[:len(r64["acc"])]):
            t64, t32 = r64["theta"][i], r32["theta"][i]
            traj = ((t32 - t64).norm() / t64.norm()).item()
            ra = f"{ref['acc'][i]:.4f}" if ref and i < len(ref["acc"]) else "-"
            rl = f"{ref['loss'][i]:.5f}" if ref and i < len(ref["loss"]) else "-"
            lines.append(f"| {k} | {ra} | {r64['acc'][i]:.4f} | {r32['acc'][i]:.4f} | {rl} | {r64['loss'][i]:.5f} | {r32['loss'][i]:.5f} | {traj:.2e} |")
        lines.append("")
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    with open(os.path.splitext(args.out)[0] + ".json", "w") as f:
        json.dump(results, f)
    print("\n".join(lines))


if __name__ == "__main__":
    main()
