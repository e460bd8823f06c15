#!/usr/bin/env python
"""Headline benchmark: consensus rounds/sec of DiNNO on the dist_mnist_PAPER config.

    python bench.py --gpus N --steps K --warmup W [--impl ours|reference|nccl] [--dtype fp64|fp32] [--dump-outputs DIR]
    (N > 1: launched by the driver through torch.distributed.run, one rank per GPU)

Config (reference: experiments/dist_mnist_PAPER.yaml problem1): MNISTConvNet(3,5,64),
DiNNO rho0=0.5 x1.0003/round, 2 primal Adam steps/round (lr log 5e-3 -> 5e-4, moments reset
every round), batch 64, cycle graph, one class per node (hetero split).  Weak scaling: every
GPU hosts 10 graph nodes, so N GPUs train a 10*N-node cycle (the node range of the
reference's own scaling experiment, experiments/dist_mnist_scaling.yaml: 10..100 nodes).
A *step* is one communication round of the whole network.  ``value`` is node-rounds/sec =
rounds/sec x number of graph nodes (whole job).  Synthetic MNIST-shaped uint8 data and
random-init weights (no dataset can be downloaded); evaluation is excluded from the timed
region in both arms.

Precision.  The reference runs float64 end to end (experiments/dist_mnist_ex.py:19), so the
headline of BOTH arms is float64 (``--dtype fp64``, the default): ours = the hand-written fp64
cluster kernel (csrc/mnist_cl64.cu: K-split over 6-CTA clusters, fp64 CUDA cores, DSMEM reductions)
+ the fp64 instantiation of the fused consensus kernels.  ``extra.fp32`` carries the same measurement
at float32 for both arms (ours = csrc/mnist_tc.cu, tcgen05 / TMEM / tensor-map TMA with 3xTF32;
reference = the same stock classes under torch.set_default_dtype(float32)).

* ``value``  — device-timed (CUDA events on the launching stream, max over ranks), shards
  resident in HBM (the framework's native pipeline); each GPU's shard set is sized > L2 and
  rows are gathered at random, so inputs are not L2-resident between iterations.
* ``e2e``    — same metric through the public API ``DiNNO(problem, device, conf).run_rounds``
  with the host-fed input pipeline: every round copies that round's minibatches from
  pinned host memory (H2D) and reads the per-node losses back (D2H).
* timing protocol — W warm-up rounds, then the CUDA graphs of the K timed rounds are captured
  (not run); every rank enqueues [device rank barrier, event, K rounds, event] behind a gate
  kernel and the host opens the gate: the K rounds start within an NVLink flag latency on all
  GPUs and no host-side skew (NCCL barrier exit, NVML, Python) is inside the events.
* ``extra.one_per_gpu`` — the communication-bound regime (N > 1): ONE graph node per GPU,
  ring / complete (NVLS) / random graph x DiNNO / DSGD / DSGT, every edge crosses NVLink.
* ``extra.multi_gpu_selfcheck`` — (N > 1, untimed) the distributed run's parameters after a few
  rounds against a single-process recomputation on rank 0.
* ``--impl reference`` — the unmodified reference (oracle/_ref, installed by ``build()``) through its own public API
  (DistMNISTProblem + DiNNO(...).train(profiler=hook)), all nodes on one device.
* ``--impl nccl`` — one-rank-per-GPU PyTorch + NCCL re-expression (batched cuDNN/cuBLAS
  forward/backward of all local nodes, all_gather of the parameter rows, torch elementwise
  mixing/Adam, CUDA-graph captured): "the NCCL baseline" a library-only solution would be.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NODES_PER_GPU = 10
BATCH = 64
REF_MAX_SECONDS = 120.0
REF_SEC_PER_NODE_ROUND = 0.00465
PITS = 2
SAMPLES_PER_NODE = 22000          # 10 nodes x 22000 x 784 B = 172 MB of uint8 rows per GPU (> 126 MB L2)
REF_SAMPLES_PER_NODE = 6000       # the paper's 60000 / 10 (the reference streams from host memory anyway)
PAPER_ROUNDS = 2000
DUMP_MAX_BYTES = 64 << 20
METRIC = "consensus node-rounds/sec (DiNNO, dist_mnist_PAPER; rounds/sec x graph nodes)"


def opt_conf(outer_iterations: int, alg: str = "dinno"):
    if alg == "dsgd":       # experiments/dist_mnist_PAPER.yaml problem3
        return {"alg_name": "dsgd", "alpha0": 0.005, "mu": 0.001, "outer_iterations": outer_iterations, "profile": False}
    if alg == "dsgt":       # problem2
        return {"alg_name": "dsgt", "alpha": 0.005, "init_grads": True, "outer_iterations": outer_iterations, "profile": False}
    return {"alg_name": "dinno", "rho_init": 0.5, "rho_scaling": 1.0003, "outer_iterations": outer_iterations,
            "primal_iterations": PITS, "primal_optimizer": "adam", "persistant_primal_opt": False,
            "primal_lr_start": 0.005, "primal_lr_finish": 0.0005, "lr_decay_type": "log", "profile": False}


def prob_conf(oc, eval_every, extra=None):
    c = {"problem_name": oc["alg_name"], "train_batch_size": BATCH, "val_batch_size": 128, "verbose_evals": True,
         "metrics": ["forward_pass_count", "validation_loss", "consensus_error", "top1_accuracy", "current_epoch"],
         "metrics_config": {"evaluate_frequency": eval_every}, "optimizer_config": oc}
    c.update(extra or {})
    return c


def headline_config(n_gpus: int):
    """Identical in both arms (the driver compares the dicts)."""
    n = NODES_PER_GPU * n_gpus
    return {"model": "MNISTConvNet(3,5,64) 28440 params", "yaml": "dist_mnist_PAPER.yaml/problem1 (DiNNO)",
            "graph": f"cycle, {n} nodes ({NODES_PER_GPU} per GPU)", "global_batch": BATCH * n,
            "primal_iterations": PITS, "seq_len": None,
            "parallelism": f"consensus graph, {NODES_PER_GPU} nodes/GPU x {n_gpus} GPU",
            "eval": "excluded from timed region",
            "l2": "inputs > L2 or streamed from host memory every step; no flush"}


# ------------------------------------------------------------------ clocks ----
class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self._h = None
        self._t = threading.Thread(target=self._loop, daemon=True)
        self.active = False

    def _once(self):
        if self._h is None:
            return
        nv = self._nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h) if hasattr(
                nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
                     0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}
            for bit, name in names.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:  # noqa: BLE001
            pass

    def _loop(self):
        while not self._stop.is_set():
            if self.active:
                self._once()
            time.sleep(0.0005)

    def start(self):
        """Spawn the sampling thread (call BEFORE the barrier that precedes the timed region)."""
        self._t.start()

    def stop(self):
        self._once()
        self._stop.set()
        self._t.join(timeout=1)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


class StepTimer:
    """``profiler.step()`` hook of the reference arm: records a CUDA event after every round; the timed region
    is rounds [warmup, warmup+steps)."""

    def __init__(self, warmup, steps, on_start=None, on_stop=None):
        import torch
        self.torch = torch
        self.warmup, self.steps = warmup, steps
        self.count = 0
        self.ev0 = self.ev1 = None
        self.on_start, self.on_stop = on_start, on_stop
        self.wall = None

    def step(self):
        torch = self.torch
        self.count += 1
        if self.count == self.warmup:
            if self.on_start:
                self.on_start()
            torch.cuda.synchronize()
            self._t0 = time.perf_counter()
            self.ev0 = torch.cuda.Event(enable_timing=True)
            self.ev0.record()
        elif self.count == self.warmup + self.steps:
            self.ev1 = torch.cuda.Event(enable_timing=True)
            self.ev1.record()
            torch.cuda.synchronize()
            self.wall = time.perf_counter() - self._t0
            if self.on_stop:
                self.on_stop()

    def ms(self):
        return self.ev0.elapsed_time(self.ev1)


# -------------------------------------------------------------------- ours ----
_SHARD_CACHE = {}


def _shard(n, seed, classes):
    from nn_distributed_training_b200.data.mnist import synthetic_mnist
    key = (n, seed, tuple(classes) if classes is not None else None)
    if key not in _SHARD_CACHE:
        _SHARD_CACHE[key] = synthetic_mnist(n, seed=seed, classes=classes)
    return _SHARD_CACHE[key]


class _Stub:
    def __init__(self, n):
        self.n = n

    def __len__(self):
        return self.n


def build_problem(ctx, graph, oc, eval_every, extra=None, samples_per_node=SAMPLES_PER_NODE, backend="fused",
                  dtype="fp32"):
    import torch
    from nn_distributed_training_b200.models import MNISTConvNet
    from nn_distributed_training_b200.parallel.context import Placement
    from nn_distributed_training_b200.problems.dist_mnist_problem import DistMNISTProblem

    n_nodes = graph.number_of_nodes()
    pl = Placement(n_nodes, ctx.world_size, ctx.rank)
    train = [(_shard(samples_per_node, 100 + g, [g % 10]) if pl.is_local(g) else _Stub(samples_per_node))
             for g in range(n_nodes)]
    val = _shard(10000, 1, None)
    torch.manual_seed(0)
    base = MNISTConvNet(3, 5, 64)
    if dtype == "fp64":
        base = base.double()
    return DistMNISTProblem(graph, base, torch.nn.NLLLoss(), train, val, ctx.device,
                            prob_conf(oc, eval_every, extra), ctx=ctx, backend=backend)


class Harness:
    """Aligned device timing of ``opt.run_rounds(K)`` (see the module docstring)."""

    def __init__(self, ctx):
        import torch
        from nn_distributed_training_b200.parallel.symm import DeviceBarrier
        self.torch, self.ctx = torch, ctx
        self.bar = DeviceBarrier(ctx)

    def maxreduce(self, x):
        torch = self.torch
        t = torch.tensor([x], dtype=torch.float64, device=self.ctx.device)
        return float(self.ctx.all_reduce_max(t).item())

    def time_rounds(self, opt, K, sampler=None):
        torch, ctx = self.torch, self.ctx
        opt.prepare_rounds(K)                 # capture (not run) the graphs of the timed call
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ctx.barrier()
        if sampler is not None:
            sampler.active = True
        t0 = time.perf_counter()
        self.bar.enqueue(gate=True)           # spins until the host opens the gate, then aligns all ranks on the device
        e0.record()
        opt.run_rounds(K)
        e1.record()
        self.bar.open_gate()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if sampler is not None:
            sampler.active = False
        ctx.barrier()
        return self.maxreduce(e0.elapsed_time(e1)), self.maxreduce(wall * 1e3)


def _cycle(n):
    import networkx as nx
    if os.environ.get("NNDT_BENCH_GRAPH") == "disjoint":      # diagnostic: one closed cycle per GPU, no edge crosses NVLink
        return nx.disjoint_union_all([nx.cycle_graph(NODES_PER_GPU) for _ in range(max(1, n // NODES_PER_GPU))])
    return nx.cycle_graph(n) if n > 2 else nx.path_graph(n)


def dump_outputs(out_dir, ctx, pr, opt):
    """Write what the timed ``run_rounds(K)`` hands its caller after the last timed round, one row per graph node:
    ``theta`` (parameters, ``parameters_to_vector`` order), ``duals`` (DiNNO dual variables) and ``losses`` (minibatch
    loss of the round's last primal step).  Above DUMP_MAX_BYTES, theta and duals keep a fixed seeded sample of columns."""
    import numpy as np
    arrays = {"theta": pr.arena.compact(pr.gather_rows(pr.arena.theta)), "duals": pr.arena.compact(pr.gather_rows(opt.duals)),
              "losses": pr.gather_rows(pr.fused.loss_part.sum(1))}
    if not ctx.is_main:
        return
    arrays = {k: v.cpu().numpy() for k, v in arrays.items()}
    n = arrays["theta"].shape[1]
    keep = int((DUMP_MAX_BYTES - arrays["losses"].nbytes) * n // (arrays["theta"].nbytes + arrays["duals"].nbytes))
    if keep < n:
        cols = np.sort(np.random.RandomState(0).choice(n, keep, replace=False))
        arrays["theta"], arrays["duals"] = arrays["theta"][:, cols], arrays["duals"][:, cols]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure_headline(h, ctx, args, dtype, sampler=None, probe=False, dump_dir=None):
    """value (resident/staged shards) + e2e (host-fed) of the headline config at ``dtype``; with ``dump_dir`` the
    outputs of the last timed round are written there (``dump_outputs``)."""
    import torch
    from nn_distributed_training_b200.optimizers import DiNNO

    n_nodes = NODES_PER_GPU * args.gpus
    W, K = max(args.warmup, 3), args.steps
    oits = max(PAPER_ROUNDS, 8 * (W + K) + 1024)
    dev = ctx.device
    pipeline = os.environ.get("NNDT_BENCH_PIPELINE", "auto")      # auto (= staged-resident) | resident (A/B switch)
    pr = build_problem(ctx, _cycle(n_nodes), opt_conf(oits), 10 ** 9, extra={"input_pipeline": pipeline}, dtype=dtype)
    opt = DiNNO(pr, dev, pr.conf["optimizer_config"])
    opt.run_rounds(W)                     # warm-up (captures + runs its own graph)
    ms, _ = h.time_rounds(opt, K, sampler)
    if dump_dir:
        dump_outputs(dump_dir, ctx, pr, opt)
    prog = opt._program
    out = {"ms_per_step": ms / K, "value": n_nodes * K / (ms / 1e3), "launches": K * prog.launches_per_round(),
           "pipeline": prog.pipeline, "symm": prog.eng.pub_buf.how, "flags": prog.eng.flag_mode,
           "fwd_bwd_kernel": ("convnet_generic_kernel<%s> (CUDA cores)" % ("double" if dtype == "fp64" else "float"))
           if (pr.fused.generic and not pr.fused.cl64) else pr.fused.kernel_name}
    if probe:   # per-call fixed cost: t(K) = intercept + slope K  (K = 20 is the production chunk, evaluate_frequency 20)
        pts = []
        for kk in (4, 20, 64, 256):
            m, _ = h.time_rounds(opt, kk)
            pts.append((kk, m))
        n = len(pts); sx = sum(p[0] for p in pts); sy = sum(p[1] for p in pts)
        sxx = sum(p[0] ** 2 for p in pts); sxy = sum(p[0] * p[1] for p in pts)
        slope = (n * sxy - sx * sy) / (n * sxx - sx * sx)
        out["fixed_cost_probe"] = {"ms_by_K": {str(k): round(m, 4) for k, m in pts}, "slope_ms_per_round": round(slope, 5),
                                   "intercept_ms": round((sy - slope * sx) / n, 4)}
    pr.evaluate_metrics()                 # model quality after the rounds run so far (not timed)
    out["top1_after_rounds"] = float(pr.metrics["top1_accuracy"][-1].mean())
    out["rounds_done"] = opt.k
    prog.eng.check()
    del opt, pr, prog
    torch.cuda.empty_cache()

    # ---------------- end to end through the public API, host-fed inputs -------
    try:
        W2 = max(W, 6)
        pr2 = build_problem(ctx, _cycle(n_nodes), opt_conf(oits), 10 ** 9, extra={"input_pipeline": "host"}, dtype=dtype)
        opt2 = DiNNO(pr2, dev, pr2.conf["optimizer_config"])
        opt2.run_rounds(W2)                      # warm-up: captures the round graphs, stages the first batch
        ms2, wall2 = h.time_rounds(opt2, K)      # public stepping API: K rounds, each with its H2D copy + D2H loss read
        last_losses = pr2.fused.loss_host.sum(1).tolist()
        hf = pr2.fused.host_feed
        if pr2.fused.loader is not None:
            pr2.fused.loader.stop()
        out["e2e"] = {"value": n_nodes * K / (ms2 / 1e3), "unit": "node-rounds/s", "ms_per_step": ms2 / K,
                      "h2d_bytes_per_step": int(hf["h2d_bytes"]), "d2h_bytes_per_step": int(hf["d2h_bytes"]),
                      "api": "DiNNO(problem, device, conf).run_rounds(K) with problem conf input_pipeline=host",
                      "h2d": hf["mode"] + ": every round's uint8 rows + labels are pulled from the pinned host dataset over PCIe",
                      "d2h": ("the training kernel stores every step's per-CTA losses into a pinned host buffer (device-initiated PCIe write)"
                              if getattr(pr2.fused, "loss_mode", "") == "mirror" else "cudaMemcpyAsync D2H node per round"),
                      "wall_ms_per_step": wall2 / K, "last_round_losses_read_back": last_losses[:3]}
        opt2._program.eng.check()
        del opt2, pr2
    except Exception as e:  # noqa: BLE001
        out["e2e"] = {"error": repr(e)[:300]}
    torch.cuda.empty_cache()
    return out


def measure_one_per_gpu(h, ctx, args):
    """Communication-bound regime: one graph node per GPU, every edge over NVLink (BASELINE.json configs 2-3)."""
    import networkx as nx
    import torch
    from nn_distributed_training_b200.optimizers import build_optimizer
    G = args.gpus
    graphs = {"cycle": _cycle(G), "complete": nx.complete_graph(G)}
    if G >= 4:
        graphs["random"] = _seeded_random_graph(G)       # Erdos-Renyi p = 0.5, connected (dist_mnist_PAPER-style random graph)
    K, W = max(args.steps, 40), 5
    res = {}
    for gname, g in graphs.items():
        for alg in ("dinno", "dsgd", "dsgt"):
            key = f"{alg}/{gname}"
            try:
                oc = opt_conf(8 * (W + K) + 64, alg)
                pr = build_problem(ctx, g, oc, 10 ** 9, samples_per_node=2048, dtype="fp32")
                opt = build_optimizer(pr, ctx.device, oc)
                opt.run_rounds(W)
                ms, _ = h.time_rounds(opt, K)
                eng = opt._program.eng
                eng.check()
                res[key] = {"ms_per_round": round(ms / K, 5), "node_rounds_per_s": round(G * K / (ms / 1e3), 1),
                            "edges_over_nvlink": g.number_of_edges(), "max_degree": max(dict(g.degree()).values()),
                            "nvls_sum_mode": bool(eng.sum_mode), "multicast": bool(eng.sum_buf is not None and eng.sum_buf.multicast_ptr)}
                del opt, pr
            except Exception as e:  # noqa: BLE001
                res[key] = {"error": repr(e)[:200]}
            torch.cuda.empty_cache()
    return res


def _seeded_random_graph(n, p=0.5, seed=7):
    import networkx as nx
    for s in range(seed, seed + 200):
        g = nx.erdos_renyi_graph(n, p, seed=s)
        if nx.is_connected(g):
            return g
    return nx.cycle_graph(n)


def selfcheck(ctx, args):
    """Distributed run == single-process recomputation (what tests/dist_worker.py asserts), at the bench's node count."""
    import copy
    import torch
    from nn_distributed_training_b200.optimizers import build_optimizer
    from nn_distributed_training_b200.parallel.context import DistContext

    n_nodes, R = NODES_PER_GPU * args.gpus, 6
    worst, detail = 0.0, {}
    for alg in ("dinno", "dsgt"):
        oc = opt_conf(R, alg)
        pr = build_problem(ctx, _cycle(n_nodes), oc, 10 ** 9, samples_per_node=640)
        opt = build_optimizer(pr, ctx.device, copy.deepcopy(oc))
        opt.run_rounds(R)
        torch.cuda.synchronize()
        opt._program.eng.check()
        theta = pr.gather_rows(pr.arena.theta).cpu()
        if ctx.is_main:
            solo = DistContext.single(ctx.device)
            pr1 = build_problem(solo, _cycle(n_nodes), oc, 10 ** 9, samples_per_node=640)
            opt1 = build_optimizer(pr1, solo.device, copy.deepcopy(oc))
            opt1.run_rounds(R)
            torch.cuda.synchronize()
            ref = pr1.arena.theta.cpu()
            rel = ((theta - ref).norm() / ref.norm()).item()
            detail[alg] = rel
            worst = max(worst, rel)
            del opt1, pr1
        ctx.barrier()
        del opt, pr
    # not bitwise: a rank with L nodes picks another batch split (samples per CTA) than the single process with N nodes,
    # so fp32 partial sums associate differently and Adam amplifies the last-bit differences over the rounds
    return {"status": "pass" if worst < 1e-3 else "fail", "max_rel": worst, "rounds": R, "nodes": n_nodes, "per_alg": detail}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from nn_distributed_training_b200.parallel.context import DistContext

    ctx = DistContext.from_env(use_cuda=True)
    assert ctx.world_size == args.gpus, f"launched with WORLD_SIZE={ctx.world_size} but --gpus {args.gpus}"
    dev = ctx.device
    h = Harness(ctx)
    sampler = ClockSampler(dev.index or 0)
    sampler.start()                       # thread + NVML handle exist before any barrier of a timed region
    main = measure_headline(h, ctx, args, args.dtype, sampler, probe=args.extras, dump_dir=args.dump_outputs)
    clocks = sampler.stop()
    extra = {"top1_after_rounds": main["top1_after_rounds"], "rounds_done": main["rounds_done"]}
    if "fixed_cost_probe" in main:
        extra["fixed_cost_probe"] = main["fixed_cost_probe"]
    if args.extras:
        other = "fp32" if args.dtype == "fp64" else "fp64"
        try:
            o = measure_headline(h, ctx, args, other)
            extra[other] = {"value": o["value"], "ms_per_step": o["ms_per_step"], "e2e": o["e2e"], "dtype": other,
                            "fwd_bwd_kernel": o["fwd_bwd_kernel"], "gpu_launches": o["launches"],
                            "top1_after_rounds": o["top1_after_rounds"]}
        except Exception as e:  # noqa: BLE001
            extra[other] = {"error": repr(e)[:300]}
        if args.gpus > 1:
            try:
                extra["multi_gpu_selfcheck"] = selfcheck(ctx, args)
            except Exception as e:  # noqa: BLE001
                extra["multi_gpu_selfcheck"] = {"status": "error", "error": repr(e)[:300]}
            try:
                extra["one_per_gpu"] = measure_one_per_gpu(h, ctx, args)
            except Exception as e:  # noqa: BLE001
                extra["one_per_gpu"] = {"error": repr(e)[:300]}
    if ctx.is_main:
        K = args.steps
        cfg = headline_config(args.gpus)
        out = {
            "metric": METRIC, "value": main["value"], "unit": "node-rounds/s", "n_gpus": args.gpus, "steps": K,
            "warmup": max(args.warmup, 3), "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic", "impl": "ours",
            "config": cfg, "clocks": clocks, "e2e": main["e2e"], "gpu_launches": main["launches"],
            "multi_gpu_selfcheck": extra.get("multi_gpu_selfcheck", {}).get("status", "n/a (1 GPU)" if args.gpus == 1 else "skipped"),
            "details": {"rounds_per_sec": K / (main["ms_per_step"] * K / 1e3), "fwd_bwd_kernel": main["fwd_bwd_kernel"],
                        "input_pipeline": main["pipeline"], "exchange": f"in-kernel P2P pulls of neighbor rows ({main['symm']} peer mapping, "
                        f"{main['flags']} flags); no NCCL on the hot path",
                        "timing": "W warm-up rounds; graphs of the K timed rounds captured beforehand; device rank barrier + host gate; "
                                  "CUDA events, max over ranks",
                        "l2": f"inputs {NODES_PER_GPU * SAMPLES_PER_NODE * 784 / 1e6:.0f} MB/GPU > L2: every round's rows are gathered at "
                              f"random from the HBM-resident shards (never re-used within {SAMPLES_PER_NODE // BATCH} steps); no flush",
                        "host_placement": (f"rank bound to the {ctx.local_cpus} CPUs NVML reports local to its GPU (pinned staging buffers on that socket)"
                                           if getattr(ctx, "local_cpus", None) else "process affinity unchanged")},
            "extra": extra,
        }
        print(json.dumps(out))
    if dist.is_initialized():
        dist.destroy_process_group()


# ----------------------------------------------------------- NCCL baseline ----
def run_nccl_baseline(args):
    from baseline.nccl_baseline import run as run_nccl
    run_nccl(args, METRIC, NODES_PER_GPU, BATCH, PITS, opt_conf, _shard)


# --------------------------------------------------------------- reference ----
def ensure_reference():
    """The unmodified reference tree that ``build()`` installed (oracle/install_reference.py), or None."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    return ref if os.path.isdir(os.path.join(ref, "optimizers")) else None


def run_reference(args):
    ref = ensure_reference()
    if ref is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref missing: build() installs the reference there from a checkout of it"}))
        return
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world > 1:
        # the reference has no multi-process / multi-GPU mode: rank 0 simulates every node on
        # its GPU (the stock path), the other ranks only join the barriers.
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo", rank=rank, world_size=world)
    if rank == 0:
        import contextlib
        try:
            with contextlib.redirect_stdout(sys.stderr):      # the reference prints its metrics; stdout carries one JSON line
                out = _reference_rank0(args, ref, args.dtype, REF_MAX_SECONDS * (0.6 if args.extras else 1.0))
                if args.extras:
                    other = "fp32" if args.dtype == "fp64" else "fp64"
                    try:
                        o = _reference_rank0(args, ref, other, REF_MAX_SECONDS * 0.4)
                        out["extra"] = {other: {"value": o["value"], "ms_per_step": o["ms_per_step"], "steps": o["steps"], "dtype": other}}
                    except Exception as e:  # noqa: BLE001
                        out["extra"] = {other: {"error": repr(e)[:200]}}
        except Exception as e:  # noqa: BLE001
            out = {"impl": "reference", "unavailable": "reference run failed: " + repr(e)[:200]}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _reference_rank0(args, ref, dtype, budget_s):
    import torch
    if ref not in sys.path:
        sys.path.insert(0, ref)
    # float64 is what the stock runner sets on import (experiments/dist_mnist_ex.py:19); the fp32 run uses the same
    # unmodified classes with the other default dtype
    torch.set_default_dtype(torch.float64 if dtype == "fp64" else torch.float32)
    from models.mnist_conv_nn import MNISTConvNet
    from optimizers.dinno import DiNNO
    from problems.dist_mnist_problem import DistMNISTProblem
    from utils import graph_generation
    from nn_distributed_training_b200.data.mnist import MNIST_MEAN, MNIST_STD

    class U8Images(torch.utils.data.Dataset):
        """uint8 images -> normalised default-dtype tensors per item (the job torchvision's
        ToTensor+Normalize transform does in the stock runner)."""

        def __init__(self, shard):
            self.x, self.y = shard.x, shard.y

        def __len__(self):
            return self.x.shape[0]

        def __getitem__(self, i):
            return ((self.x[i].to(torch.get_default_dtype()) / 255.0) - MNIST_MEAN) / MNIST_STD, int(self.y[i])

    n_nodes = NODES_PER_GPU * args.gpus
    W, K_req = max(args.warmup, 3), args.steps
    # The stock path simulates every node sequentially (measured 4.65 ms per node-round on B200): bound the timed
    # region so `--gpus 8 --steps 1000` (6 minutes of reference rounds) cannot time the driver out.
    # The JSON reports the steps actually timed.
    K = min(K_req, max(5, int(budget_s / (REF_SEC_PER_NODE_ROUND * n_nodes)) - W))
    device = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    N, graph = graph_generation.generate_from_conf({"num_nodes": n_nodes, "type": "cycle", "p": 0.3, "gen_attempts": 100})
    train = [U8Images(_shard(REF_SAMPLES_PER_NODE, 100 + g, [g % 10])) for g in range(N)]
    val = U8Images(_shard(10000, 1, None))
    torch.manual_seed(0)
    base = MNISTConvNet(3, 5, 64)
    oc = opt_conf(W + K + 1)
    pc = prob_conf(oc, 10 ** 9)
    prob = DistMNISTProblem(graph, base, torch.nn.NLLLoss(), train, val, device, pc)
    dopt = DiNNO(prob, device, oc)
    sampler = ClockSampler(0)
    sampler.start()

    def on():
        sampler.active = True

    timer = StepTimer(W, K, on_start=on)
    dopt.train(profiler=timer)     # evaluates at k=0 (before warm-up) and at the last, untimed, round
    clocks = sampler.stop()
    ms = timer.ms()
    itemsize = 8 if dtype == "fp64" else 4
    h2d = N * PITS * BATCH * (784 * itemsize + 8)
    out = {"metric": METRIC, "value": N * K / (ms / 1e3), "unit": "node-rounds/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
           "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": dtype, "data": "synthetic", "impl": "reference", "steps_requested": K_req,
           "config": headline_config(args.gpus),
           "clocks": clocks,
           "e2e": {"value": N * K / (ms / 1e3), "unit": "node-rounds/s", "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": 0, "note": "stock path already feeds every batch from host memory"},
           "gpu_launches": None,
           "details": {"rounds_per_sec": K / (ms / 1e3), "graph": f"cycle, {N} nodes, all simulated on one device: the reference's only mode",
                       "parallelism": "single process, single device", "l2": "inputs streamed from host memory every step"}}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="timed rounds; --impl reference times at most REF_MAX_SECONDS of rounds (at its measured rate "
                         "per node-round) and reports the rounds it timed as steps, the requested ones as steps_requested")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "nccl"])
    ap.add_argument("--dtype", default=os.environ.get("NNDT_BENCH_DTYPE", "fp64"), choices=["fp64", "fp32"])
    ap.add_argument("--no-extras", dest="extras", action="store_false",
                    help="headline only: skip the other-precision run, the one-node-per-GPU sweep, the self-check and the probe")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed round as DIR/<name>.npy (--impl ours)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs is implemented for --impl ours")
    if args.impl == "reference":
        if "--steps" not in " ".join(sys.argv):
            args.steps = 100
        run_reference(args)
    elif args.impl == "nccl":
        if "--steps" not in " ".join(sys.argv):
            args.steps = 100
        run_nccl_baseline(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
