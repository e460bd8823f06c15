"""Generates the experiment YAMLs under experiments/ from one table of hyper-parameters
(the values are those of the reference's shipped configs: experiments/*.yaml; the missing
``dist_mnist_template.yaml`` and the stale ``dist_dense_v2.yaml`` schema are re-authored —
SURVEY Q12/Q13).  Run: python scripts/make_configs.py"""
import copy
import os

import yaml

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "experiments")

MNIST_METRICS = ["forward_pass_count", "validation_loss", "consensus_error", "top1_accuracy", "current_epoch"]
DENSE_METRICS = ["forward_pass_count", "train_loss_moving_average", "validation_loss", "consensus_error",
                 "mesh_grid_density", "current_epoch"]


def mnist_problem(name, opt, metrics=None, bs=64):
    return {"problem_name": name, "train_batch_size": bs, "val_batch_size": 128, "verbose_evals": True,
            "metrics": list(metrics or MNIST_METRICS), "metrics_config": {"evaluate_frequency": 20},
            "optimizer_config": opt}


def dinno(oits, rho0, rs, pits, lr0, lr1, decay="log"):
    return {"alg_name": "dinno", "rho_init": rho0, "rho_scaling": rs, "outer_iterations": oits,
            "primal_iterations": pits, "primal_optimizer": "adam", "persistant_primal_opt": False,
            "primal_lr_start": lr0, "primal_lr_finish": lr1, "lr_decay_type": decay, "profile": False}


def dsgt(oits, alpha):
    return {"alg_name": "dsgt", "outer_iterations": oits, "alpha": alpha, "init_grads": True, "profile": False}


def dsgd(oits, alpha0, mu):
    return {"alg_name": "dsgd", "outer_iterations": oits, "alpha0": alpha0, "mu": mu, "profile": False}


SOLO = {"train_solo": False, "optimizer": "adam", "lr": 0.005, "epochs": 6, "train_batch_size": 100,
        "val_batch_size": 100, "verbose": True}
MNIST_MODEL = {"num_filters": 3, "kernel_size": 5, "linear_width": 64}


def mnist_exp(name, graph, split="hetero", **kw):
    e = {"name": name, "data_dir": "../data/", "output_metadir": "../results/", "use_cuda": True,
         "writeout": True, "data_split_type": split, "loss": "NLL", "graph": graph, "model": dict(MNIST_MODEL),
         "individual_training": dict(SOLO)}
    e.update(kw)
    return e


configs = {}
cycle10 = {"num_nodes": 10, "type": "cycle", "p": 0.3, "gen_attempts": 100}
configs["dist_mnist_PAPER.yaml"] = {
    "experiment": mnist_exp("dist_mnist_PAPER", cycle10),
    "problem_configs": {
        "problem1": mnist_problem("dinno", dinno(2000, 0.5, 1.0003, 2, 0.005, 0.0005)),
        "problem2": mnist_problem("dsgt", dsgt(2000, 0.005)),
        "problem3": mnist_problem("dsgd", dsgd(2000, 0.005, 0.001)),
    }}
configs["dist_mnist_anim.yaml"] = {
    "experiment": mnist_exp("dist_mnist_anim", cycle10),
    "problem_configs": {"problem1": mnist_problem("dinno", dinno(3000, 0.5, 1.0003, 2, 0.005, 0.0005),
                                                  metrics=MNIST_METRICS + ["validation_as_vector"])}}
# the README's getting-started config (README.md:71,78) that the reference never shipped:
# DSGD, 2 nodes, CPU, no files written.
configs["dist_mnist_template.yaml"] = {
    "experiment": mnist_exp("dist_mnist_template", {"num_nodes": 2, "type": "cycle", "p": 0.3, "gen_attempts": 100},
                            split="random", use_cuda=False, writeout=False),
    "problem_configs": {"problem1": mnist_problem("dsgd", dsgd(100, 0.005, 0.001))}}
# 8 nodes = 8 GPUs on a random graph, all three algorithms (BASELINE.json config 2)
configs["dist_mnist_8gpu.yaml"] = {
    "experiment": mnist_exp("dist_mnist_8gpu", {"num_nodes": 8, "type": "random", "p": 0.4, "gen_attempts": 100, "seed": 0},
                            split="hetero"),
    "problem_configs": copy.deepcopy(configs["dist_mnist_PAPER.yaml"]["problem_configs"])}
configs["dist_mnist_scaling.yaml"] = {
    "experiment": {"name": "scaling_dinno_const_fied", "data_dir": "../data/", "output_metadir": "../results_scaling/",
                   "use_cuda": True, "writeout": True, "loss": "NLL", "model": dict(MNIST_MODEL),
                   "scaling": {"const": "fiedler", "min_N": 10, "max_N": 100, "target_fied": 1.0, "min_fied": 0.1,
                               "max_fied": 2.0, "num_nodes": 20, "num_trials": 10}},
    "problem": mnist_problem("dinno", dinno(1500, 0.5, 1.0003, 2, 0.005, 0.0005))}

LIDAR = {"data_dir": "../floorplans/32_data/", "waypoint_subdir": "tight_paths", "split_type": "trajectory",
         "num_beams": 20, "beam_samps": 25, "beam_length": 0.2, "collision_samps": 50, "fine_samps": 3,
         "samp_distribution_factor": 1.0, "border_width": 30, "round_density": True}
FOURIER = {"shape": [2, 256, 64, 64, 64, 1], "scale": 0.05}


def online_problem(name, bs, opt, metrics=None, mesh_end=True):
    return {"problem_name": name, "train_batch_size": bs, "val_batch_size": 10000, "comm_radius": 1500.0,
            "verbose_evals": True, "dynamic_graph": True, "save_models": True,
            "metrics": list(metrics or DENSE_METRICS),
            "metrics_config": {"evaluate_frequency": 20, "tloss_decay": 0.2, "mesh_only_at_end": mesh_end},
            "optimizer_config": opt}


def online_exp(name, solo_bs, train_solo):
    return {"name": name, "output_metadir": "../results/", "writeout": True, "use_cuda": True, "seed": 0,
            "data": dict(LIDAR, num_scans_in_window=800, spline_res=30, num_validation_scans=500),
            "loss": "BCE", "model": dict(FOURIER),
            "individual_training": {"train_solo": train_solo, "optimizer": "adam", "lr": 0.001, "epochs": 1,
                                    "train_batch_size": solo_bs, "val_batch_size": 10000, "verbose": True}}


configs["dist_online_dense_PAPER.yaml"] = {
    "experiment": online_exp("dist_online_dense_PAPER", 10000, True),
    "problem_configs": {
        "problem1": online_problem("dinno_log", 12500, dinno(4000, 0.3, 1.0004, 5, 0.001, 0.0001)),
        "problem2": online_problem("dsgt", 20000, dsgt(4000, 0.001)),
        "problem3": online_problem("dsgd", 20000, dsgd(4000, 0.001, 0.001)),
    }}
# the PAPER run with the reference's precision (float64 everywhere, csrc/mlp_f64.cu forward/backward)
configs["dist_online_dense_PAPER_f64.yaml"] = copy.deepcopy(configs["dist_online_dense_PAPER.yaml"])
configs["dist_online_dense_PAPER_f64.yaml"]["experiment"].update(name="dist_online_dense_PAPER_f64", dtype="float64")
configs["dist_online_dense_anim.yaml"] = {
    "experiment": online_exp("dist_online_dense_anim", 15000, False),
    "problem_configs": {"problem1": online_problem(
        "dinno", 12500, dinno(4000, 0.3, 1.0004, 5, 0.001, 0.0001),
        metrics=DENSE_METRICS + ["current_position", "current_graph"], mesh_end=False)}}
configs["dist_dense_v2.yaml"] = {
    "experiment": {"name": "dist_dense_v2", "output_metadir": "../results/", "writeout": True, "use_cuda": True,
                   "data": dict(LIDAR, clipped_lidar=False, num_scans=3000, spline_res=80, num_validation_scans=500),
                   "loss": "BCE", "graph": {"num_nodes": 6, "type": "random", "p": 0.75, "gen_attempts": 10},
                   "model": dict(FOURIER),
                   "individual_training": {"train_solo": False, "optimizer": "adam", "lr": 0.005, "epochs": 6,
                                           "train_batch_size": 10000, "val_batch_size": 10000, "verbose": True}},
    "problem_configs": {"problem1": {
        "problem_name": "dinno", "train_batch_size": 8000, "val_batch_size": 10000, "verbose_evals": True,
        "metrics": ["forward_pass_count", "validation_loss", "consensus_error", "mesh_grid_density", "current_epoch"],
        "metrics_config": {"evaluate_frequency": 20},
        "optimizer_config": dinno(1750, 0.5, 1.0, 5, 0.001, 0.001, decay="constant")}}}
# small self-contained variants on the procedural floor plan (no data files needed)
configs["dist_online_dense_synthetic.yaml"] = copy.deepcopy(configs["dist_online_dense_PAPER.yaml"])
e = configs["dist_online_dense_synthetic.yaml"]["experiment"]
e["name"] = "dist_online_dense_synthetic"
e["data"].update(data_dir="synthetic", synthetic_paths=8, num_nodes=8, num_scans_in_window=200, spline_res=20,
                 num_validation_scans=200, border_width=8)
e["individual_training"]["train_solo"] = False
for pc in configs["dist_online_dense_synthetic.yaml"]["problem_configs"].values():
    pc["comm_radius"] = 350.0
    pc["optimizer_config"]["outer_iterations"] = 400

HEADER = "# generated by scripts/make_configs.py — schema: SURVEY.md Appendix A / utils/config.py\n"
for name, conf in configs.items():
    with open(os.path.join(OUT, name), "w") as f:
        f.write(HEADER)
        yaml.safe_dump(conf, f, sort_keys=False, default_flow_style=None)
print("wrote", sorted(configs))
