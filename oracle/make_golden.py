"""Write the reference results the oracle tests compare against (tests/golden/*.npz).

    python oracle/make_golden.py PATH_TO_REFERENCE_CHECKOUT

Runs the unmodified reference (javieryu/nn_distributed_training) on the inputs the tests build and stores what the
tests compare: for the optimizers a sample of every node's parameters plus full-vector signed sums
(tests/test_oracle_optimizers.py), the Metropolis weights and the lidar scans (tests/test_properties.py).
"""
import copy
import importlib
import importlib.util
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def optimizers(ref):
    import test_oracle_optimizers as T
    mods = {n: importlib.import_module(n) for n in ("optimizers.dinno", "optimizers.dsgd", "optimizers.dsgt",
                                                    "problems.dist_mnist_problem", "models.mnist_conv_nn")}
    classes = {"dinno": mods["optimizers.dinno"].DiNNO, "dsgd": mods["optimizers.dsgd"].DSGD,
               "dsgt": mods["optimizers.dsgt"].DSGT}
    torch.set_default_dtype(torch.float64)
    out = {}
    for name, (conf, kind) in T.cases().items():
        base = T.base_model()
        ref_base = mods["models.mnist_conv_nn"].MNISTConvNet(3, 5, 64).double()
        ref_base.load_state_dict(base.state_dict())
        train, val = T._data()
        rp = mods["problems.dist_mnist_problem"].DistMNISTProblem(T._graph(kind), ref_base, torch.nn.NLLLoss(), train,
                                                                  val, torch.device("cpu"), T._prob_conf(copy.deepcopy(conf)))
        ro = classes[conf["alg_name"]](rp, torch.device("cpu"), copy.deepcopy(conf))
        ro.train()
        idx = T.sample_index(base, T.PER_TENSOR[T.strict(conf)])
        rows = {"theta": torch.stack([torch.nn.utils.parameters_to_vector(rp.models[i].parameters()).detach()
                                      for i in range(T.N)])}
        if conf["alg_name"] == "dinno":
            rows["duals"] = torch.stack([ro.duals[i] for i in range(T.N)])
            if not conf["persistant_primal_opt"]:
                out.update({f"{name}/{k}": v for k, v in T.metrics_arrays(rp.metrics).items()})
        if conf["alg_name"] == "dsgt":
            rows["y"] = torch.stack([torch.cat([t.reshape(-1) for t in ro.ylists[i]]) for i in range(T.N)])
        for what, r in rows.items():
            out.update({f"{name}/{what}/{k}": v for k, v in T.summarize(r, idx).items()})
        print(name, flush=True)
    np.savez_compressed(os.path.join(GOLDEN, "oracle_optimizers.npz"), **out)


def properties(ref):
    import test_properties as P
    torch.set_default_dtype(torch.float64)
    graphs = importlib.import_module("utils.graph_generation")
    out = {f"metropolis/{i}": graphs.get_metropolis(g).double().numpy() for i, g in enumerate(P.metropolis_graphs())}
    spec = importlib.util.spec_from_file_location("reflidar", os.path.join(ref, "floorplans", "lidar", "lidar.py"))
    lid = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(lid)
    img, wp = P.lidar_inputs()
    args = (img, 12, 0.2, 15, 1.0, 30, 3)
    full, clipped = lid.Lidar2D(*args, border_width=30), lid.ClippedLidar2D(img, 12, 0.2, 15, border_width=30)
    out["lidar/interp3"] = lid.interpolate_waypoints(wp[:, 0], wp[:, 1], 3)
    traj = P.lidar_trajectory(lid.interpolate_waypoints, wp, full)
    out["lidar/scans"] = np.stack([full.scan(p.reshape(1, 2)) for p in traj])
    out.update({f"lidar/clipped/{i}": clipped.scan(p.reshape(1, 2)) for i, p in enumerate(traj[:4])})
    np.savez_compressed(os.path.join(GOLDEN, "reference_properties.npz"), **out)


if __name__ == "__main__":
    ref = os.path.abspath(sys.argv[1])
    sys.path.insert(0, ref)
    os.makedirs(GOLDEN, exist_ok=True)
    properties(ref)
    optimizers(ref)
