"""Oracle tests: our optimizers vs the unmodified reference, fp64, CPU.

Each node's shard holds exactly one batch, so both frameworks see the same
samples every step regardless of their (different) shuffling machinery.

The reference's results are stored in tests/golden/oracle_optimizers.npz
(written by oracle/make_golden.py from the reference's own DiNNO / DSGD / DSGT
classes on the inputs built here): per node, a fixed sample of parameter
coordinates from every tensor of the network, signed sums over contiguous blocks
of the whole parameter vector, and the DiNNO metrics.  The generator imports
cases(), _data(), base_model(), sample_index() and summarize() from this module:
a change to any of them (or to the inputs they build) invalidates the stored
file until it is regenerated.
"""
import copy
import os

import networkx as nx
import numpy as np
import pytest
import torch

from nn_distributed_training_b200.models import MNISTConvNet
from nn_distributed_training_b200.optimizers import DiNNO, DSGD, DSGT
from nn_distributed_training_b200.problems.dist_mnist_problem import DistMNISTProblem

N, B, ROUNDS = 5, 12, 6
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_optimizers.npz")
# sampled coordinates per parameter tensor (all of a smaller tensor): strict runs, which also check the block sums, and
# Adam runs, whose few chaotic coordinates (see _assert_close) rule the sums out
PER_TENSOR = {True: 16, False: 24}
N_BLOCKS = 8            # contiguous blocks of the flat parameter vector with one signed sum each


def dinno_conf(opt):
    return {"alg_name": "dinno", "rho_init": 0.5, "rho_scaling": 1.01, "outer_iterations": ROUNDS,
            "primal_iterations": 2, "primal_optimizer": opt, "persistant_primal_opt": False,
            "primal_lr_start": 0.005, "primal_lr_finish": 0.0005, "lr_decay_type": "log", "profile": False}


DINNO_PERSISTENT = {"alg_name": "dinno", "rho_init": 0.3, "rho_scaling": 1.0, "outer_iterations": ROUNDS,
                    "primal_iterations": 3, "primal_optimizer": "adam", "persistant_primal_opt": True,
                    "primal_lr_start": 0.004, "primal_lr_finish": 0.001, "lr_decay_type": "linear", "profile": False}


def dsgd_conf():
    return {"alg_name": "dsgd", "alpha0": 0.05, "mu": 0.01, "outer_iterations": ROUNDS, "profile": False,
            "mixing_order": "reference"}


def dsgt_conf(init_grads):
    return {"alg_name": "dsgt", "alpha": 0.02, "init_grads": init_grads, "outer_iterations": ROUNDS,
            "profile": False, "mixing_order": "reference"}


KINDS = ["cycle", "wheel", "random"]


def cases():
    """case name -> (optimizer config, graph kind); the keys of the golden file."""
    c = {}
    for kind in KINDS:
        for opt in ("adam", "sgd", "adamw"):
            c[f"dinno_{opt}_{kind}"] = (dinno_conf(opt), kind)
    c["dinno_persistent_cycle"] = (DINNO_PERSISTENT, "cycle")
    for kind in KINDS:
        c[f"dsgd_{kind}"] = (dsgd_conf(), kind)
        for init_grads in (True, False):
            c[f"dsgt_{kind}_{int(init_grads)}"] = (dsgt_conf(init_grads), kind)
    return c


@pytest.fixture(autouse=True)
def _fp64_default():
    """The reference only works with float64 as the global default dtype
    (experiments/dist_mnist_ex.py:19); ours takes dtype from the model."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    yield
    torch.set_default_dtype(old)


def _data(seed=0):
    g = torch.Generator().manual_seed(seed)
    train = [torch.utils.data.TensorDataset(torch.randn(B, 1, 28, 28, generator=g, dtype=torch.float64),
                                            torch.randint(0, 10, (B,), generator=g)) for _ in range(N)]
    val = torch.utils.data.TensorDataset(torch.randn(40, 1, 28, 28, generator=g, dtype=torch.float64),
                                         torch.randint(0, 10, (40,), generator=g))
    return train, val


def _prob_conf(opt_conf):
    return {"problem_name": "t", "train_batch_size": B, "val_batch_size": 16,
            "metrics": ["forward_pass_count", "validation_loss", "consensus_error", "top1_accuracy", "current_epoch"],
            "metrics_config": {"evaluate_frequency": 3}, "optimizer_config": opt_conf}


def _graph(kind):
    if kind == "cycle":
        return nx.cycle_graph(N)
    if kind == "wheel":
        return nx.wheel_graph(N)
    return nx.erdos_renyi_graph(N, 0.6, seed=3)


def base_model():
    torch.manual_seed(0)
    return MNISTConvNet(3, 5, 64, dtype=torch.float64)


def strict(opt_conf):
    return opt_conf.get("primal_optimizer", "sgd") == "sgd"


def sample_index(model, per_tensor):
    """Sorted coordinates of the flat parameter vector: ``per_tensor`` of every parameter tensor (legacy NumPy stream,
    which is frozen across NumPy versions)."""
    rs, idx, off = np.random.RandomState(0), [], 0
    for p in model.parameters():
        n = p.numel()
        idx.append(off + np.sort(rs.permutation(n)[:min(n, per_tensor)]))
        off += n
    return np.concatenate(idx)


def block_edges(n):
    return np.linspace(0, n, N_BLOCKS + 1).astype(np.int64)


def summarize(rows, idx):
    """[N, n] rows -> what the golden file keeps of them: the sampled coordinates, and per block of the row a signed
    sum and the sum of |x|."""
    rows = rows.detach().double()
    e = block_edges(rows.shape[1])
    signed = rows * torch.as_tensor(np.random.RandomState(1).choice([-1.0, 1.0], size=rows.shape[1]))
    return {"sample": rows[:, idx].numpy(),
            "proj": torch.stack([signed[:, a:b].sum(1) for a, b in zip(e[:-1], e[1:])], 1).numpy(),
            "abssum": torch.stack([rows[:, a:b].abs().sum(1) for a, b in zip(e[:-1], e[1:])], 1).numpy()}


def metrics_arrays(metrics):
    """The reference's metric lists as arrays (one row per evaluation)."""
    st = lambda xs: np.stack([torch.as_tensor(x).double().numpy() for x in xs])
    return {"validation_loss": st(metrics["validation_loss"]), "top1_accuracy": st(metrics["top1_accuracy"]),
            "consensus_error_0": st([c[0] for c in metrics["consensus_error"]]),
            "consensus_error_1": st([c[1] for c in metrics["consensus_error"]]),
            "forward_pass_count": np.asarray(metrics["forward_pass_count"], dtype=np.float64),
            "current_epoch": st(metrics["current_epoch"])}


@pytest.fixture(scope="module")
def golden():
    with np.load(GOLDEN) as z:
        return dict(z)


def _run_ours(our_cls, opt_conf, graph):
    base = base_model()
    train, val = _data()
    op = DistMNISTProblem(graph, base, torch.nn.NLLLoss(), train, val, "cpu", _prob_conf(opt_conf), backend="torch")
    oo = our_cls(op, "cpu", copy.deepcopy(opt_conf))
    oo.train()
    return op, oo


def _assert_close(ours, ref, strict, rtol=1e-6, atol=1e-8):
    """Adam divides by sqrt(v)+eps: a parameter whose loss gradient is exactly 0
    on a node (dead ReLU unit, 12 samples) sees only ~1e-17 rounding noise, which
    Adam amplifies by lr/eps per step.  Those few coordinates are chaotic in the
    reference itself, so Adam runs must match on >= 99.9% of coordinates."""
    ours, ref = torch.as_tensor(ours), torch.as_tensor(ref)
    if strict:
        torch.testing.assert_close(ours, ref, rtol=rtol, atol=atol)
        return
    bad = (ours - ref).abs() > atol + rtol * ref.abs()
    assert bad.double().mean().item() < 1e-3, f"{int(bad.sum())} coordinates differ"


def _check_rows(golden, key, ours_rows, is_strict, rtol=1e-6, atol=1e-8):
    """Sampled coordinates under the per-coordinate tolerance; in strict runs also every block's signed sum, within the
    bound the per-coordinate tolerance implies (sum of atol + rtol |ref| over the block)."""
    ours = summarize(ours_rows, sample_index(base_model(), PER_TENSOR[is_strict]))
    _assert_close(ours["sample"], golden[key + "/sample"], is_strict, rtol, atol)
    if is_strict:
        bound = atol * np.diff(block_edges(ours_rows.shape[1])) + rtol * golden[key + "/abssum"]
        err = np.abs(ours["proj"] - golden[key + "/proj"])
        assert (err <= bound).all(), (err.max(), bound.min())


def _theta_rows(op):
    return torch.stack([torch.nn.utils.parameters_to_vector(op.models[i].parameters()).detach() for i in range(N)])


def _check_case(golden, name, our_cls):
    opt_conf, kind = cases()[name]
    op, oo = _run_ours(our_cls, opt_conf, _graph(kind))
    is_strict = strict(opt_conf)
    _check_rows(golden, name + "/theta", _theta_rows(op), is_strict)
    return op, oo, is_strict


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("opt", ["adam", "sgd", "adamw"])
def test_dinno_matches_reference(golden, kind, opt):
    name = f"dinno_{opt}_{kind}"
    op, oo, is_strict = _check_case(golden, name, DiNNO)
    _check_rows(golden, name + "/duals", torch.stack([op.arena.compact(oo.duals[i]) for i in range(N)]), is_strict)
    # metric parity: same evaluation cadence and values
    ours, g = metrics_arrays(op.metrics), lambda k: golden[f"{name}/{k}"]
    assert ours["validation_loss"].shape == g("validation_loss").shape
    np.testing.assert_allclose(ours["validation_loss"], g("validation_loss"), rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(ours["top1_accuracy"], g("top1_accuracy"), rtol=1e-7, atol=1e-7)
    np.testing.assert_allclose(ours["consensus_error_0"], g("consensus_error_0"), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(ours["consensus_error_1"], g("consensus_error_1"), rtol=1e-4, atol=1e-5)
    assert np.array_equal(ours["forward_pass_count"], g("forward_pass_count"))
    assert np.array_equal(ours["current_epoch"], g("current_epoch"))


def test_dinno_persistent_matches_reference(golden):
    _check_case(golden, "dinno_persistent_cycle", DiNNO)


@pytest.mark.parametrize("kind", KINDS)
def test_dsgd_reference_order(golden, kind):
    _check_case(golden, f"dsgd_{kind}", DSGD)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("init_grads", [True, False])
def test_dsgt_reference_order(golden, kind, init_grads):
    name = f"dsgt_{kind}_{int(init_grads)}"
    op, oo, _ = _check_case(golden, name, DSGT)
    _check_rows(golden, name + "/y", torch.stack([op.arena.compact(oo.y[i]) for i in range(N)]), True)
