"""Python side of the implicit-density MLP kernels: float32 on the tcgen05 kernels (csrc/mlp_tc.cu, bf16 operands),
float64 on the CUDA-core fp64 kernels (csrc/mlp_f64.cu)."""
from __future__ import annotations

import numpy as np
import torch

from . import load_ext
from ..models.spec import MLPSpec

FIRST = {"relu": 0, "sin_relu": 1}
LAST = {"none": 0, "sigmoid": 1}
LOSS = {"BCELoss": 0, "MSELoss": 1, "L1Loss": 2}
TRAIN_KERNEL_READY = True


def shape_supported(spec: MLPSpec) -> bool:
    s = spec.shape
    return (len(s) == 6 and s[0] == 2 and s[1] in (64, 128, 256) and tuple(s[2:5]) == (64, 64, 64) and s[5] == 1
            and spec.first in FIRST and spec.hidden == "relu" and spec.last in LAST)


def supports(spec: MLPSpec, base_loss, dtype=torch.float32) -> bool:
    """Both arms cover the same network family and losses."""
    return (TRAIN_KERNEL_READY and dtype in (torch.float32, torch.float64) and shape_supported(spec)
            and type(base_loss).__name__ in LOSS and getattr(base_loss, "reduction", "mean") == "mean")


F64_TILE = 64       # batch rows per tile of the fp64 kernels


def _op_class(ext, dtype):
    return ext.MlpOp if dtype == torch.float32 else ext.MlpOpF64


def op_dict(arena, spec: MLPSpec, L: int):
    off = [s.offset for s in arena.layout.slots]
    assert len(off) == 10
    return dict(theta=arena.theta.data_ptr(), n_pad=arena.n_pad, L=L, off=off, d_in=spec.shape[0], h1=spec.shape[1],
                first_act=FIRST[spec.first], last_act=LAST[spec.last], scale=float(spec.scale))


class MlpForward:
    """Forward-only evaluation of every local node's network on shared inputs ``x [M, d_in]``, in the arena's dtype."""

    def __init__(self, arena, spec: MLPSpec, L: int, device):
        self.ext = load_ext(required=True)
        self.arena, self.spec, self.L, self.device = arena, spec, L, device
        self.dtype = arena.dtype
        self.sms = torch.cuda.get_device_properties(device).multi_processor_count
        self._cache = {}

    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        x = x.to(self.dtype).contiguous()
        M = x.shape[0]
        out = torch.empty(self.L, M, dtype=self.dtype, device=self.device)
        d = op_dict(self.arena, self.spec, self.L)
        if self.dtype == torch.float32:
            ctas = max(1, min(-(-M // 128), max(1, (2 * self.sms) // max(1, self.L))))
        else:       # one fp64 CTA per SM
            ctas = max(1, min(-(-M // F64_TILE), self.sms // max(1, self.L)))
        d.update(x=x.data_ptr(), n_rows=M, out=out.data_ptr(), fwd_ctas=ctas)
        op = _op_class(self.ext, self.dtype)(d)
        op.forward()
        self._keep = (x, out, op)
        return out


class FusedMLP:
    """Fused training/eval engine of a density problem (FourierNet family) — the analogue of
    ``FusedMnist``: device-resident shards, stateless sampling, per-CTA gradient partials that
    the consensus update kernel sums.  Shards, partials and outputs are kept in the arena dtype."""

    def __init__(self, problem):
        self.pr = problem
        self.ext = load_ext(required=True)
        dev = problem.device
        a, pl = problem.arena, problem.placement
        self.spec = problem.base_model.spec
        self.L, self.n_pad, self.B = pl.L, a.n_pad, problem.train_batch_size
        self.dtype = a.dtype
        self.sms = torch.cuda.get_device_properties(dev).multi_processor_count
        if self.dtype == torch.float32:
            # static partition of the (node, 128-row tile) items over G CTAs; a node spans at most S of them
            tmax = -(-self.B // 128)
            self.G = max(1, min(self.sms, self.L * tmax))
            self.S = -(-self.G // self.L) + 1
        else:
            # grid (S, L), one CTA per SM: CTA s of a node takes its tiles s, s + S, ...
            self.S = max(1, min(-(-self.B // F64_TILE), self.sms // self.L))
            self.G = self.S * self.L
        sh = problem.shards
        self.x = sh.x.to(self.dtype).contiguous()
        self.y = sh.y.to(self.dtype).contiguous()
        self.shard_off = torch.tensor(sh.offsets[:-1], dtype=torch.int32, device=dev)
        self.shard_len = torch.tensor(sh.sizes, dtype=torch.int32, device=dev)
        self.calls = torch.zeros(self.L, dtype=torch.int32, device=dev)
        self.grad_part = torch.zeros(self.L, self.S, self.n_pad, dtype=self.dtype, device=dev)
        self.loss_part = torch.zeros(self.L, self.S, dtype=self.dtype, device=dev)
        self.win_table = self._window_table()
        d = op_dict(a, self.spec, self.L)
        d.update(win_table=None if self.win_table is None else self.win_table.data_ptr())
        d.update(loss=LOSS[type(problem.base_loss).__name__], x=self.x.data_ptr(), y=self.y.data_ptr(),
                 direct=0, batch=self.B, seed=problem.seed, node0=pl.lo,
                 shard_off=self.shard_off.data_ptr(), shard_len=self.shard_len.data_ptr(),
                 calls=self.calls.data_ptr(), grad_part=self.grad_part.data_ptr(),
                 loss_part=self.loss_part.data_ptr(), S=self.S, train_ctas=self.G)
        self.base = d
        self.train_op = _op_class(self.ext, self.dtype)(d)
        self._fwd = MlpForward(a, self.spec, self.L, dev)
        self.host_feed = None

    WIN_MAX = 64

    def _window_table(self):
        """Online problems: per-node tables of one period of the sliding-window stream
        (``data.sampler.OnlineWindowSchedule``) for the in-kernel sampler."""
        pr = self.pr
        dsets = getattr(pr, "_datasets", None)
        if dsets is None or not hasattr(dsets[0], "schedule"):
            return None
        K = self.WIN_MAX
        tab = np.zeros((self.L, 2 + (K + 1) + 2 * K), dtype=np.int64)
        for l, g in enumerate(pr.placement.local_nodes):
            sch = dsets[g].schedule
            wins = [sch.window(0)]
            while True:
                w = sch.window(len(wins))
                if w == wins[0]:
                    break
                wins.append(w)
                if len(wins) > K:
                    raise RuntimeError("online window stream has more than 64 windows per period")
            cum = np.concatenate([[0], np.cumsum([ub - lb for lb, ub, _ in wins])])
            tab[l, 0], tab[l, 1] = len(wins), cum[-1]
            tab[l, 2: 2 + len(cum)] = cum
            tab[l, 2 + K + 1: 2 + K + 1 + len(wins)] = [w[0] for w in wins]
            tab[l, 2 + 2 * K + 1: 2 + 2 * K + 1 + len(wins)] = [w[1] for w in wins]
        return torch.as_tensor(tab, device=pr.device)

    ema_in_kernel = False   # set by the consensus engine when its kernels maintain the loss EMA

    def launch(self):
        self.train_op.train()
        if getattr(self.pr, "track_tloss", False) and not self.ema_in_kernel:
            # device-side EMA of the training loss (capturable: no host sync)
            self.pr._ema_update(self.pr.tloss_local, self.loss_part.sum(1))

    def compute_grads(self) -> torch.Tensor:
        pr = self.pr
        self.launch()
        torch.sum(self.grad_part, dim=1, out=pr.arena.grad)
        self.calls += 1
        pr.count_draws_all(1)
        pr.last_losses = self.loss_part.sum(1)
        if getattr(pr, "track_tloss", False) and self.ema_in_kernel:
            pr._ema_update(pr.tloss_local, pr.last_losses)   # eager API: no consensus kernel follows
        return pr.last_losses

    def sync_calls_from_host(self):
        pl = self.pr.placement
        self.calls.copy_(torch.as_tensor(self.pr.calls[pl.lo: pl.lo + pl.L].astype(np.int32)))

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self._fwd(x)
