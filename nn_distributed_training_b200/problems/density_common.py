"""Shared pieces of the lidar implicit-density problems (offline and online)."""
from __future__ import annotations

import copy
import os

import numpy as np
import torch

from .base import ConsensusProblem, per_sample_loss, sum_of_batch_means
from ..models.spec import MLPSpec


class DensityProblemBase(ConsensusProblem):
    """FourierNet/MLP regression of occupancy density from (x, y).  Model output is squeezed
    before the loss (reference: problems/dist_dense_problem.py:110, dist_online_dense_problem.py:127)."""

    squeeze_output = True

    def _setup_mesh(self, val_set):
        """Every-8th-pixel query mesh used by ``mesh_grid_density``
        (dist_online_dense_problem.py:67-75)."""
        lidar = getattr(val_set, "lidar", None)
        if lidar is None:
            raise ValueError("mesh_grid_density needs a validation set that carries its lidar")
        X, Y = np.meshgrid(lidar.xs, lidar.ys)
        mesh = np.hstack((X[::8, ::8].reshape(-1, 1), Y[::8, ::8].reshape(-1, 1)))
        self.mesh_inputs = torch.as_tensor(mesh, dtype=self.dtype)
        self.metrics["mesh_inputs"] = self.mesh_inputs.clone()   # one-off key, for reconstruction when plotting
        self.mesh_inputs = self.mesh_inputs.to(self.device)

    # ---- forward-only passes ----------------------------------------------------
    def _forward_local(self, x: torch.Tensor, chunk: int = 65536) -> torch.Tensor:
        """Model outputs ``[L, M]`` of every local node on inputs ``x [M, d]``."""
        if self.fused is not None:
            return self.fused.forward(x)
        out = torch.empty(self.placement.L, x.shape[0], device=self.device, dtype=self.dtype)
        with torch.no_grad():
            for l, g in enumerate(self.placement.local_nodes):
                for a in range(0, x.shape[0], chunk):
                    out[l, a: a + chunk] = self.models[g](x[a: a + chunk]).reshape(-1)
        return out

    def _val_losses_local(self) -> torch.Tensor:
        """``[L]`` sums of batch-mean losses over the validation set (no normalisation:
        SURVEY Q10 keeps the reference's definition)."""
        ps_fn = per_sample_loss(self.base_loss)
        x = self.val.inputs(torch.arange(len(self.val), device=self.device), self.dtype)
        y = self.val.y.to(self.dtype)
        yh = self._forward_local(x)
        if ps_fn is not None:
            ps = ps_fn(yh, y.unsqueeze(0).expand_as(yh))
            return sum_of_batch_means(ps, self.val_batch_size)
        out = torch.zeros(yh.shape[0], device=self.device, dtype=self.dtype)
        for a in range(0, x.shape[0], self.val_batch_size):
            for l in range(yh.shape[0]):
                out[l] += self.base_loss(yh[l, a: a + self.val_batch_size], y[a: a + self.val_batch_size])
        return out

    def validate(self, i):
        return self._val_losses_local()[self.placement.local_index(i)]

    def mesh_grid_density(self, i):
        return self._forward_local(self.mesh_inputs)[self.placement.local_index(i)].reshape(-1, 1)

    def _mesh_all(self) -> torch.Tensor:
        """``[N, M, 1]`` predicted densities of every node on the mesh."""
        return self.gather_rows(self._forward_local(self.mesh_inputs)).unsqueeze(-1).cpu()

    def _fused_supported(self) -> bool:
        spec = getattr(self.base_model, "spec", None)
        if not isinstance(spec, MLPSpec):
            return False
        from ..ops import fused_available, mlp_kernel_supports
        return fused_available() and mlp_kernel_supports(spec, self.base_loss, self.dtype)

    def _setup_fused(self):
        from ..ops.mlp_fused import FusedMLP
        self.fused = FusedMLP(self)

    def save_models(self, output_dir):
        if not self.ctx.is_main:
            self.state_dicts()
            return
        path = os.path.join(output_dir, self.conf["problem_name"] + "_models.pt")
        torch.save(self.state_dicts(), path)
