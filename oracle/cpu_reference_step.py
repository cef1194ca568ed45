"""CPU port of the reference's training step — TEST / BASELINE INFRASTRUCTURE ONLY (see oracle/pfn_oracle.py header).

This is what `bench.py --impl reference` and the `cpu_baseline` leg time on the GPU box's host cores (kind "port":
/root/reference does not travel to the GPU box, and its priors need gpytorch which is not installed anywhere).
It follows the reference's own execution path, not the engine's shortcuts:
  * GP prior draw: dense RBF kernel + Cholesky with gpytorch's jitter escalation + matmul (priors/fast_gp.py:48-56)
  * dense [T,T] float mask built on the host every step (transformer.py:35-41,65)
  * nn.TransformerEncoder (post-norm, GELU) over all T rows, decoder on all rows then sliced (transformer.py:84-91)
  * FullSupportBarDistribution in plain torch ops (bar_distribution.py:89-108), mean loss, clip 1.0, Adam (train.py:92-97)
"""
import math
import time

import torch
from torch import nn

from . import pfn_oracle as O


class RefStyleModel(nn.Module):
    def __init__(self, F, E, H, nhid, L, n_out):
        super().__init__()
        self.encoder = nn.Linear(F, E)
        self.y_encoder = nn.Linear(1, E)
        layer = nn.TransformerEncoderLayer(E, H, nhid, 0.0, activation='gelu')
        self.transformer_encoder = nn.TransformerEncoder(layer, L, enable_nested_tensor=False)
        self.decoder = nn.Sequential(nn.Linear(E, nhid), nn.GELU(), nn.Linear(nhid, n_out))
        for l in self.transformer_encoder.layers:   # transformer.py:43-53
            for t in (l.linear2.weight, l.linear2.bias, l.self_attn.out_proj.weight, l.self_attn.out_proj.bias):
                nn.init.zeros_(t)

    def forward(self, x, y, sep):
        mask = O.d_q_mask(len(x), len(x) - sep)                       # built on the host each step, like the reference
        xs, ys = self.encoder(x), self.y_encoder(y.unsqueeze(-1))
        src = torch.cat([xs[:sep] + ys[:sep], xs[sep:]], 0)
        return self.decoder(self.transformer_encoder(src, mask))[sep:]


def psd_safe_cholesky(K):
    """torch.linalg.cholesky with the escalation of gpytorch's psd_safe_cholesky, which the reference's GP draw goes
    through: when a factorisation fails, 1e-6, 1e-5, then 1e-4 is added to the diagonal of the whole batch."""
    eye = torch.eye(K.shape[-1], dtype=K.dtype)
    for jitter in (0.0, 1e-6, 1e-5, 1e-4):
        Lc, info = torch.linalg.cholesky_ex(K + jitter * eye if jitter else K)
        if not info.any():
            return Lc
    raise torch.linalg.LinAlgError("kernel matrix not positive definite even with jitter 1e-4")


def sample_fast_gp_cpu(B, T, F, hps):
    x = torch.rand(B, T, F)
    ls = torch.full((B, F), float(hps["lengthscale"]))
    K = O.gp_kernel_ref(x, ls, torch.full((B,), float(hps["outputscale"])), torch.full((B,), float(hps["noise"])))
    Lc = psd_safe_cholesky(K)
    y = (Lc @ torch.randn(B, T, 1)).squeeze(-1)
    return x.transpose(0, 1).contiguous(), y.transpose(0, 1).contiguous()


def make_step(T, F, E, H, nhid, L, n_bars, sep, batch, hps, borders, threads=None):
    """Returns (step_fn, model).  step_fn() runs one full reference-style training step on `batch` sequences."""
    if threads:
        torch.set_num_threads(threads)
    model = RefStyleModel(F, E, H, nhid, L, n_bars)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    borders = borders.float().cpu()

    def step():
        x, y = sample_fast_gp_cpu(batch, T, F, hps)
        logits = model(x, y, sep)
        nll = O.bar_nll_ref(logits.reshape(-1, n_bars), y[sep:].flatten(), borders, full_support=True)
        loss = nll.mean()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.)
        opt.step()
        opt.zero_grad()
        return float(loss)

    return step, model


def time_steps(step, steps, warmup):
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return time.perf_counter() - t0
