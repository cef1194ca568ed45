"""priors.mlp (BNN tabular prior) against the UNMODIFIED reference priors/mlp.py (statistics of its batches stored by
oracle/make_golden.py in golden/mlp_prior.pt): same host hyper-sampler stream, same per-dataset distribution.  The vectorised
all-models-at-once formulation is checked on CPU here (no kernels involved: it is batched torch ops) and on the GPU through
the public `get_batch`."""
import os

import pytest
import torch

from oracle.make_golden import MLP_B as B, MLP_F as F, MLP_G as G, MLP_T as T
from oracle.make_golden import mlp_prior_hyperparameters as _hp, mlp_prior_stats as _stats, seed_all as _seed
from transformerscandobayesianinference_b200.priors import mlp, utils as su


def _reference_batch(seed):
    return torch.load(os.path.join(os.path.dirname(__file__), "golden", "mlp_prior.pt"))[seed]


def _check(ours, ref):
    # identical host stream => identical per-dataset feature counts and input scaling, exactly balanced median split
    assert torch.equal(ours["used"], ref["used"])
    assert torch.equal(ours["ymean"], ref["ymean"]) and float(ours["ymean"].mean()) == pytest.approx(0.5, abs=0.01)
    assert torch.allclose(ours["xscale"], ref["xscale"], rtol=1e-4)
    assert ours["halves_monotone"] and ref["halves_monotone"]          # order_by_y: both interleaved halves are sorted
    # function class: how predictable y is from the best single feature (two-sample z test on the mean, 4 sigma)
    a, b = ours["maxcorr"], ref["maxcorr"]
    se = (a.var() / len(a) + b.var() / len(b)).sqrt()
    assert abs(a.mean() - b.mean()) <= 4 * se, (float(a.mean()), float(b.mean()), float(se))
    assert abs(a.std() - b.std()) <= 0.05


def test_vectorised_mlp_prior_matches_reference_distribution_cpu():
    ref = _reference_batch(1)
    _seed(1)
    hp = _hp(su)
    x, y, _ = mlp._get_batch_vectorized(mlp._draw_model_specs(B // G, hp), G, T, F, 'cpu', hp, 'normal', 1)
    assert x.shape == (T, B, F) and y.shape == (T, B) and set(y.unique().tolist()) <= {0.0, 1.0}
    _check(_stats(x, y), ref)


def test_per_model_fallback_sees_the_same_models_after_replay():
    """When the vectorised path cannot be used (categorical features), the already-consumed host draws are replayed."""
    hp = _hp(su)
    _seed(3)
    specs = mlp._draw_model_specs(5, hp)
    rp = mlp._replay_hyperparameters(hp, specs)
    again = mlp._draw_model_specs(5, rp)
    assert [(s["hidden_dim"], s["num_features_used"], s["init_std"], s["noise_std"]) for s in specs] == \
           [(s["hidden_dim"], s["num_features_used"], s["init_std"], s["noise_std"]) for s in again]


@pytest.mark.gpu
def test_mlp_prior_device_path_matches_reference_distribution(cuda_device):
    ref = _reference_batch(2)
    _seed(2)
    x, y, t = mlp.get_batch(B, T, F, device='cuda:0', hyperparameters=_hp(su), batch_size_per_gp_sample=G)
    assert x.is_cuda and x.shape == (T, B, F) and torch.equal(y, t)
    _check(_stats(x, y), ref)
    # uniform causes and the regression variant (no binarisation) run through the same chain
    hp = list(_hp(su)); hp[6] = False
    x2, y2, _ = mlp.get_batch(32, 40, F, device='cuda:0', hyperparameters=tuple(hp), batch_size_per_gp_sample=4, sampling='uniform')
    assert torch.isfinite(x2).all() and torch.isfinite(y2).all() and y2.unique().numel() > 2
