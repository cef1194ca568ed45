"""CPU tests of the host-side mirror of the reference API (no CUDA needed): schedules, samplers, bucket limits,
bar-distribution inference helpers, state_dict compatibility, DataLoader adapter, and loud failure on CPU."""
import os
import random

import pytest
import torch
from torch import nn

import transformerscandobayesianinference_b200 as pfn
from transformerscandobayesianinference_b200 import bar_distribution, encoders, positional_encodings, transformer, utils
from transformerscandobayesianinference_b200.priors import utils as putils
from oracle.make_golden import MODEL_CASES, build_case_weights, checksum

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_schedules_and_samplers_match_reference():
    g = torch.load(os.path.join(GOLD, "utils.pt"))
    opt = torch.optim.SGD([nn.Parameter(torch.zeros(1))], lr=1.0)
    s = utils.get_cosine_schedule_with_warmup(opt, 3, 10)
    got = []
    for _ in range(12):
        got.append(s.get_last_lr()[0]); opt.step(); s.step()
    assert got == pytest.approx(g["cosine"], abs=1e-12)
    assert got[0] == 0.0      # lr is 0 for the whole first epoch when warmup > 0 (reference train.py:56,134)
    opt = torch.optim.SGD([nn.Parameter(torch.zeros(1))], lr=1.0)
    s = utils.get_linear_schedule_with_warmup(opt, 2, 8)
    got = []
    for _ in range(10):
        got.append(s.get_last_lr()[0]); opt.step(); s.step()
    assert got == pytest.approx(g["linear"], abs=1e-12)
    random.seed(1234)
    f = utils.get_weighted_single_eval_pos_sampler(50)
    assert [f() for _ in range(32)] == g["weighted_sep"]
    random.seed(1234)
    f = utils.get_uniform_single_eval_pos_sampler(50)
    assert [f() for _ in range(32)] == g["uniform_sep"]
    m = nn.Linear(1000, 13246)
    assert utils.get_openai_lr(m) == pytest.approx(g["openai_lr"], rel=1e-12)


def test_mask_helper_matches_reference():
    gold = torch.load(os.path.join(GOLD, "mask.pt"))
    for key, ref in gold.items():
        sz, q = map(int, key.split("_"))
        assert torch.equal(transformer.TransformerModel.generate_D_q_matrix(sz, q), ref), key


def test_bucket_limits_and_inference_helpers_match_reference():
    gold = torch.load(os.path.join(GOLD, "bar.pt"))
    lim = bar_distribution.get_bucket_limits(10, ys=gold["limits_from_ys"]["ys"].clone())
    assert torch.equal(lim, gold["limits_from_ys"]["limits"])
    assert torch.allclose(bar_distribution.get_bucket_limits(8, full_range=(-2.0, 6.0)), gold["limits_from_range"])
    for n_bars in (7, 100, 1000):
        e = gold[n_bars]
        bd = bar_distribution.BarDistribution(e["borders"])
        assert bd.num_bars == n_bars
        assert torch.allclose(bd.mean(e["logits"]), e["mean"], atol=1e-5)
        assert torch.allclose(bd.mode(e["logits"]), e["mode"])
        assert torch.allclose(bd.quantile(e["logits"]), e["quantile"], atol=1e-4, equal_nan=True)
        assert torch.allclose(bd.ei(e["logits"], 0.3, True), e["ei_max"], atol=1e-5)
        assert torch.allclose(bd.ei(e["logits"], 0.3, False), e["ei_min"], atol=1e-5)
        fs = bar_distribution.FullSupportBarDistribution(e["borders"])
        assert torch.allclose(fs.mean(e["logits"]), e["mean_full"], atol=1e-5)
    with pytest.raises(AssertionError):
        bar_distribution.BarDistribution(torch.tensor([0., 2., 1.]))


def _my_model(case):
    ctor = lambda enc, yenc: transformer.TransformerModel(enc, case["n_out"], case["E"], case["H"], case["nhid"],
                                                          case["L"], 0.0, y_encoder=yenc)
    return build_case_weights(ctor, case)


@pytest.mark.parametrize("name", ["cfg1_small", "dh128"])
def test_model_construction_reproduces_reference_init(name):
    """Same seed => same weights as the reference model (RNG order, deep-copied layers, zero-init), proven by the
    reference state_dict checksum stored in the golden file."""
    gold = torch.load(os.path.join(GOLD, f"model_{name}.pt"))
    cs = checksum(_my_model(gold["case"]).state_dict())
    assert set(cs) == set(gold["weights_checksum"])
    for k, (s, a) in gold["weights_checksum"].items():
        assert cs[k][0] == pytest.approx(s, rel=1e-9, abs=1e-9) and cs[k][1] == pytest.approx(a, rel=1e-9), k


def test_fresh_model_zero_init_and_identical_layers():
    torch.manual_seed(0)
    m = transformer.TransformerModel(encoders.Linear(3, 64), 10, 64, 2, 128, 3, 0.0, y_encoder=encoders.Linear(1, 64))
    l0, l2 = m.transformer_encoder.layers[0], m.transformer_encoder.layers[2]
    assert l0.linear2.weight.abs().sum() == 0 and l0.self_attn.out_proj.weight.abs().sum() == 0
    assert torch.equal(l0.linear1.weight, l2.linear1.weight) and torch.equal(l0.self_attn.in_proj_weight, l2.self_attn.in_proj_weight)


def test_reference_checkpoints_load_strict():
    """The reference's shipped checkpoints (their key order, shapes and dtypes in golden/checkpoints.pt; the values do not
    matter for a strict load) load into this package's TransformerModel."""
    layout = torch.load(os.path.join(GOLD, "checkpoints.pt"))
    assert len(layout) == 5
    g = torch.Generator().manual_seed(0)
    for fn, entries in layout.items():
        sd = {k: torch.randn(shape, generator=g).to(getattr(torch, dtype)) for k, shape, dtype in entries}
        E = sd["encoder.weight"].shape[0]
        F = sd["encoder.weight"].shape[1]
        nhid = sd["transformer_encoder.layers.0.linear1.weight"].shape[0]
        L = 1 + max(int(k.split(".")[2]) for k in sd if k.startswith("transformer_encoder.layers."))
        n_out = sd["decoder.2.weight"].shape[0]
        m = transformer.TransformerModel(encoders.Linear(F, E), n_out, E, 4, nhid, L, 0.0, y_encoder=encoders.Linear(1, E))
        m.load_state_dict(sd, strict=True)
        assert all(torch.equal(m.state_dict()[k], v) for k, v in sd.items()), fn


def test_forward_on_cpu_fails_loudly():
    m = transformer.TransformerModel(encoders.Linear(1, 32), 5, 32, 2, 64, 1, 0.0, y_encoder=encoders.Linear(1, 32))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m((torch.rand(4, 2, 1), torch.rand(4, 2)), single_eval_pos=2)
    bd = bar_distribution.BarDistribution(torch.linspace(-1, 1, 6))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        bd(torch.zeros(3, 5), torch.zeros(3))


def test_dataloader_adapter_contract():
    calls = []

    def gb(batch_size, seq_len, num_features, scale=1.0):
        calls.append((batch_size, seq_len, num_features, scale))
        x = torch.rand(seq_len, batch_size, num_features)
        y = x.sum(-1) * scale
        return x, y, y

    DL = putils.get_batch_to_dataloader(gb)
    DL.num_outputs = 1
    dl = DL(num_steps=3, batch_size=4, seq_len=5, num_features=2, scale=2.0)
    assert len(dl) == 3 and dl.num_features == 2 and dl.num_outputs == 1 and dl.fuse_x_y is False
    batches = list(dl)
    assert len(batches) == 3 and len(calls) == 3 and calls[0] == (4, 5, 2, 2.0)
    (x, y), t = batches[0]
    assert x.shape == (5, 4, 2) and y.shape == (5, 4) and torch.equal(y, t)
    fused, t = DL.gbm(batch_size=4, seq_len=5, num_features=2, fuse_x_y=True)
    assert fused.shape == (5, 4, 3) and (fused[0, :, -1] == 0).all()
    assert DL.get_batch_method is not None


def test_normalize_binarize_order_helpers():
    torch.manual_seed(0)
    d = torch.randn(50, 3, 2) * 4 + 1
    n = putils.normalize_data(d)
    assert torch.allclose(n.mean(0), torch.zeros(3, 2), atol=1e-5) and torch.allclose(n.std(0), torch.ones(3, 2), atol=1e-3)
    b = putils.Binarize()(torch.tensor([1., 2., 3., 4.]))
    assert b.tolist() == [0., 0., 1., 1.]          # torch.median = lower median
    random.seed(0)
    x, y = torch.rand(6, 1, 2), torch.tensor([3., 1., 2., 6., 5., 4.]).view(6, 1, 1)
    xo, yo = putils.order_by_y(x, y)
    assert sorted(yo.flatten().tolist()) == [1., 2., 3., 4., 5., 6.]


def test_positional_encodings_and_encoders():
    pe = positional_encodings.PositionalEncoding(8, max_len=16)
    assert pe.pe.shape == (16, 1, 8)
    x = torch.zeros(4, 2, 8)
    assert torch.allclose(pe(x)[:, 0, 0], torch.sin(torch.arange(4.)))
    assert positional_encodings.NoPositionalEncoding(8, 16)(x) is x
    assert positional_encodings.LearnedPositionalEncoding(8, 16)(x).shape == x.shape
    assert positional_encodings.PairedScrambledPositionalEncodings(8, 16)(x).shape == x.shape
    ce = encoders.get_Canonical(5)(2, 8)
    assert ce(torch.randint(0, 5, (4, 3, 2))).shape == (4, 3, 8)
    assert encoders.Linear is nn.Linear


def test_install_dropin_registers_reference_module_names():
    import sys
    saved = {k: sys.modules.get(k) for k in ("train", "transformer", "bar_distribution", "priors", "encoders", "utils", "positional_encodings")}
    try:
        mods = pfn.install_dropin()
        import train as t, priors as p, bar_distribution as b  # noqa: E401
        assert t.train is mods["train"].train and hasattr(p, "fast_gp") and hasattr(b, "FullSupportBarDistribution")
        assert hasattr(t, "Losses") and hasattr(t, "get_weighted_single_eval_pos_sampler")
        assert hasattr(p.fast_gp, "DataLoader") and p.fast_gp.DataLoader.num_outputs == 1
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_wgrad_split_factors_fill_the_grid_once():
    """engine._wgrad_splits: one round of work items over the persistent grid (measured optimum, tools/sweep_wgrad_splits.py)."""
    from transformerscandobayesianinference_b200 import _lib, engine
    saved = _lib.num_sms
    _lib.num_sms = lambda device=None: 148
    try:
        n = 512000
        assert engine._wgrad_splits(n, 1536, 512) == 6      # in-proj: 6 x 2 pair tiles
        assert engine._wgrad_splits(n, 1024, 512) == 9      # linear1
        assert engine._wgrad_splits(n, 512, 1024) == 9      # linear2
        assert engine._wgrad_splits(n, 512, 512) == 18      # out-proj
        assert engine._wgrad_splits(64, 512, 512) == 1      # tiny contraction: never split
        for rows, cols in ((1536, 512), (100, 1024), (1024, 100), (512, 1)):
            ks = engine._wgrad_splits(n, rows, cols)
            assert 1 <= ks <= (n // 64) // 8
    finally:
        _lib.num_sms = saved


def test_one_factor_exact_gp_predictive_identity():
    """The identity priors.fast_gp.evaluate relies on: with L = chol(K + noise I) of the FULL matrix and alpha = L^-1 y,
    the prefix-t Gaussian predictive NLL of row t is 1/2 log(2 pi) + log L_tt + alpha_t^2 / 2 (and the squared error of the
    predictive mean is (L_tt alpha_t)^2) -- checked in fp64 against the per-t restatement of reference priors/fast_gp.py:95-116."""
    import math
    from oracle import pfn_oracle as O
    torch.manual_seed(4)
    T, B, F = 24, 3, 2
    x, y = torch.rand(T, B, F, dtype=torch.float64), torch.randn(T, B, dtype=torch.float64)
    ls, os_, noise = 0.4, 1.3, 0.05
    K = O.gp_kernel_ref(x.transpose(0, 1), torch.full((B, F), ls, dtype=torch.float64), torch.full((B,), os_, dtype=torch.float64),
                        torch.full((B,), noise, dtype=torch.float64))
    Lf = torch.linalg.cholesky(K)
    alpha = torch.linalg.solve_triangular(Lf, y.transpose(0, 1).unsqueeze(-1), upper=False).squeeze(-1)
    d = torch.diagonal(Lf, dim1=1, dim2=2)
    nll = (0.5 * math.log(2 * math.pi) + torch.log(d) + 0.5 * alpha ** 2)[:, 1:].transpose(0, 1)
    mse = ((d * alpha) ** 2)[:, 1:].transpose(0, 1)
    assert torch.allclose(nll, O.gp_exact_predictive_ref(x, y, ls, os_, noise), rtol=1e-9, atol=1e-9)
    assert torch.allclose(mse, O.gp_exact_predictive_ref(x, y, ls, os_, noise, use_mse=True), rtol=1e-8, atol=1e-10)


def test_gp_kernel_oracle_known_answers():
    """The GP parts of the oracle cannot be pinned against gpytorch (not installed, no reference vectors): pin them against the
    PUBLISHED closed forms instead (Rasmussen & Williams, GPML: squared exponential eq. 4.9; Matern nu = 1/2, 3/2, 5/2
    eq. 4.14-4.17 -- the formulas gpytorch.kernels.RBFKernel / MaternKernel implement), at hand-computed points, plus the
    semantics the reference relies on: noise on the diagonal only (GaussianLikelihood), outputscale multiplies the kernel
    (ScaleKernel), per-dimension lengthscales divide the inputs (ARD), and psd_safe_cholesky's jitter ladder 1e-6, 1e-5, 1e-4."""
    import math
    from oracle import pfn_oracle as O
    from transformerscandobayesianinference_b200.priors import fast_gp
    x = torch.tensor([[[0.0, 0.0], [1.0, 0.0], [0.0, 2.0]]], dtype=torch.float64)         # one dataset, 3 points, 2 dims
    one = torch.ones(1, dtype=torch.float64)
    ls1 = torch.ones(1, 2, dtype=torch.float64)
    want = {"rbf": math.exp(-0.5), "matern12": math.exp(-1.0), "matern32": (1 + math.sqrt(3)) * math.exp(-math.sqrt(3)),
            "matern52": (1 + math.sqrt(5) + 5.0 / 3.0) * math.exp(-math.sqrt(5))}
    known = {"rbf": 0.60653066, "matern12": 0.36787944, "matern32": 0.48335772, "matern52": 0.52399411}   # 8 significant digits
    for name, v in want.items():
        assert abs(v - known[name]) < 1e-8
        K = O.gp_kernel_ref(x, ls1, 3.0 * one, 0.25 * one, kernel=name)[0]
        assert abs(K[0, 1].item() - 3.0 * v) < 1e-12                         # unit distance, outputscale 3
        assert abs(K[0, 0].item() - (3.0 + 0.25)) < 1e-12                    # k(x,x) = 1, noise on the diagonal only
        assert abs(K[1, 0].item() - K[0, 1].item()) < 1e-15
    # ARD: distance 2 along a dimension with lengthscale 2 is a unit distance again
    K = O.gp_kernel_ref(x, torch.tensor([[1.0, 2.0]], dtype=torch.float64), one, 0 * one, kernel="rbf")[0]
    assert abs(K[0, 2].item() - math.exp(-0.5)) < 1e-12 and abs(K[1, 2].item() - math.exp(-1.0)) < 1e-12
    assert fast_gp._JITTERS == (0.0, 1e-6, 1e-5, 1e-4)


def test_cpu_port_gp_draw_escalates_jitter_like_gpytorch():
    """The CPU port of the reference step (bench.py's CPU baseline) retries a failed Cholesky with psd_safe_cholesky's
    ladder, adding the jitter to the whole batch, and leaves a factorable batch untouched."""
    from oracle import cpu_reference_step as C
    K = torch.stack([torch.ones(6, 6), torch.eye(6)]).double()  # PSD but singular first element: plain Cholesky fails
    assert torch.linalg.cholesky_ex(K).info.any()
    Lc = C.psd_safe_cholesky(K)
    added = (Lc @ Lc.transpose(-1, -2) - K).diagonal(dim1=-2, dim2=-1)
    assert any(torch.allclose(added, torch.full_like(added, j), rtol=1e-6, atol=0) for j in (1e-6, 1e-5, 1e-4))
    assert torch.equal(C.psd_safe_cholesky(torch.eye(3) * 4), torch.eye(3) * 2)


def test_cli_resolves_the_reference_command_line(tmp_path):
    """`python -m ....train` takes the reference script's arguments (reference train.py:151-287): prior / loss / encoder /
    positional-encoding names resolve to this package's classes, `nhid` defaults to 2 * emsize, a yaml `--config` overrides
    defaults and explicit flags override the file."""
    from transformerscandobayesianinference_b200 import train as train_mod
    from transformerscandobayesianinference_b200 import priors
    prior, crit, enc, kw = train_mod.resolve_cli(
        ["gp", "--min_y", "-3", "--max_y", "3", "--num_buckets", "50", "--emsize", "256", "--bptt", "40",
         "--extra_prior_kwargs_dict", "num_features=1", "noise=0.1", "--permutation_invariant_max_eval_pos", "30"])
    assert prior is priors.fast_gp.DataLoader
    assert isinstance(crit, bar_distribution.BarDistribution) and not isinstance(crit, bar_distribution.FullSupportBarDistribution)
    assert crit.borders.numel() == 51 and float(crit.borders[0]) == -3.0 and float(crit.borders[-1]) == 3.0
    assert enc is encoders.Linear and kw["y_encoder_generator"] is encoders.Linear
    assert kw["pos_encoder_generator"] is positional_encodings.PositionalEncoding
    assert kw["nhid"] == 512 and kw["emsize"] == 256 and kw["bptt"] == 40 and kw["lr"] == 1e-3 and kw["dropout"] == 0.0
    assert kw["extra_prior_kwargs_dict"] == {"num_features": 1, "noise": 0.1}
    assert callable(kw["single_eval_pos_gen"]) and 0 <= kw["single_eval_pos_gen"]() < 30
    for k in ("prior", "loss_function", "encoder", "pos_encoder", "min_y", "num_buckets", "config"):
        assert k not in kw                      # everything left is a `train()` keyword
    import inspect
    assert set(kw) <= set(inspect.signature(train_mod.train).parameters)

    cfg = tmp_path / "c.yaml"
    cfg.write_text("epochs: 7\nnlayers: 3\npos_encoder: none\nloss_function: mse\n")
    prior, crit, enc, kw = train_mod.resolve_cli(["mix_gp", "--config", str(cfg), "--nlayers", "4"])
    assert prior is priors.fast_gp_mix.DataLoader and isinstance(crit, nn.MSELoss)
    assert kw["epochs"] == 7 and kw["nlayers"] == 4 and kw["pos_encoder_generator"] is None
    with pytest.raises(NotImplementedError):
        train_mod.resolve_cli(["stroke"])
    with pytest.raises(NotImplementedError):
        train_mod.resolve_cli(["gp", "--min_y", "0", "--max_y", "1", "--encoder", "mlp"])


def test_src_mask_other_than_the_single_eval_pos_mask_is_rejected():
    """reference transformer.py:60-65: a caller may pass the mask explicitly.  The engine accepts exactly the mask it implements
    (then proceeds to the device check) and refuses any other pattern."""
    m = transformer.TransformerModel(nn.Linear(1, 32), 10, 32, 2, 64, 1, 0.0, y_encoder=nn.Linear(1, 32))
    x, y = torch.zeros(6, 2, 1), torch.zeros(6, 2)
    good = m.generate_D_q_matrix(6, 2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):          # accepted -> fails later, on the CPU tensors
        m((x, y), src_mask=good, single_eval_pos=4)
    with pytest.raises(NotImplementedError):
        m((x, y), src_mask=m.generate_D_q_matrix(6, 3), single_eval_pos=4)
    with pytest.raises(NotImplementedError):
        m((x, y), src_mask=torch.zeros(6, 6), single_eval_pos=4)


def test_bench_reference_arm_prints_one_json_line_with_the_engine_arms_metric():
    """The driver divides the engine arm's line by the `--impl reference` line only when both name the same metric / workload:
    stdout carries exactly ONE JSON line, with the engine arm's METRIC string and workload name (BASELINE.json cfg 2 at batch
    512/GPU), the bounded CPU sample stated separately, and zero host<->device bytes.  The arm times the reference's own
    train.train where oracle/_ref was built and the oracle's CPU port of the step otherwise."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    kind = "reference" if os.path.exists(os.path.join(root, "oracle", "_ref", "train.py")) else "port"
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--ref-batch", "2"], capture_output=True, text=True, timeout=600, cwd=root,
                       env=dict(os.environ, PFN_CPU_THREADS="8"))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    sys.path.insert(0, root)
    import bench
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == "seq/s" and d["higher_is_better"] is True
    assert d["config"]["workload"] == bench.workload_name("cfg2", bench.CONFIGS["cfg2"], bench.CONFIGS["cfg2"]["batch"])
    assert d["config"]["global_batch"] == 512 and d["config"]["parallelism"] == "dp1" and d["config"]["bounded_sample_batch"] == 2
    assert d["cpu_baseline"]["kind"] == kind and d["cpu_baseline"]["cores"] == 8 and d["cpu_baseline"]["value"] == d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "seq/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["vs_baseline"] is None


def test_bench_dump_outputs_are_float32_host_arrays_of_bounded_size():
    """bench.py --dump-outputs: the step's results as float32 host tensors; an array over the size bound is replaced by the
    same seeded sample on every run, so the files of two runs (or two builds) compare element for element."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    model = nn.Linear(3, 2)
    out = bench.step_outputs(torch.tensor(1.5, dtype=torch.float64), torch.ones(4, 2), model)
    assert set(out) == {"loss", "losses", "params_sample"}
    assert all(t.dtype == torch.float32 and t.device.type == "cpu" for t in out.values())
    assert out["loss"].item() == 1.5 and out["losses"].shape == (4, 2)
    assert torch.equal(out["params_sample"], torch.cat([model.weight.flatten(), model.bias]).detach())
    big = torch.arange(bench.DUMP_MAX_ELEMS + 10, dtype=torch.float32)
    s = bench.dump_sample(big)
    assert s.numel() == bench.DUMP_MAX_ELEMS and torch.equal(s, bench.dump_sample(big)) and s.unique().numel() == s.numel()
    assert len(out) * bench.DUMP_MAX_ELEMS * 4 <= 64 << 20


def _equal_f32(a, b):
    """Equal up to float32 rounding.  Stored reference values were computed on another CPU, whose vectorised math may round
    the last bit differently; each side lies within 3e-7 of the float64 result."""
    return a.shape == b.shape and torch.allclose(a, b, rtol=0, atol=1e-6)


def test_positional_encodings_equal_the_unmodified_reference_modules():
    """Same seed -> same initial table, same output, same randperm consumption, same state-dict keys, for all four classes
    (reference positional_encodings.py:13-62; its outputs in golden/ref_modules.pt)."""
    from oracle.make_golden import PE_CLASSES
    gold = torch.load(os.path.join(GOLD, "ref_modules.pt"))["positional_encodings"]
    x = gold["x"]
    for name in PE_CLASSES:
        ref = gold[name]
        torch.manual_seed(11); a = getattr(positional_encodings, name)(12, 20)
        assert list(a.state_dict()) == list(ref["state"])
        for k, v in ref["state"].items():
            assert _equal_f32(a.state_dict()[k], v), (name, k)
        a.load_state_dict(ref["state"], strict=True)
        torch.manual_seed(5); ya = a(x)
        assert _equal_f32(ya, ref["out"]), name
        torch.manual_seed(5); a(x); ra = torch.rand(4)
        assert torch.equal(ra, ref["rand_after"]), f"{name}: RNG consumption differs"
    with pytest.raises(AssertionError):
        positional_encodings.LearnedPositionalEncoding(12, 4)(x)
    with pytest.raises(AssertionError):
        positional_encodings.PairedScrambledPositionalEncodings(12, 9)(x)


def test_utils_helpers_equal_the_unmodified_reference_module():
    """SeqBN, set_locals_in_self, StoreDictKeyPair and every step of both schedules against reference utils.py (its outputs
    in golden/ref_modules.pt)."""
    import argparse
    from oracle.make_golden import SCHEDULE_CASES, SEP_SAMPLERS, sep_sampler_draws
    gold = torch.load(os.path.join(GOLD, "ref_modules.pt"))
    for warm, total, cycles in SCHEDULE_CASES:
        for fn, kw in (("get_cosine_schedule_with_warmup", dict(num_cycles=cycles)), ("get_linear_schedule_with_warmup", {})):
            opt = torch.optim.SGD([nn.Parameter(torch.zeros(1))], lr=0.7)
            s = getattr(utils, fn)(opt, warm, total, **kw)
            cur = []
            for _ in range(total + 5):
                cur.append(s.get_last_lr()[0]); opt.step(); s.step()
            assert cur == gold["schedules"][f"{fn}/{warm}/{total}"], (fn, warm, total)
    for n in (1, 2, 37):
        for fn in SEP_SAMPLERS:
            assert sep_sampler_draws(utils, fn, n) == gold["sep_samplers"][f"{fn}/{n}"], (fn, n)
    ref = gold["seqbn"]
    torch.manual_seed(0); sa = utils.SeqBN(6)
    x = torch.randn(5, 4, 6)
    assert torch.equal(x, ref["x"]), "SeqBN construction consumes the RNG differently"
    assert list(sa.state_dict()) == ref["keys"] and _equal_f32(sa(x), ref["out"])

    class Holder:
        def __init__(self, mod, alpha, beta=3):
            mod.set_locals_in_self(locals())
    h = Holder(utils, 1.5)
    assert h.alpha == 1.5 and h.beta == 3 and h.mod is utils and not hasattr(h, "self")
    ap = argparse.ArgumentParser()
    ap.add_argument("--kw", action=utils.StoreDictKeyPair, nargs="+", default={"d": 1})
    out = (ap.parse_args(["--kw", "a=1", "b=2.5", "c=name", "d=[1,2]", "e=None"]).kw, ap.parse_args([]).kw)
    with pytest.raises(ValueError):
        ap.parse_args(["--kw", "a=1=2"])
    assert out == ({"a": 1, "b": 2.5, "c": "name", "d": [1, 2], "e": None}, {"d": 1})
