"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference modules
(/root/reference/{transformer,bar_distribution,utils}.py) on CPU under this container's torch.

Run here (the GPU box has no /root/reference):   python oracle/make_golden.py
The fixtures are small: inputs, seeds and reference OUTPUTS only — model weights are re-created from the recorded
seed by `build_case_weights` (same torch version on both boxes), and a per-tensor checksum of the reference's
state_dict is stored so that tests can prove they rebuilt exactly the same weights.
"""
import importlib.util
import os
import random
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")

MODEL_CASES = {
    # name: dict(T, B, F, E, nhid, L, H, n_out, sep, seed)
    "cfg1_small": dict(T=50, B=8, F=1, E=128, nhid=256, L=2, H=4, n_out=100, sep=25, seed=1234),
    "sep0": dict(T=12, B=3, F=2, E=64, nhid=128, L=2, H=2, n_out=10, sep=0, seed=7),
    "sep_last": dict(T=12, B=3, F=2, E=64, nhid=128, L=2, H=2, n_out=10, sep=11, seed=8),
    "dh128": dict(T=160, B=4, F=1, E=256, nhid=512, L=2, H=2, n_out=100, sep=96, seed=99),
    "feat5_ragged": dict(T=77, B=5, F=5, E=256, nhid=512, L=3, H=2, n_out=200, sep=40, seed=5),
}


# BASELINE.json configurations at their MODEL shape (sequence length, width, depth, heads, bars, single_eval_pos) with a
# small batch so the unmodified reference finishes in seconds on CPU; the per-sequence maths is batch-invariant.
# `head`: "bar" = FullSupportBarDistribution, "bce" = BCEWithLogitsLoss on a binarised target (cfg 3, train.py:84-85).
CONFIG_CASES = {
    "cfg1_b64": dict(T=50, B=64, F=1, E=128, nhid=256, L=2, H=4, n_out=100, sep=25, seed=101, head="bar"),
    "cfg2_b4": dict(T=1000, B=4, F=1, E=512, nhid=1024, L=6, H=4, n_out=100, sep=500, seed=102, head="bar"),
    "cfg3_b4_bar": dict(T=512, B=4, F=18, E=512, nhid=1024, L=12, H=4, n_out=100, sep=256, seed=103, head="bar"),
    "cfg3_b4_bce": dict(T=512, B=4, F=18, E=512, nhid=1024, L=12, H=4, n_out=1, sep=256, seed=104, head="bce"),
    "cfg4_b2": dict(T=2000, B=2, F=1, E=512, nhid=1024, L=6, H=4, n_out=100, sep=1000, seed=105, head="bar"),
}
N_PROBE = 96   # gradient elements stored per parameter tensor (seeded positions), for per-element comparisons

PE_CLASSES = ("NoPositionalEncoding", "PositionalEncoding", "LearnedPositionalEncoding", "PairedScrambledPositionalEncodings")
SCHEDULE_CASES = [(0, 10, 0.5), (3, 10, 0.5), (5, 40, 1.5), (10, 10, 0.5)]     # (warmup, total, cosine cycles)
SEP_SAMPLERS = ("get_weighted_single_eval_pos_sampler", "get_uniform_single_eval_pos_sampler")
MLP_T, MLP_B, MLP_G, MLP_F = 64, 256, 8, 18      # BNN prior batch: seq_len, datasets, datasets per model, features
MLP_SEEDS = (1, 2)


def mlp_prior_hyperparameters(u):
    """The shipped BNN-prior configuration (reference tabular.py:47-70 / TabularEvalSimple.ipynb:154-176); `u` is a
    priors.utils module providing the samplers."""
    return (lambda: 3, u.scaled_beta_sampler_f(2, 4, 150, 2), torch.nn.Tanh, u.gamma_sampler_f(3.62, .0677),
            u.gamma_sampler_f(1.87, .0528), lambda: 0.0, True, u.scaled_beta_sampler_f(1, 1.6, 18, 2), None, False, None,
            None, None, True, True, lambda n: ([], []), 0.0)


def mlp_prior_stats(x, y):
    """Per-dataset statistics of a BNN prior batch: what a different implementation of the same prior must reproduce."""
    x, y = x.double().cpu(), y.double().cpu()
    used = (x.abs().sum(0) > 0).sum(-1).double()
    xc, yc = x - x.mean(0), y - y.mean(0)
    corr = (xc * yc.unsqueeze(-1)).sum(0) / (xc.norm(dim=0) * yc.norm(dim=0).unsqueeze(-1) + 1e-12)
    halves_monotone = all(((y[k::2, i].diff() >= 0).all() or (y[k::2, i].diff() <= 0).all()) for i in range(y.shape[1]) for k in (0, 1))
    return dict(ymean=y.mean(0), used=used, maxcorr=corr.abs().max(-1).values, xscale=x.std(0).sum(-1) / used.clamp(min=1),
                halves_monotone=halves_monotone)


def seed_all(s):
    np.random.seed(s); random.seed(s); torch.manual_seed(s)


def sep_sampler_draws(mod, fn, n):
    """Three fresh samplers drawn once each, then one sampler drawn 20 times, after random.seed(n)."""
    random.seed(n)
    return [getattr(mod, fn)(n)() for _ in range(3)] + [f() for f in [getattr(mod, fn)(n)] for _ in range(20)]


def grad_probe_index(numel, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, numel, (min(N_PROBE, numel),), generator=g)


def case_targets(case, y):
    """Targets of the query rows: y itself for the bar head, a binarised y for the BCE head."""
    t = y[case["sep"]:]
    return (t > 0).float() if case.get("head") == "bce" else t


def _load_ref(name):
    if REF not in sys.path:
        sys.path.insert(0, REF)
    spec = importlib.util.spec_from_file_location(f"ref_{name}", os.path.join(REF, f"{name}.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def build_case_weights(model_ctor, case):
    """Construct a model exactly the way train() does (encoder, y_encoder, then the model), then overwrite the
    reference's zero-initialised tensors (out_proj, linear2) and de-duplicate the deep-copied layers with seeded
    noise so that attention and the MLP actually contribute.  `model_ctor(encoder, y_encoder)` builds the model."""
    torch.manual_seed(case["seed"])
    encoder = torch.nn.Linear(case["F"], case["E"])
    y_encoder = torch.nn.Linear(1, case["E"])
    model = model_ctor(encoder, y_encoder)
    g = torch.Generator().manual_seed(case["seed"] + 1)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if "transformer_encoder" in name or "decoder" in name:
                scale = 0.5 / (p.shape[-1] ** 0.5) if p.dim() == 2 else 0.1
                if "norm" in name and "weight" in name:
                    p.copy_(1.0 + 0.1 * torch.randn(p.shape, generator=g))
                else:
                    p.add_(scale * torch.randn(p.shape, generator=g))
    return model


def case_inputs(case):
    g = torch.Generator().manual_seed(case["seed"] + 2)
    x = torch.rand(case["T"], case["B"], case["F"], generator=g)
    y = torch.randn(case["T"], case["B"], generator=g)
    return x, y


def case_borders(case):
    g = torch.Generator().manual_seed(case["seed"] + 3)
    inner = torch.sort(torch.randn(case["n_out"] - 1, generator=g) * 1.5).values
    return torch.cat([torch.tensor([-6.0]), inner.clamp(-5.9, 5.9), torch.tensor([6.0])]).sort().values


def checksum(sd):
    return {k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in sd.items() if v.is_floating_point()}


def main():
    os.makedirs(OUT, exist_ok=True)
    ref_transformer = _load_ref("transformer")
    ref_bar = _load_ref("bar_distribution")
    ref_utils = _load_ref("utils")
    torch.set_num_threads(8)

    # ---- mask known answers (transformer.py:35-41)
    masks = {f"{sz}_{q}": ref_transformer.TransformerModel.generate_D_q_matrix(sz, q) for sz, q in
             [(6, 2), (5, 6), (4, 0), (4, 4), (1, 1), (7, 3)]}
    torch.save(masks, os.path.join(OUT, "mask.pt"))

    # ---- model forward / loss / grads
    for name, case in MODEL_CASES.items():
        ctor = lambda enc, yenc: ref_transformer.TransformerModel(enc, case["n_out"], case["E"], case["H"], case["nhid"],
                                                                  case["L"], 0.0, y_encoder=yenc)
        model = build_case_weights(ctor, case)
        x, y = case_inputs(case)
        borders = case_borders(case)
        crit = ref_bar.FullSupportBarDistribution(borders)
        model.train()
        logits = model((x, y), single_eval_pos=case["sep"])
        targets = y[case["sep"]:]
        losses = crit(logits.reshape(-1, case["n_out"]), targets.flatten()).view(*logits.shape[:2])
        loss = losses.mean()
        loss.backward()
        grads = {k: p.grad.clone() for k, p in model.named_parameters()}
        torch.save({
            "case": case,
            "weights_checksum": checksum(model.state_dict()),
            "logits": logits.detach().clone(), "losses": losses.detach(), "loss": loss.detach(),
            "grad_checksum": {k: (float(g.double().sum()), float(g.double().abs().sum()), float(g.double().norm()))
                              for k, g in grads.items()},
            "grad_samples": {k: g.flatten()[:16].clone() for k, g in grads.items()},
            "torch_version": str(torch.__version__),
        }, os.path.join(OUT, f"model_{name}.pt"))
        print(name, "loss", float(loss))

    # ---- BASELINE.json configurations at model shape: loss, logits, grad norms and seeded per-element gradient probes
    for name, case in CONFIG_CASES.items():
        ctor = lambda enc, yenc: ref_transformer.TransformerModel(enc, case["n_out"], case["E"], case["H"], case["nhid"],
                                                                  case["L"], 0.0, y_encoder=yenc)
        model = build_case_weights(ctor, case)
        x, y = case_inputs(case)
        model.train()
        logits = model((x, y), single_eval_pos=case["sep"])
        targets = case_targets(case, y)
        if case["head"] == "bar":
            crit = ref_bar.FullSupportBarDistribution(case_borders(case))
            losses = crit(logits.reshape(-1, case["n_out"]), targets.flatten()).view(*logits.shape[:2])
        else:
            crit = torch.nn.BCEWithLogitsLoss(reduction='none')
            losses = crit(logits.flatten(), targets.flatten()).view(*logits.shape[:2])
        loss = losses.mean()
        loss.backward()
        probes = {}
        for i, (k, p) in enumerate(model.named_parameters()):
            idx = grad_probe_index(p.numel(), case["seed"] * 1000 + i)
            probes[k] = (idx, p.grad.flatten()[idx].clone())
        torch.save({
            "case": case,
            "weights_checksum": checksum(model.state_dict()),
            # clone: the logits are a view of the whole (T, B, n_out) output, whose storage torch.save would write in full
            "logits": logits.detach().to(torch.float32).clone(), "losses": losses.detach(), "loss": loss.detach(),
            "grad_checksum": {k: (float(p.grad.double().sum()), float(p.grad.double().abs().sum()), float(p.grad.double().norm()),
                                  float(p.grad.double().abs().max()))
                              for k, p in model.named_parameters()},
            "grad_probes": probes,
            "torch_version": str(torch.__version__),
        }, os.path.join(OUT, f"model_{name}.pt"))
        print(name, "loss", float(loss), flush=True)

    # ---- bar distribution (bar_distribution.py:19-117) incl. edge cases
    g = torch.Generator().manual_seed(42)
    bars = {}
    for n_bars in (1, 7, 100, 1000):
        inner = torch.sort(torch.randn(max(n_bars - 1, 0), generator=g)).values
        borders = torch.cat([torch.tensor([-4.0]), inner.clamp(-3.9, 3.9), torch.tensor([4.0])]).sort().values
        rows = 64
        logits = torch.randn(rows, n_bars, generator=g) * 2
        y = torch.rand(rows, generator=g) * 8 - 4
        y[0], y[1] = borders[0], borders[-1]
        if n_bars > 3:
            y[2], y[3] = borders[2], borders[1]
        entry = {"borders": borders, "logits": logits, "y": y}
        bd = ref_bar.BarDistribution(borders)
        entry["idx"] = bd.map_to_bucket_idx(y.clone())
        entry["nll"] = bd(logits, y.clone())
        entry["mean"] = bd.mean(logits)
        entry["mode"] = bd.mode(logits)
        if n_bars > 1:
            entry["quantile"] = bd.quantile(logits)
            entry["ei_max"] = bd.ei(logits, 0.3, maximize=True)
            entry["ei_min"] = bd.ei(logits, 0.3, maximize=False)
            fs = ref_bar.FullSupportBarDistribution(borders)
            y_out = y.clone()
            y_out[4], y_out[5] = -5.5, 6.25        # outside the support: half-normal tails
            entry["y_full"] = y_out
            entry["nll_full"] = fs(logits, y_out.clone())
            entry["mean_full"] = fs.mean(logits)
        bars[n_bars] = entry
    ys = torch.randn(1003, generator=g)
    bars["limits_from_ys"] = {"ys": ys, "limits": ref_bar.get_bucket_limits(10, ys=ys.clone())}
    bars["limits_from_range"] = ref_bar.get_bucket_limits(8, full_range=(-2.0, 6.0))
    torch.save(bars, os.path.join(OUT, "bar.pt"))

    # ---- utils: schedules + sep sampler stream (utils.py:10-73)
    opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=1.0)
    sched = ref_utils.get_cosine_schedule_with_warmup(opt, 3, 10)
    cos = []
    for _ in range(12):
        cos.append(sched.get_last_lr()[0])
        opt.step()
        sched.step()
    opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=1.0)
    sched = ref_utils.get_linear_schedule_with_warmup(opt, 2, 8)
    lin = []
    for _ in range(10):
        lin.append(sched.get_last_lr()[0])
        opt.step()
        sched.step()
    random.seed(1234)
    s = ref_utils.get_weighted_single_eval_pos_sampler(50)
    weighted = [s() for _ in range(32)]
    random.seed(1234)
    s = ref_utils.get_uniform_single_eval_pos_sampler(50)
    uniform = [s() for _ in range(32)]
    lr_model = torch.nn.Linear(1000, 13246)
    torch.save({"cosine": cos, "linear": lin, "weighted_sep": weighted, "uniform_sep": uniform,
                "openai_lr": ref_utils.get_openai_lr(lr_model), "openai_lr_nparams": sum(p.numel() for p in lr_model.parameters())},
               os.path.join(OUT, "utils.pt"))
    reference_module_fixtures(_load_ref("positional_encodings"), ref_utils)
    checkpoint_layout_fixture()
    mlp_prior_fixture()
    print("golden fixtures written to", OUT)


def reference_module_fixtures(ref_pe, ref_utils):
    """positional_encodings.py (all four classes: initial state, output, RNG consumption) and utils.py (every step of both
    schedules, the sep samplers, SeqBN) -> ref_modules.pt."""
    torch.manual_seed(0)
    x = torch.randn(7, 3, 12)
    pe = {"x": x}
    for name in PE_CLASSES:
        torch.manual_seed(11); m = getattr(ref_pe, name)(12, 20)
        torch.manual_seed(5); out = m(x).detach()
        torch.manual_seed(5); m(x); after = torch.rand(4)
        pe[name] = {"state": m.state_dict(), "out": out, "rand_after": after}
    schedules = {}
    for warm, total, cycles in SCHEDULE_CASES:
        for fn, kw in (("get_cosine_schedule_with_warmup", dict(num_cycles=cycles)), ("get_linear_schedule_with_warmup", {})):
            opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=0.7)
            s = getattr(ref_utils, fn)(opt, warm, total, **kw)
            cur = []
            for _ in range(total + 5):
                cur.append(s.get_last_lr()[0]); opt.step(); s.step()
            schedules[f"{fn}/{warm}/{total}"] = cur
    samplers = {f"{fn}/{n}": sep_sampler_draws(ref_utils, fn, n) for n in (1, 2, 37) for fn in SEP_SAMPLERS}
    torch.manual_seed(0); bn = ref_utils.SeqBN(6)
    bx = torch.randn(5, 4, 6)
    seqbn = {"keys": list(bn.state_dict()), "x": bx, "out": bn(bx).detach()}
    torch.save({"positional_encodings": pe, "schedules": schedules, "sep_samplers": samplers, "seqbn": seqbn},
               os.path.join(OUT, "ref_modules.pt"))


def checkpoint_layout_fixture():
    """State-dict layout (key order and shapes) of the model checkpoints shipped in the reference's results/ ->
    checkpoints.pt; the weights themselves are not needed to check that they load."""
    res = os.path.join(REF, "results")
    layout = {}
    for fn in sorted(os.listdir(res)):
        sd = torch.load(os.path.join(res, fn), map_location="cpu", weights_only=False)[0]
        layout[fn] = [(k, list(v.shape), str(v.dtype).replace("torch.", "")) for k, v in sd.items()]
    torch.save(layout, os.path.join(OUT, "checkpoints.pt"))


def mlp_prior_fixture():
    """Statistics of the reference BNN prior (priors/mlp.py through the vendored oracle/_ref tree) on CPU -> mlp_prior.pt."""
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    from oracle import build_ref, ref_runner
    build_ref.build(verbose=False)
    mods = ref_runner.load()
    stats = {}
    for seed in MLP_SEEDS:
        seed_all(seed)
        x, y, _ = mods["priors"].mlp.get_batch(MLP_B, MLP_T, MLP_F, device='cpu',
                                               hyperparameters=mlp_prior_hyperparameters(mods["priors"].utils),
                                               batch_size_per_gp_sample=MLP_G)
        stats[seed] = mlp_prior_stats(x, y)
    torch.save(stats, os.path.join(OUT, "mlp_prior.pt"))


if __name__ == "__main__":
    main()
