#!/usr/bin/env python
"""Benchmark of the PFN training hot path on B200 (contract: see task statement / DESIGN.md section "Measurement").

    python bench.py --gpus 1 --steps 6 --warmup 3                 # this repo's CUDA engine (default), config cfg2
    python bench.py --config cfg3|cfg4 ...                         # the other single-GPU BASELINE.json configurations
    torchrun --nproc-per-node N ... bench.py --gpus N ...          # data parallel, one rank per GPU
    python bench.py --impl reference --steps 3 --warmup 1          # the UNMODIFIED reference train.train on the host cores
    python bench.py ... --dump-outputs DIR                         # also save the last timed step's results as DIR/*.npy

One "step" = one full training step on one batch of synthetic prior data, driven through the public API
(`train.build_trainer(...)` -> `Trainer.step`, batches from the prior's `DataLoader`):
    prior draw (side stream, one batch ahead) -> embed -> L x {QKV GEMM, masked attention, out-proj, LN, GELU-MLP, LN}
    -> decoder on the query rows -> criterion -> backward -> [NCCL grad all-reduce] -> clip -> Adam.
Metric (BASELINE.json): prior-sampled sequences / second.  Default workload = configs[1] (cfg2): priors.fast_gp,
seq_len 1000, 1 feature, emsize 512, 6 layers, nhid 1024, 4 heads, 100 bars, single_eval_pos 500, bf16, batch 512 per GPU.
"""
import argparse
import contextlib
import json
import os
import random
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "prior-sampled sequences/sec, full training step (prior sample + fwd + bwd + allreduce + clip + Adam)"

GP_HPS = {"noise": 1e-4, "outputscale": 1., "lengthscale": .6, "fast_computations": (False, False, False)}
CONFIGS = {
    # BASELINE.json configs[1]
    "cfg2": dict(prior="fast_gp", T=1000, F=1, E=512, H=4, nhid=1024, L=6, n_out=100, head="bar", sep=500, batch=512,
                 prior_kwargs={"hyperparameters": GP_HPS}),
    # configs[2]: BNN tabular prior, 18 features, 12 layers, binary classification head
    "cfg3": dict(prior="mlp", T=512, F=18, E=512, H=4, nhid=1024, L=12, n_out=1, head="bce", sep=256, batch=512,
                 prior_kwargs={"batch_size_per_gp_sample": 8}),
    # configs[3]: mixture-of-GPs hyperprior, seq_len 2000, 512 datasets per GPU (4096 global on 8 GPUs)
    "cfg4": dict(prior="fast_gp_mix", T=2000, F=1, E=512, H=4, nhid=1024, L=6, n_out=100, head="bar", sep=1000, batch=512,
                 prior_kwargs={"batch_size_per_gp_sample": 64, "hyperparameters": {"fast_computations": (False, False, False)}}),
}


def step_flops(T, B, F, E, nhid, L, n_out, sep):
    """Algorithmic (mask-aware) FLOPs of one training step, SURVEY.md section 8d."""
    dense = T * B * L * (8 * E * E + 4 * E * nhid)
    attn = 4 * E * B * L * (T * sep + (T - sep))
    dec = (T - sep) * B * (2 * E * nhid + 2 * nhid * n_out)
    enc = T * B * 2 * F * E + sep * B * 2 * E
    return 3 * (dense + attn + dec + enc)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(bf16_sustained=p.get("bf16_tflops_sustained"), bf16_burst=p.get("bf16_tflops"), hbm=p.get("hbm_gbs"),
                    source="MEASURED_PEAKS.json (measured)")
    return dict(bf16_sustained=1400.0, bf16_burst=1590.0, hbm=6650.0, source="B200_PROFILING.md fallback")


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_threads():
    """Threads for the CPU arm: torch's intra-op pool scales poorly past a few dozen threads on this small per-step
    problem (128 threads measured 40x slower than 8), so use at most 32 and report the number actually used."""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get("PFN_CPU_THREADS", "32"))))


def workload_name(name, cfg, batch):
    head = {"bar": f"{cfg['n_out']} bars FullSupport", "bce": "BCE head"}[cfg["head"]]
    prior = {"fast_gp": "priors.fast_gp hps(noise 1e-4, os 1, ls .6)", "mlp": "priors.mlp (BNN tabular prior, tanh, 3 layers)",
             "fast_gp_mix": "priors.fast_gp_mix (Gamma hyperpriors, Matern-5/2, 64 per group)"}[cfg["prior"]]
    return (f"{name}: {prior} T={cfg['T']} F={cfg['F']}, emsize {cfg['E']}, {cfg['L']} layers, nhid {cfg['nhid']}, "
            f"{cfg['H']} heads, {head}, single_eval_pos {cfg['sep']}, batch {batch}/GPU")


def mlp_hyperparameters(priors_utils, torch_nn):
    """The 17-tuple of reference tabular.get_mlp_prior_hyperparameters (tabular.py:47-70) for the shipped BNN config
    (TabularEvalSimple.ipynb:154-176): 3 layers, tanh, Gamma init/noise std, no dropout, binary target, order_y."""
    su = priors_utils
    return (lambda: 3, su.scaled_beta_sampler_f(2, 4, 150, 2), torch_nn.Tanh, su.gamma_sampler_f(3.62, .0677),
            su.gamma_sampler_f(1.87, .0528), lambda: 0.0, True, su.scaled_beta_sampler_f(1, 1.6, 18, 2), None, False, None,
            None, None, True, True, lambda n: ([], []), 0.0)


def trainer_args(name, cfg, batch, mods, device, n_steps):
    """(priordataloader_class, criterion, kwargs) for train.build_trainer / the reference's train.train, from a module
    namespace `mods` exposing priors / bar_distribution / encoders (this package or the vendored reference)."""
    priors, bar, enc = mods["priors"], mods["bar_distribution"], mods["encoders"]
    pk = dict(cfg["prior_kwargs"])
    pk["num_features"] = cfg["F"]
    pk["device"] = device
    if "batch_size_per_gp_sample" in pk:          # bounded CPU samples use a smaller batch: keep the group size a divisor
        import math
        pk["batch_size_per_gp_sample"] = math.gcd(int(pk["batch_size_per_gp_sample"]), int(batch))
    if cfg["prior"] == "mlp":
        pk["hyperparameters"] = mlp_hyperparameters(priors.utils, torch.nn)
    prior_mod = getattr(priors, cfg["prior"])
    if cfg["head"] == "bar":
        with contextlib.redirect_stdout(sys.stderr):     # the reference-style helper prints; stdout carries the JSON line only
            ys = prior_mod.get_batch(64, cfg["T"], cfg["F"], **{k: v for k, v in pk.items() if k != "num_features"})[1]
            borders = bar.get_bucket_limits(cfg["n_out"], ys=ys.float().cpu())
        crit = bar.FullSupportBarDistribution(borders)
        crit = crit.to(device)
    else:
        crit = torch.nn.BCEWithLogitsLoss(reduction='none')
    kw = dict(emsize=cfg["E"], nhid=cfg["nhid"], nlayers=cfg["L"], nhead=cfg["H"], dropout=0.0, epochs=1,
              steps_per_epoch=n_steps, batch_size=batch, bptt=cfg["T"], lr=1e-4, warmup_epochs=0,
              y_encoder_generator=enc.Linear, extra_prior_kwargs_dict=pk, single_eval_pos_gen=cfg["sep"],
              gpu_device=device, verbose=False)
    return prior_mod.DataLoader, crit, enc.Linear, kw


DUMP_MAX_ELEMS = 1 << 22      # per dumped array: 16 MB in float32, so the three arrays stay under 64 MB together


def dump_sample(t, n=DUMP_MAX_ELEMS):
    """`t` itself when it has at most `n` elements, else its elements at `n` fixed, seeded positions (flattened)."""
    if t.numel() <= n:
        return t
    idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:n].sort().values
    return t.flatten()[idx.to(t.device)]


def step_outputs(loss, losses, model):
    """What one Trainer.step hands its caller -- the mean loss, the per-position losses -- and the parameters its optimizer
    update left in the model, as float32 host tensors (a fixed sample of the concatenated parameters)."""
    params = torch.cat([p.detach().float().flatten() for p in model.parameters()])
    return {name: dump_sample(t.detach().float()).cpu()
            for name, t in (("loss", loss), ("losses", losses), ("params_sample", params))}


def randomise_zero_init(model, seed=4321):
    """The reference zero-initialises out_proj / linear2 (transformer.py:43-53): at step 0 dattn, du and dqkv would be
    all-zero tensors, which under an active power cap changes clocks (operand toggling).  The bench measures the
    steady state of training, where these weights are dense, so they get small seeded values."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    with torch.no_grad():
        for l in model.transformer_encoder.layers:
            for w in (l.linear2.weight, l.self_attn.out_proj.weight):
                w.copy_((torch.randn(w.shape, generator=g) * (0.5 / w.shape[1] ** 0.5)).to(w.device))


# ----------------------------------------------------------------------------------------------------------------
def reference_cpu_measure(name, cfg, sample_b, steps, warmup, threads):
    """Times the reference's own train.train (unmodified, from oracle/_ref) on the host cores at batch `sample_b`.
    Falls back to the oracle port (kind 'port') when oracle/_ref was not built.  Returns (seq/s, seconds, kind, note)."""
    torch.set_num_threads(threads)
    from oracle import ref_runner as R
    if R.available():
        mods = R.load()
        n = warmup + steps + 1
        with contextlib.redirect_stdout(sys.stderr):
            dl_cls, crit, enc_gen, kw = trainer_args(name, cfg, sample_b, mods, "cpu", n)
            timer = R.StepTimer(dl_cls)
            mods["train"].train(timer.cls, crit, enc_gen, **dict(kw, gpu_device="cpu"))
        dt = timer.seconds(warmup, steps)
        return steps * sample_b / dt, dt, "reference", "unmodified reference train.train / TransformerModel / BarDistribution from oracle/_ref"
    from oracle import cpu_reference_step as C
    assert name == "cfg2", "the oracle port only covers cfg2; build oracle/_ref for the other configs"
    borders = torch.linspace(-4.0, 4.0, cfg["n_out"] + 1)
    step, _ = C.make_step(cfg["T"], cfg["F"], cfg["E"], cfg["H"], cfg["nhid"], cfg["L"], cfg["n_out"], cfg["sep"], sample_b,
                          GP_HPS, borders, threads)
    dt = C.time_steps(step, steps, warmup)
    return steps * sample_b / dt, dt, "port", "oracle/cpu_reference_step.py (oracle/_ref not built)"


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path, all usable host threads, rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    threads = cpu_threads()
    sample_b = args.ref_batch
    value, dt, kind, note = reference_cpu_measure(args.config, cfg, sample_b, args.steps, args.warmup, threads)
    sample = (f"{args.steps} timed steps of the {args.config} shape at batch {sample_b} (per-sequence cost is batch-invariant); "
              f"{note}; torch {torch.__version__} CPU, {threads} threads")
    line = {"impl": "reference", "metric": METRIC, "value": value,
            "unit": "seq/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic (prior draws on the host, random-init weights)",
            # the engine arm's workload (same name, global batch and parallelism keys); each CPU step is a bounded sample of it
            "config": {"workload": workload_name(args.config, cfg, args.batch or cfg["batch"]),
                       "global_batch": (args.batch or cfg["batch"]) * max(1, args.gpus), "parallelism": f"dp{max(1, args.gpus)}",
                       "bounded_sample_batch": sample_b, "precision": "fp32",
                       "api": "unmodified reference train.train on the host cores (rank 0 only)"},
            "cpu_baseline": {"value": value, "unit": "seq/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "seq/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit_line(line)


def gpu_eager_baseline(name, cfg, batch, dev, steps=4, warmup=2):
    """The reference's own eager PyTorch path on THIS GPU (unmodified train.train from oracle/_ref: nn.TransformerEncoder
    + SDPA + ATen, cuSOLVER Cholesky for the prior) in fp32 and under bf16 autocast — the library kernels to beat."""
    from oracle import ref_runner as R
    if not R.available():
        return {"unavailable": "oracle/_ref not built"}
    out = {"batch": batch, "steps": steps, "warmup": warmup, "what": "unmodified reference train.train on cuda (oracle/_ref), eager"}
    mods = R.load()
    sync = lambda: torch.cuda.synchronize(dev)
    for label, ctx in (("fp32", contextlib.nullcontext), ("bf16_autocast", lambda: torch.autocast("cuda", dtype=torch.bfloat16))):
        b = batch
        while b >= 8:
            try:
                torch.cuda.empty_cache()
                n = warmup + steps + 1
                with contextlib.redirect_stdout(sys.stderr):
                    dl_cls, crit, enc_gen, kw = trainer_args(name, cfg, b, mods, str(dev), n)
                    timer = R.StepTimer(dl_cls, sync=sync)
                    with ctx():
                        mods["train"].train(timer.cls, crit, enc_gen, **kw)
                dt = timer.seconds(warmup, steps)
                out[label] = {"seq_per_s": steps * b / dt, "ms_per_step": 1e3 * dt / steps, "batch": b}
                break
            except torch.cuda.OutOfMemoryError:
                b //= 2
        else:
            out[label] = {"unavailable": "out of memory down to batch 8"}
    # which attention kernel did SDPA pick?  (one profiled forward+backward of the reference model at a small batch)
    try:
        from torch.profiler import profile, ProfilerActivity
        ref_t = mods["transformer"]
        m = ref_t.TransformerModel(torch.nn.Linear(cfg["F"], cfg["E"]), cfg["n_out"], cfg["E"], cfg["H"], cfg["nhid"], 1, 0.0,
                                   y_encoder=torch.nn.Linear(1, cfg["E"])).to(dev)
        x = torch.rand(cfg["T"], 8, cfg["F"], device=dev); y = torch.randn(cfg["T"], 8, device=dev)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            with torch.autocast("cuda", dtype=torch.bfloat16):
                m((x, y), single_eval_pos=cfg["sep"]).float().sum().backward()
            torch.cuda.synchronize(dev)
        names = sorted({e.key for e in prof.key_averages() if any(s in e.key.lower() for s in ("fmha", "flash", "attention", "softmax"))})
        out["sdpa_kernels_bf16"] = names[:8]
        del m, x, y
    except Exception as e:   # profiling is informational
        out["sdpa_kernels_bf16"] = [f"profiler failed: {type(e).__name__}: {e}"]
    torch.cuda.empty_cache()
    return out


def run_engine(args):
    import transformerscandobayesianinference_b200 as pkg
    from transformerscandobayesianinference_b200 import _lib as L, bar_distribution, encoders, parallel, priors, train as T_
    import torch.distributed as dist

    rank, world, dev = parallel.init_from_env("cuda")
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the hot path has no CPU fallback)"
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    name = args.config
    cfg = CONFIGS[name]
    B = args.batch or cfg["batch"]
    peaks = load_peaks()
    os.environ["PFN_B200_PRECISION"] = args.precision
    # every generator a prior draws from (the BNN prior samples its hyperparameters with numpy and random): the same
    # arguments give the same inputs, so that outputs of two builds can be compared
    torch.manual_seed(1234); np.random.seed(1234); random.seed(1234)
    mods = {"priors": priors, "bar_distribution": bar_distribution, "encoders": encoders}
    n_total = 2 * (args.warmup + args.steps) + 8
    with contextlib.redirect_stdout(sys.stderr):
        dl_cls, crit, enc_gen, kw = trainer_args(name, cfg, B * world, mods, str(dev), n_total)
        tr = T_.build_trainer(dl_cls, crit, enc_gen, **kw)      # seeds each rank's sampler differently, broadcasts weights
    tr.model.precision = args.precision
    randomise_zero_init(tr.model)
    parallel.broadcast_parameters(tr.model)
    tr.model.train()
    sep = cfg["sep"]
    batches = iter(tr.dl)                                        # prefetching loader: next batch sampled on a side stream
    last = {}

    def train_step():
        data, targets = next(batches)
        last["loss"], last["losses"] = tr.step(data, targets, sep)
        return last["loss"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    bar_distribution.BarDistribution.defer_support_check = True
    for _ in range(args.warmup):
        train_step()
    # ---- device-resident throughput (value)
    sampler = ClockSampler(dev.index or 0)
    if rank == 0:
        sampler.start()
    L.reset_launch_count()
    L.PROFILE_GEMM = [] if rank == 0 else None
    ms = timed(train_step, args.steps)
    gemm_prof_concurrent = L.PROFILE_GEMM
    L.PROFILE_GEMM = None
    launches = L.launch_count()
    clocks = sampler.stop() if rank == 0 else None
    outputs = step_outputs(last["loss"], last["losses"], tr.model) if args.dump_outputs and rank == 0 else None
    # Roofline pass for the dominant kernel: the same steps, but with the prior sampled on the MAIN stream (prefetch off), so
    # that no other kernel runs inside the CUDA-event brackets of the GEMM launches (in the timed region above the sampler
    # of the next batch shares the SMs with them, which inflates the bracketed durations without changing the step time).
    prev_pf = os.environ.get("PFN_B200_PREFETCH")
    os.environ["PFN_B200_PREFETCH"] = "0"
    batches = iter(tr.dl)
    train_step()
    L.PROFILE_GEMM = [] if rank == 0 else None
    n_roof = min(args.steps, 4)
    ms_roof = timed(train_step, n_roof)
    gemm_prof = L.PROFILE_GEMM
    L.PROFILE_GEMM = None
    if prev_pf is None:
        os.environ.pop("PFN_B200_PREFETCH", None)
    else:
        os.environ["PFN_B200_PREFETCH"] = prev_pf
    value = args.steps * B * world / (ms / 1e3)
    del batches

    # ---- end to end with HOST inputs: every step copies that step's prior inputs from pinned host memory (fast_gp: the
    #      uniform x and the normal z the sampler consumes; mlp: the finished x, y batch) and reads the loss back.
    n_host = min(args.steps, 4)
    e2e = None
    if cfg["prior"] in ("fast_gp", "fast_gp_mix"):
        hx = [torch.rand(B, cfg["T"], cfg["F"]).pin_memory() for _ in range(n_host)]
        hz = [torch.randn(B, cfg["T"]).pin_memory() for _ in range(n_host)]
        h2d = hx[0].numel() * 4 + hz[0].numel() * 4
        gb_kw = {k: v for k, v in tr.dl.get_batch_kwargs.items() if k not in ("batch_size", "seq_len", "num_features")}
        gb = getattr(priors, cfg["prior"]).get_batch
        counter = [0]

        def e2e_step():
            i = counter[0] % n_host
            counter[0] += 1
            x, y, tgt = gb(B, cfg["T"], cfg["F"], x=hx[i], z=hz[i], **gb_kw)     # H2D of x, z inside; sampler kernel on device
            loss, _ = tr.step((x, y), tgt, sep)
            return loss.item()
    else:
        with contextlib.redirect_stdout(sys.stderr):
            host = []
            for _ in range(n_host):
                x, y, tgt = priors.mlp.get_batch(B, cfg["T"], cfg["F"], **{k: v for k, v in tr.dl.get_batch_kwargs.items()
                                                                             if k not in ("batch_size", "seq_len", "num_features")})
                host.append((x.cpu().pin_memory(), y.cpu().pin_memory()))
        h2d = host[0][0].numel() * 4 + host[0][1].numel() * 4
        counter = [0]

        def e2e_step():
            i = counter[0] % n_host
            counter[0] += 1
            x = host[i][0].to(dev, non_blocking=True)
            y = host[i][1].to(dev, non_blocking=True)
            loss, _ = tr.step((x, y), y, sep)
            return loss.item()
    e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    e2e = {"value": args.steps * B * world / (ms_e2e / 1e3), "unit": "seq/s", "ms_per_step": ms_e2e / args.steps,
           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4}

    if rank != 0:
        return
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for key, t in outputs.items():
            np.save(os.path.join(args.dump_outputs, key + ".npy"), t.numpy())
    flops = step_flops(cfg["T"], B, cfg["F"], cfg["E"], cfg["nhid"], cfg["L"], cfg["n_out"], sep)
    achieved_step = flops * args.steps / (ms / 1e3) / 1e12
    # dominant kernel: the tcgen05 GEMM (all dense-layer launches of the timed region, CUDA events on the launch stream)
    g_flops = sum(r[0] for r in gemm_prof)
    g_ms = sum(r[1].elapsed_time(r[2]) for r in gemm_prof)
    gemm_tf = g_flops / (g_ms / 1e3) / 1e12 if g_ms > 0 else None
    gc_ms = sum(r[1].elapsed_time(r[2]) for r in gemm_prof_concurrent)
    gemm_tf_concurrent = sum(r[0] for r in gemm_prof_concurrent) / (gc_ms / 1e3) / 1e12 if gc_ms > 0 else None
    # DRAM traffic of the same kernel from the committed `ncu --set full` capture of this command (profiles/, not measured live)
    traffic, traffic_src, traffic_alg = None, None, None
    for tname in ("r2_gemm_traffic.json", "r1_gemm_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if os.path.exists(tpath) and name == "cfg2" and B == cfg["batch"] and args.precision == "bf16":
            with open(tpath) as f:
                tj = json.load(f)
            traffic, traffic_src = tj["mean_dram_bytes_per_launch"], "profiles/" + tname
            traffic_alg = tj.get("mean_algorithmic_bytes_per_launch")
            break
    g_bytes = sum(r[3] for r in gemm_prof)
    roofline = {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 GEMM, all launches of the timed steps)",
                "achieved": gemm_tf, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                "frac": (gemm_tf / peaks["bf16_sustained"]) if gemm_tf else None,
                "traffic": traffic, "traffic_unit": "bytes/launch (dram read+write, mean over the captured launches)",
                "traffic_source": traffic_src, "traffic_algorithmic": traffic_alg,
                "algorithmic_bytes_per_launch": g_bytes / max(len(gemm_prof), 1),
                "launches": len(gemm_prof), "kernel_ms_per_step": g_ms / n_roof, "peak_source": peaks["source"] + ", sustained bf16",
                "measured_in": f"{n_roof} extra steps with the prior sampled on the main stream ({ms_roof / n_roof:.2f} ms/step): nothing else runs "
                               "inside the CUDA-event brackets of the GEMM launches",
                "achieved_with_concurrent_sampler": gemm_tf_concurrent,
                "step": {"achieved": achieved_step, "frac": achieved_step / peaks["bf16_sustained"], "flops_per_step": flops}}

    # ---- CPU baseline on a bounded sample, rank 0 only: the unmodified reference train.train on the host cores
    cpu_baseline = None
    if not args.no_cpu_baseline:
        threads = cpu_threads()
        cb = args.ref_batch
        v, dtc, kind, note = reference_cpu_measure(name, cfg, cb, 3, 1, threads)
        cpu_baseline = {"value": v, "unit": "seq/s", "cores": threads, "kind": kind,
                        "sample": f"3 timed steps (+1 warm-up) of the same workload at batch {cb}; {note}; torch {torch.__version__} CPU fp32"}
    eager = None
    if world == 1 and not args.no_eager_baseline:
        del tr
        torch.cuda.empty_cache()
        eager = gpu_eager_baseline(name, cfg, B, dev)

    line = {"metric": METRIC, "value": value,
            "unit": "seq/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32",
            "data": f"synthetic (priors.{cfg['prior']} draws, random weights; out_proj/linear2 seeded non-zero)",
            "config": {"workload": workload_name(name, cfg, B), "global_batch": B * world, "parallelism": f"dp{world}",
                       "l2_policy": "inputs larger than L2 (activations ~0.5 GB per tensor)", "precision": args.precision,
                       "api": "train.build_trainer -> Trainer.step, batches from priors.<prior>.DataLoader (prefetching)"},
            "clocks": clocks, "gpu_launches": launches, "e2e": e2e,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "gpu_eager_baseline": eager}
    emit_line(line)


_REAL_STDOUT = None


def emit_line(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the config's 512)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--ref-batch", type=int, default=4, help="bounded CPU sample: sequences per CPU step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last one's loss, per-position losses and a fixed sample of the "
                         "updated parameters to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs saves the CUDA engine's step (--impl b200)")
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on fd 1 when
    # NCCL_DEBUG is set), so fd 1 points at stderr while the run is in progress and the line goes to the saved descriptor.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_engine(args)
    sys.stdout.flush()
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
