#!/usr/bin/env python
"""bench.py -- jets/s of one LGAE training step (encoder fwd + decoder fwd + chamfer + L1 + full backward) on the
configuration BASELINE.json quotes: 30-particle jets, batch 512 per GPU, maxdim 2, enc 3 3 4 4 / dec 4 4 3 3,
'min&max' latent, chamfer loss, fp64 (cfg-1/cfg-2; cfg-3 is the same step sharded over 2/4/8 GPUs, weak scaling).

    python bench.py --gpus N --steps K --warmup W            # one process per GPU (torchrun for N > 1)
    python bench.py --impl reference ...                     # the reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR                   # + the results of the last timed step as DIR/<name>.npy (float64)

Prints ONE JSON line (rank 0).  `value` = whole-job jets/s with the inputs resident in HBM; `e2e` = the same step
through the public module API with the jets starting in pinned HOST memory and the loss read back every step;
`roofline` = the dominant kernel against the measured fp64 peak; `cpu_baseline` = the CPU oracle (a restatement of
the reference's algorithm in plain torch, oracle/lgae_oracle.py) on a bounded sample, all host cores."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(n=30, batch=512, maxdim=2, enc_channels=[3, 3, 4, 4], dec_channels=[4, 4, 3, 3], tau_s=1, tau_v=8, map_to_latent="min&max",
           num_basis_fn=10, mlp_depth=6, mlp_width=6, l1_lambda=1e-8)
WORKLOAD = "cfg1: LGAE train step, 30p jets, bs 512/GPU, maxdim 2, enc 3-3-4-4 / dec 4-4-3-3, min&max latent, chamfer + 1e-8 L1, fp64"
FP64_PEAK_TFLOPS = 37.1   # measured on this pool's B200 with tools/fp64_peak.cu (DMMA m8n8k4 37.1, DFMA 33.7): profiles/fp64_peak_r01.json


def synthetic_jets(batch, n, seed):
    """SURVEY.md section 8(d): near-massless QCD-like jets."""
    import torch
    g = torch.Generator().manual_seed(seed)
    u = lambda *s: torch.rand(*s, generator=g, dtype=torch.float64)
    pt = 0.2 * u(batch, n) ** 3 + 1e-3
    eta, phi, m = 0.8 * u(batch, n) - 0.4, 0.8 * u(batch, n) - 0.4, 1e-6 * u(batch, n)
    e = torch.sqrt((pt * torch.cosh(eta)) ** 2 + m ** 2)
    return torch.stack([e, pt * torch.cos(phi), pt * torch.sin(phi), pt * torch.sinh(eta)], -1)


def build_models(device, seed=0):
    import torch
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    torch.manual_seed(seed)
    common = dict(maxdim=[CFG["maxdim"]], num_basis_fn=CFG["num_basis_fn"], max_zf=[1], weight_init="randn", level_gain=[1.0],
                  activation="leakyrelu", mlp=True, mlp_depth=CFG["mlp_depth"], mlp_width=CFG["mlp_width"], device=torch.device("cpu"),
                  dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=CFG["n"], tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=CFG["tau_s"],
                     tau_latent_vectors=CFG["tau_v"], num_channels=CFG["enc_channels"], jet_features=False,
                     map_to_latent=CFG["map_to_latent"], **common)
    dec = LGNDecoder(tau_latent_scalars=2 * CFG["tau_s"], tau_latent_vectors=2 * CFG["tau_v"], num_output_particles=CFG["n"],
                     tau_output_scalars=1, tau_output_vectors=1, num_channels=CFG["dec_channels"], cg_dict=enc.cg_dict, **common)
    return enc.to(device), dec.to(device)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return None
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
            out, _ = self.p.communicate()
        sm, smax, reasons = [], 0, set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6 or not f[0].isdigit():
                continue
            sm.append(int(f[0]))
            smax = max(smax, int(f[1]))
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


REF = os.path.join(ROOT, "baseline", "_ref")        # the unmodified reference, copied by tools/setup_reference.py (git-ignored, ships with gpurun)
STUBS = os.path.join(ROOT, "baseline", "stubs")     # matplotlib / jetnet stand-ins the reference's `utils` package imports at module top


def bench_config(world, batch):
    """`config` of the JSON line, identical for both arms."""
    return {"workload": WORKLOAD, "global_batch": batch * world, "parallelism": f"dp{world}", "l2": "flushed (256 MB write) between timed steps"}


def oracle_step(enc_sd_in, dec_sd_in, p4, steps=1, warmup=0, threads=None):
    """The CPU oracle (oracle/lgae_oracle.py: the reference's algorithm restated in plain torch, pinned to the reference's golden
    vectors) on the given state dicts and jets: the CHECKER of the bench line's `parity` object and, when the reference copy is
    absent, the CPU baseline.  Returns (median seconds per step, dict of results of the last step)."""
    import torch
    from oracle import lgae_oracle as orc
    torch.set_num_threads(threads or os.cpu_count())
    enc_sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in enc_sd_in.items()}
    dec_sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in dec_sd_in.items()}
    ecfg = dict(num_channels=CFG["enc_channels"], maxdim=[2], max_zf=[1], map_to_latent=CFG["map_to_latent"])
    dcfg = dict(num_channels=CFG["dec_channels"], maxdim=[2], max_zf=[1])
    pn, _ = orc.normalize_p4_overall_max(p4.cpu())
    times, res = [], None
    for it in range(warmup + steps):
        for sd in (enc_sd, dec_sd):
            for v in sd.values():
                v.grad = None
        t0 = time.perf_counter()
        loss, latent, recon = orc.training_step(enc_sd, dec_sd, ecfg, dcfg, {"p4": pn}, l1_lambda=CFG["l1_lambda"], get_real_method="sum")
        loss.backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        res = {"loss": loss.detach(), "latent": {k: v.detach() for k, v in latent.items()}, "recon": recon.detach(),
               "grads_enc": {k: v.grad for k, v in enc_sd.items()}, "grads_dec": {k: v.grad for k, v in dec_sd.items()}}
    return statistics.median(times), res


def reference_models(device):
    """The UNMODIFIED reference's LGNEncoder / LGNDecoder (baseline/_ref/lgn), built with the constructor arguments of
    utils/initialize.py:91-141.  This repository's own `lgn` shim must not be importable in this process."""
    import torch
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or ".") != ROOT]
    sys.path.insert(0, STUBS)
    sys.path.insert(0, REF)
    import lgn.models   # noqa: F401  (first: the reference's import-order quirk, SURVEY.md appendix C.2)
    from lgn.models import LGNDecoder, LGNEncoder
    assert os.path.abspath(lgn.models.__file__).startswith(REF), lgn.models.__file__
    assert "lgn_autoencoder_b200" not in sys.modules
    torch.manual_seed(0)
    common = dict(maxdim=[CFG["maxdim"]], num_basis_fn=CFG["num_basis_fn"], max_zf=[1], weight_init="randn", level_gain=[1.0],
                  activation="leakyrelu", mlp=True, mlp_depth=CFG["mlp_depth"], mlp_width=CFG["mlp_width"], device=device, dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=CFG["n"], tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=CFG["tau_s"],
                     tau_latent_vectors=CFG["tau_v"], num_channels=CFG["enc_channels"], scale=1.0, jet_features=False,
                     map_to_latent=CFG["map_to_latent"], **common)
    dec = LGNDecoder(tau_latent_scalars=2 * CFG["tau_s"], tau_latent_vectors=2 * CFG["tau_v"], num_output_particles=CFG["n"],
                     tau_output_scalars=1, tau_output_vectors=1, num_channels=CFG["dec_channels"], cg_dict=enc.cg_dict, **common)
    return enc, dec


def reference_rate(sample_batch, steps, warmup, device="cpu", threads=None):
    """jets/s of the unmodified reference's training step (utils/train.py:283-327 minus the optimizer: normalize_p4 -> encoder ->
    decoder -> get_real('sum') -> ChamferLoss + 1e-8 L1 -> backward) on `device`, through the reference's own modules."""
    import torch
    torch.set_num_threads(threads or os.cpu_count())
    dev = torch.device(device)
    enc, dec = reference_models(dev)
    from utils.losses.chamfer_loss.chamfer_loss import ChamferLoss
    from utils.normalize_p4 import normalize_p4
    from utils.utils import get_real
    chamfer = ChamferLoss(device=dev)
    p4 = synthetic_jets(sample_batch, CFG["n"], seed=100)
    times = []
    for it in range(warmup + steps):
        enc.zero_grad(set_to_none=True)
        dec.zero_grad(set_to_none=True)
        if dev.type == "cuda":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        pn, _ = normalize_p4(p4.clone(), "overall_max")
        recon = dec(enc({"p4": pn}, covariance_test=False), covariance_test=False)
        loss = chamfer(get_real(recon, "sum"), pn.to(dev)) + CFG["l1_lambda"] * (enc.l1_norm() + dec.l1_norm())
        loss.backward()
        lv = loss.item()   # the reference's loop reads the loss every step (utils/train.py:320)
        if dev.type == "cuda":
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    sec = statistics.median(times)
    peak = torch.cuda.max_memory_allocated() / 2 ** 30 if dev.type == "cuda" else None
    return sample_batch / sec, sec, lv, peak


def reference_noise_floor(n_jets=64):
    """Max-norm relative difference between the unmodified reference on the CPU and on CUDA (stock ATen kernels) for the same
    weights and jets: reconstruction, loss and gradients.  This is the floor any 'matches the reference' tolerance sits on for
    near-massless jets (BASELINE.md section 4)."""
    import torch
    from utils.losses.chamfer_loss.chamfer_loss import ChamferLoss
    from utils.normalize_p4 import normalize_p4
    from utils.utils import get_real
    cpu_models = reference_models(torch.device("cpu"))
    p4 = synthetic_jets(n_jets, CFG["n"], seed=100)
    out = {}
    for dev in ("cpu", "cuda"):
        d = torch.device(dev)
        e, dd = cpu_models if dev == "cpu" else reference_models(d)
        if dev == "cuda":   # same weights: the generator streams differ between devices
            with torch.no_grad():
                for src, dst in zip(cpu_models, (e, dd)):
                    for ps, pd in zip(src.parameters(), dst.parameters(), strict=True):
                        pd.copy_(ps)
        pn, _ = normalize_p4(p4.clone(), "overall_max")
        recon = dd(e({"p4": pn}, covariance_test=False), covariance_test=False)
        loss = ChamferLoss(device=d)(get_real(recon, "sum"), pn.to(d)) + CFG["l1_lambda"] * (e.l1_norm() + dd.l1_norm())
        loss.backward()
        out[dev] = (recon.detach().cpu(), loss.item(), [p.grad.detach().cpu() for m in (e, dd) for p in m.parameters() if p.grad is not None])
    rc, rg = out["cpu"], out["cuda"]
    gmax = max(g.abs().max().item() for g in rc[2])
    return {"jets": n_jets, "recon_rel": ((rc[0] - rg[0]).abs().max() / rc[0].abs().max()).item(), "loss_rel": abs(rc[1] - rg[1]) / abs(rc[1]),
            "grads_rel_to_model_max": max((a - b).abs().max().item() for a, b in zip(rc[2], rg[2])) / gmax}


def run_reference(args):
    """The reference arm: the reference's own implementation of the path on the box's host cores (all threads), one bounded
    step = the full per-GPU batch of the workload.  kind = "reference" (the unmodified code from baseline/_ref) when that copy is
    present, else "port" (the CPU oracle).  With --ref-device cuda the same unmodified code runs on the GPU through stock ATen
    kernels (an extra, informative line: "what a user of the reference gets on this B200 today")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    cores = os.cpu_count()
    peak = None
    have_ref = os.path.isdir(os.path.join(REF, "lgn"))
    if not have_ref and args.ref_device != "cpu":
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref is absent: the unmodified reference cannot run on cuda here"}))
        return
    if have_ref:
        kind = "reference"
        what = f"unmodified reference (baseline/_ref, torch {torch.__version__}) on {args.ref_device}"
        run = lambda n, k, w: reference_rate(n, k, w, device=args.ref_device)[:3]
    else:
        kind = "port"
        what = "CPU oracle (oracle/lgae_oracle.py)"
        g = torch.load(os.path.join(ROOT, "tests", "golden", "cfg1_b3.pt"), weights_only=False)   # reference-made cfg-1 weights

        def run(n, k, w):
            sec = oracle_step(g["enc_state"], g["dec_state"], synthetic_jets(n, CFG["n"], seed=100), k, w)[0]
            return n / sec, sec, None
    # Bounded sample: every step processes `sample` jets of the workload's batch, sized from a probe step so that the
    # whole --steps K --warmup W run ends within a few minutes (the full per-GPU batch when K is small).
    sample = args.batch
    if args.ref_device == "cpu" and (steps + warmup) > 4:
        probe_rate = run(min(64, args.batch), 1, 1)[0]
        sample = int(max(16, min(args.batch, (150.0 * probe_rate / (steps + warmup)) // 16 * 16)))
    rate, sec, _ = run(sample, steps, warmup)
    noise = None
    if args.ref_device != "cpu":
        peak = torch.cuda.max_memory_allocated() / 2 ** 30
        try:
            noise = reference_noise_floor()
        except Exception as e:   # noqa: BLE001  (informative only)
            noise = {"error": repr(e)[:200]}
    on_cpu = args.ref_device == "cpu"
    line = {"impl": "reference", "metric": "jets/sec LGAE fwd+bwd (30p, maxdim 2)", "value": rate, "unit": "jets/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": bench_config(args.gpus, args.batch), "sample": f"{sample} jets per step, {what}",
            "cpu_baseline": {"value": rate, "unit": "jets/s", "cores": cores if on_cpu else 0, "kind": kind,
                             "sample": f"{steps} steps of {sample} jets after {warmup} warm-up, fwd+bwd, fp64, {what}"
                                       + (f", {cores} threads" if on_cpu else f", peak {peak:.1f} GiB")},
            "e2e": {"value": rate, "unit": "jets/s", "h2d_bytes_per_step": 0 if on_cpu else sample * CFG["n"] * 32, "d2h_bytes_per_step": 0 if on_cpu else 8},
            "gpu_launches": 0, "device": args.ref_device}
    if noise is not None:
        line["cpu_vs_cuda_noise_floor"] = noise
    print(json.dumps(line))


def reference_subprocess(extra, timeout=600):
    """Run this script's reference arm in a fresh interpreter (the reference's `lgn` and this repository's `lgn` shim cannot
    live in one process) and parse its JSON line."""
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference"] + extra, capture_output=True, text=True,
                             timeout=timeout, env={k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")})
        for ln in reversed(out.stdout.splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"unavailable": (out.stderr or "no output").strip().splitlines()[-1][:300]}
    except (subprocess.TimeoutExpired, OSError) as e:
        return {"unavailable": repr(e)[:300]}


DUMP_LIMIT_BYTES = 64 * 2 ** 20


def dump_outputs(out_dir, fstep):
    """Write what the step computed in its last run, the results a caller of FusedTrainStep receives, as float64 .npy files:
    loss, recon, latent00, latent11, norm_factor, and grad_encoder / grad_decoder (every parameter's .grad flattened and
    concatenated in named_parameters() order).  The inputs are seeded, so two builds can be compared output for output.  When
    the per-jet arrays would take the files past DUMP_LIMIT_BYTES, they keep a fixed, seeded sample of jets, listed in
    jet_index.npy."""
    import numpy as np
    import torch
    torch.cuda.synchronize()
    out = {"loss": fstep.loss}
    for tag, model in (("encoder", fstep.enc), ("decoder", fstep.dec)):
        out[f"grad_{tag}"] = torch.cat([p.grad.reshape(-1) for _, p in model.named_parameters()])
    per_jet = {"recon": (fstep.recon, 1), "latent00": (fstep.latent00, 1), "latent11": (fstep.latent11, 1), "norm_factor": (fstep.norm_factor, 0)}
    B = fstep.B
    fixed_bytes = sum(t.numel() * 8 for t in out.values()) + 256 * (len(out) + len(per_jet) + 1)   # + .npy headers
    jet_bytes = sum(t.numel() // B * 8 for t, _ in per_jet.values())
    keep = (DUMP_LIMIT_BYTES - fixed_bytes) // (jet_bytes + 8)
    idx = None
    if B > keep:
        idx = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        out["jet_index"] = idx
    for name, (t, axis) in per_jet.items():
        out[name] = t if idx is None else t.index_select(axis, idx.to(t.device))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().to(torch.float64).cpu().numpy())


def extra_cfg3_strong(enc, dec, world, rank, dev, timed, W, K):
    """BASELINE configs[2] as written: GLOBAL batch 4096 sharded over the ranks (strong scaling: 4096 / world jets per GPU)."""
    import torch
    from lgn_autoencoder_b200.train import FusedTrainStep
    G = 4096
    b = G // world
    step = FusedTrainStep(enc, dec, b, l1_lambda=CFG["l1_lambda"], l1_scale=1.0 / world, normalize=True, get_real="sum")
    step.load(synthetic_jets(b, CFG["n"], seed=300 + rank).to(dev))
    for _ in range(W):
        step.run()
    ms, _ = timed(step.run, K)
    step.graph = None
    return {"workload": "cfg3: the cfg1 step data-parallel at GLOBAL batch 4096 (strong scaling)", "global_batch": G, "jets_per_gpu": b,
            "n_gpus": world, "ms_per_step": ms, "value": G / (ms * 1e-3), "unit": "jets/s", "scaling": "strong"}


def extra_module_path(enc, dec, host_p4, dev, world, timed, K):
    """The step as an UNCHANGED caller of the reference's module API gets it (utils/train.py:283-327 through LGNEncoder /
    LGNDecoder forward + torch autograd, no FusedTrainStep): eager launches, one autograd node per model."""
    import torch
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200.train import training_step
    p4 = host_p4.to(dev)
    params = [p for m in (enc, dec) for p in m.parameters()]

    def step():
        for p in params:
            p.grad = None
        loss, _, _ = training_step(enc, dec, p4, l1_lambda=CFG["l1_lambda"], l1_scale=1.0 / world, get_real="sum")
        loss.backward()
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    step()
    torch.cuda.synchronize()
    lib_launches = _lib.launch_count() - n0
    ms, _ = timed(step, max(3, min(K, 50)))
    B = host_p4.shape[0]
    return {"what": "module API + autograd (what the reference's unchanged utils/train.py loop runs), eager", "ms_per_step": ms,
            "value": B * world / (ms * 1e-3), "unit": "jets/s", "library_launches": lib_launches}


def extra_cfg4(dev, rank, world, timed, K):
    """BASELINE configs[3]: the wide maxdim-3 model (enc 6 6 8 8 / dec 8 8 6 6, 'mix' latent map), training step at bs 1024 per GPU
    through the module API (forward + autograd adjoint on this library's kernels), replayed as one CUDA graph."""
    import gc
    import torch
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    from lgn_autoencoder_b200.train import training_step
    B, N, ENC, DEC = 1024, 30, [6, 6, 8, 8], [8, 8, 6, 6]
    torch.manual_seed(0)
    common = dict(maxdim=[3], num_basis_fn=10, max_zf=[1], weight_init="randn", level_gain=[1.0], activation="leakyrelu", mlp=True, mlp_depth=6,
                  mlp_width=6, device=dev, dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=N, tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=1, tau_latent_vectors=8,
                     num_channels=ENC, jet_features=False, map_to_latent="mix", **common)
    dec = LGNDecoder(tau_latent_scalars=1, tau_latent_vectors=8, num_output_particles=N, tau_output_scalars=1, tau_output_vectors=1,
                     num_channels=DEC, cg_dict=enc.cg_dict, **common)
    p4 = synthetic_jets(B, N, seed=2 + rank).to(dev)
    params = [p for m in (enc, dec) for p in m.parameters()]

    def eager():
        for p in params:
            p.grad = None
        loss, _, _ = training_step(enc, dec, p4, get_real="sum")
        loss.backward()
        return loss.detach()

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            eager()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    gc.collect()
    graph = torch.cuda.CUDAGraph()
    for p in params:
        p.grad = None
    with torch.cuda.graph(graph):
        static_loss, _, _ = training_step(enc, dec, p4, get_real="sum")
        static_loss.backward()
    for _ in range(2):
        graph.replay()
    ms, _ = timed(graph.replay, max(3, min(K, 10)))
    mflop = 198.0   # SURVEY.md 8(d): reference-faithful count of cfg-4, fwd + bwd, per jet
    tf = B * mflop * 1e6 / (ms * 1e-3) / 1e12
    out = {"workload": "cfg4: maxdim 3, enc 6-6-8-8 / dec 8-8-6-6, 'mix' latent, bs 1024/GPU, train step (module API + autograd, CUDA graph)",
           "jets_per_gpu": B, "ms_per_step": ms, "value": B * world / (ms * 1e-3), "unit": "jets/s", "mflop_per_jet": mflop, "tflops_per_gpu": tf,
           "frac_of_fp64_peak": tf / FP64_PEAK_TFLOPS, "loss": static_loss.item(), "peak_mem_gib": torch.cuda.max_memory_allocated() / 2 ** 30,
           "parity": "tests/test_models_gpu.py::test_module_forward_backward_matches_reference[cfg4_b2] (same shapes, 2 jets, vs the unmodified reference)"}
    del graph
    return out


def extra_cfg5(dev, rank, world, timed, K):
    """BASELINE configs[4]: forward-only anomaly scoring, 150-particle jets, 8192 jets sharded over the ranks (no communication)."""
    import torch
    from lgn_autoencoder_b200.flop_model import step_flops_per_jet
    from lgn_autoencoder_b200.train import FusedInference
    n0 = CFG["n"]
    CFG["n"] = 150
    try:
        enc, dec = build_models(dev)
        G = 8192
        b = G // world
        inf = FusedInference(enc, dec, b, get_real="sum")
        inf.score(synthetic_jets(b, 150, seed=500 + rank).to(dev))
        for _ in range(2):
            inf.run()
        ms, _ = timed(inf.run, max(3, min(K, 10)))
        fl = step_flops_per_jet(150, CFG["enc_channels"], CFG["dec_channels"], backward=False)
        tf = G * fl / (ms * 1e-3) / 1e12
        return {"workload": "cfg5: encoder + decoder forward + per-jet scores, 150-particle jets, 8192 jets sharded over the GPUs", "global_batch": G,
                "jets_per_gpu": b, "n_gpus": world, "ms_per_pass": ms, "value": G / (ms * 1e-3), "unit": "jets/s", "mflop_per_jet": fl / 1e6,
                "tflops": tf, "frac_of_fp64_peak": tf / (FP64_PEAK_TFLOPS * world), "mean_score": inf.scores.mean().item(),
                "parity": "tests/test_train_step_gpu.py::test_fused_inference_matches_module_forward_and_oracle_at_150_particles"}
    finally:
        CFG["n"] = n0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=CFG["batch"], help="jets per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg3 (global batch 4096) / cfg4 / cfg5 objects of the line")
    ap.add_argument("--ref-device", default="cpu", help="reference arm only: cpu (the baseline) or cuda (stock ATen kernels, informative)")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the results of the last one as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 step")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200.flop_model import level_flops, step_flops_per_jet
    from lgn_autoencoder_b200.train import FusedTrainStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    W, K, B, N = max(args.warmup, 3), args.steps, args.batch, CFG["n"]

    enc, dec = build_models(dev)
    host_p4 = synthetic_jets(B, N, seed=100 + rank).pin_memory()
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)   # > 126 MB L2
    # The public training-step API: static buffers + one CUDA graph per step (lgn_autoencoder_b200/train.py)
    fstep = FusedTrainStep(enc, dec, B, l1_lambda=CFG["l1_lambda"], l1_scale=1.0 / world, normalize=True, use_graph=not args.no_graph, get_real="sum")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        """n steps, each timed with CUDA events on the launching stream; L2 flushed (untimed) between steps."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        barrier()
        t0 = time.perf_counter()
        for a, b in evs:
            flush.zero_()
            a.record()
            fn()
            b.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t[0].item() / n, t[1].item() / n

    # ---- per-kernel durations of one eager step (CUDA events around every launch of the library), rank 0 ----
    fstep.load(host_p4)
    n0 = _lib.launch_count()
    fstep._launch()
    torch.cuda.synchronize()
    launches = _lib.launch_count() - n0          # kernels of one step (the CUDA graph replays exactly these)
    # (every rank runs it: the step contains the gradient all-reduce, so the launch sequences must match across ranks)
    def eager():
        flush.zero_()
        fstep._launch()
    eager()
    kern = _lib.kernel_timings(eager, reps=5)

    # ---- value: jets resident in HBM ----
    sampler = ClockSampler(local) if rank == 0 else None   # clocks / throttle reasons from the warm-up to the end of the e2e loop
    for _ in range(W):
        fstep.run()
    ms_step, _ = timed(fstep.run, K)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fstep)

    # ---- end to end: pinned host jets -> device, loss back to the host, every step ----
    # (the jets of the step sit in pinned host memory; the H2D copy, the step and the D2H copy of the loss are one graph launch)
    fstep.host_p4.copy_(host_p4)

    def e2e_step():
        return fstep.step_host()

    for _ in range(2):
        e2e_step()
    ms_e2e, _ = timed(e2e_step, K)
    clocks = sampler.stop() if sampler else None

    # ---- roofline of the dominant kernel (largest share of the step), against the measured fp64 peak ----
    roofline, table = None, None
    if rank == 0 and kern:
        Kb = 2 * CFG["num_basis_fn"]
        ech, dch = CFG["enc_channels"], CFG["dec_channels"]

        def lvl(chs, enc_side, l):
            return level_flops(N, chs[l], chs[l + 1], Kb, enc_side, CFG["mlp_width"] * 2 * chs[l + 1], CFG["mlp_depth"])
        # algorithmic flops per step of each kernel family (reference-faithful counts, SURVEY.md section 8(d); adjoint = 2 x forward;
        # the last level's MLP is dead in the backward pass)
        fam = {k: 0.0 for k in ("level_fwd", "level_bwd", "radial_fwd", "radial_bwd", "mlp_fwd", "mlp_bwd")}
        executed = {"mlp_fwd": 0.0, "mlp_bwd": 0.0, "level_fwd": 0.0, "level_bwd": 0.0}
        # which fp64 pipe bounds each family, and its busy fraction from this round's `ncu --set full` captures (profiles/)
        pipe = {"level_fwd": "fp64 DFMA", "level_bwd": "fp64 DFMA", "radial_fwd": "fp64 DMMA", "radial_bwd": "fp64 DMMA", "mlp_fwd": "fp64 DMMA",
                "mlp_bwd": "fp64 DMMA"}
        try:
            ncu_pipe = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_pipe.json")))
        except (OSError, ValueError):
            ncu_pipe = {}
        for chs, enc_side in ((ech, True), (dch, False)):
            for l in range(len(chs) - 1):
                f = lvl(chs, enc_side, l)
                cg = f["edge"] + f["aggregate"] + f["power"] + f["mix"]
                fam["level_fwd"] += B * cg
                fam["level_bwd"] += 2 * B * cg
                fam["radial_fwd"] += B * f["radial"]
                fam["radial_bwd"] += 2 * B * f["radial"]
                # the decoder's last-level MLP forward is not run (dead: see `detail.dead_code`) -- its flops are not credited to the
                # mlp_fwd family either (the whole-step figure keeps the reference's full count)
                if enc_side or l < len(chs) - 2:
                    fam["mlp_fwd"] += B * f["mlp"]
                if l < len(chs) - 2:
                    fam["mlp_bwd"] += 2 * B * f["mlp"]
                    # flops the DMMA pipe actually executes: tiles padded to multiples of 8 (widths 36 -> 40, inputs 6 -> 8)
                pad8 = lambda v: 8 * ((v + 7) // 8)
                w_, ni_ = pad8(CFG["mlp_width"] * 2 * chs[l + 1]), pad8(2 * chs[l + 1])
                ex = N * 2 * (ni_ * w_ + (CFG["mlp_depth"] - 1) * w_ * w_ + w_ * ni_)
                if enc_side or l < len(chs) - 2:
                    executed["mlp_fwd"] += B * ex
                if l < len(chs) - 2:
                    executed["mlp_bwd"] += 2 * B * ex
                # flops the level kernels issue (counted from the kernels' inner loops, csrc/lgae_level.cu): the encoder's
                # neighbour loop is 52 DFMA per (i, j, channel) forward and 96 in the adjoint (the structured Y and the shared
                # R_ij = R_ji save ~40 % of the reference's count); the decoder runs the O(N) closed form (~300 / ~700 DFMA per
                # (particle, channel)); the channel mix and its adjoint are executed as counted.  The decoder launches are the
                # ones whose reference-faithful credit (O(N^2)) exceeds what they execute.
                c_in = chs[l]
                mix_ex = f["mix"]
                if enc_side:
                    executed["level_fwd"] += B * (N * N * c_in * 2 * 52 + mix_ex + f["power"])
                    executed["level_bwd"] += B * (N * N * c_in * 2 * 96 + 3 * mix_ex + 2 * f["power"])
                else:
                    executed["level_fwd"] += B * (N * c_in * 2 * 300 + mix_ex + f["power"])
                    executed["level_bwd"] += B * (N * c_in * 2 * 700 + 3 * mix_ex + 2 * f["power"])
        total_ms = sum(n * ms for n, ms in kern.values()) / 5.0
        table = {}
        for name, (n, ms) in sorted(kern.items(), key=lambda kv: -kv[1][0] * kv[1][1]):
            per_step = n / 5.0
            ent = {"launches_per_step": per_step, "ms_per_launch": ms, "share": per_step * ms / total_ms}
            if name in fam:
                ent["tflops"] = fam[name] / (per_step * ms * 1e-3) / 1e12
                ent["frac_of_fp64_peak"] = ent["tflops"] / FP64_PEAK_TFLOPS
                ent["bound"] = pipe[name]
                if name in executed:   # flops the kernel really issues (padded MMA tiles) / peak
                    ent["executed_frac"] = executed[name] / (per_step * ms * 1e-3) / 1e12 / FP64_PEAK_TFLOPS
                if name in ncu_pipe:   # ncu: busy fraction of that pipe over the kernel's duration
                    ent["ncu_pipe_busy"] = ncu_pipe[name]
            table[name] = ent
        top = max((k for k in table if k in fam), key=lambda k: table[k]["share"])
        t = table[top]
        # DRAM bytes per launch of that kernel from this round's `ncu --set full` capture (profiles/r01_traffic.json)
        traffic = None
        try:
            tf_ = "r02_traffic.json" if os.path.exists(os.path.join(ROOT, "profiles", "r02_traffic.json")) else "r01_traffic.json"
            tr = json.load(open(os.path.join(ROOT, "profiles", tf_)))["kernels"][top]
            traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
        except (OSError, KeyError, ValueError):
            pass
        roofline = {"bound": pipe[top], "executed_frac": t.get("executed_frac"), "ncu_pipe_busy": t.get("ncu_pipe_busy"), "kernel": top, "achieved": t["tflops"], "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s",
                    "frac": t["frac_of_fp64_peak"], "traffic": traffic, "kernel_ms": t["ms_per_launch"], "launches_per_step": t["launches_per_step"],
                    "flops_per_launch": fam[top] / t["launches_per_step"],
                    "peak_source": "fp64 pipe: DMMA m8n8k4 37.1 TFLOP/s / DFMA 33.7 TFLOP/s measured with tools/fp64_peak.cu on this pool "
                                   "(profiles/fp64_peak_r01.json; MEASURED_PEAKS.json holds no fp64 figure)",
                    "note": "achieved = reference-faithful algorithmic flops of this kernel family per step / its measured time per step "
                            "(CUDA events around every launch, eager step, L2 flushed); `kernels` lists every kernel of the step"}

    cpu, parity, ref_cuda = None, None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # ---- parity of THIS run's step against the CPU oracle on the same weights and the same 512 jets (the checker) ----
        fstep._bind_grads()
        loss_gpu = fstep.step(host_p4.to(dev)).item()
        sec_o, ref = oracle_step(enc.state_dict(), dec.state_dict(), host_p4, steps=1, warmup=0)

        def rel(a, b):
            a, b = a.detach().double().cpu(), b.detach().double().cpu()
            return ((a - b).abs().max() / b.abs().max()).item()
        gmax = max(v.abs().max().item() for v in list(ref["grads_enc"].values()) + list(ref["grads_dec"].values()))
        gerr = max((p.grad.detach().cpu() - sd[k]).abs().max().item() / gmax
                   for m, sd in ((enc, ref["grads_enc"]), (dec, ref["grads_dec"])) for k, p in m.named_parameters())
        parity = {"vs": "oracle/lgae_oracle.py (pinned to the reference's golden vectors) on the same weights and jets", "jets": B,
                  "loss_rel": abs(loss_gpu - ref["loss"].item()) / abs(ref["loss"].item()), "recon_rel": rel(fstep.recon, ref["recon"]),
                  "latent00_rel": rel(fstep.latent00, ref["latent"][(0, 0)]), "latent11_rel": rel(fstep.latent11, ref["latent"][(1, 1)]),
                  "grads_rel_to_model_max": gerr, "tolerance": 1e-10}
        # ---- CPU baseline: the unmodified reference (fresh interpreter), else the oracle port ----
        r = reference_subprocess(["--batch", str(B), "--steps", "2", "--warmup", "1"])
        if "value" in r:
            cpu = dict(r["cpu_baseline"])
        else:
            cpu = {"value": B / sec_o, "unit": "jets/s", "cores": os.cpu_count(), "kind": "port",
                   "sample": f"1 step of {B} jets ({sec_o:.2f} s), fwd+bwd, torch fp64 on {os.cpu_count()} threads, oracle/lgae_oracle.py",
                   "note": r.get("unavailable")}
        # ---- the unmodified reference on this GPU (stock ATen fp64 kernels): what a user of the reference gets today ----
        r = reference_subprocess(["--batch", str(B), "--steps", "3", "--warmup", "1", "--ref-device", "cuda"])
        ref_cuda = {"value": r["value"], "unit": "jets/s", "ms_per_step": r["ms_per_step"], "sample": r["cpu_baseline"]["sample"],
                    "cpu_vs_cuda_noise_floor": r.get("cpu_vs_cuda_noise_floor")} if "value" in r else r

    # ---- the other configurations of BASELINE.json, as extra objects of the same line (every rank runs them) ----
    extras = {}
    if not args.no_extras:
        fstep.graph = None
        fstep.graph_host = None
        for name, fn in (("module_path", lambda: extra_module_path(enc, dec, host_p4, dev, world, timed, K)), ("cfg3_global4096", lambda: extra_cfg3_strong(enc, dec, world, rank, dev, timed, W, min(K, 30))),
                         ("cfg5", lambda: extra_cfg5(dev, rank, world, timed, K)), ("cfg4", lambda: extra_cfg4(dev, rank, world, timed, K))):
            try:
                extras[name] = fn()
            except Exception as e:   # noqa: BLE001  (an extra must never take the headline line down)
                extras[name] = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()

    if rank == 0:
        jets = B * world
        fl = step_flops_per_jet(N, CFG["enc_channels"], CFG["dec_channels"])
        line = {
            "metric": "jets/sec LGAE fwd+bwd (30p, maxdim 2)", "value": jets / (ms_step * 1e-3), "unit": "jets/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": bench_config(world, B),
            "detail": {"step": "FusedTrainStep: one CUDA graph per step (normalize, encoder, decoder, chamfer, both adjoints, L1, grad all-reduce)"
                               if not args.no_graph else "FusedTrainStep, eager launches",
                       "dead_code": "the decoder's last-level scalar MLP (its output reaches no result of the training step: loss, gradients, "
                                    "reconstruction, latents) is not run, LGAE_KEEP_DEAD_MLP=1 restores it; the flop count stays the reference's",
                       "step_tflops": jets * fl / (ms_step * 1e-3) / 1e12, "step_frac_of_fp64_peak": jets * fl / (ms_step * 1e-3) / 1e12 / (FP64_PEAK_TFLOPS * world),
                       "mflop_per_jet": fl / 1e6},
            "e2e": {"value": jets / (ms_e2e * 1e-3), "unit": "jets/s", "h2d_bytes_per_step": host_p4.numel() * 8, "d2h_bytes_per_step": 8,
                    "ms_per_step": ms_e2e},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "reference_cuda": ref_cuda,
            "kernels": table, **extras,
        }
        print(json.dumps(line))
    if world > 1:
        # the captured step holds NCCL kernels: drop the graph before tearing the communicator down, and never let a slow
        # teardown keep the job alive after the result line is out
        import gc
        import threading
        sys.stdout.flush()
        threading.Timer(20.0, lambda: os._exit(0)).start()
        fstep.graph = None
        fstep.graph_host = None
        gc.collect()
        barrier()
        dist.destroy_process_group()
        os._exit(0)


if __name__ == "__main__":
    main()
