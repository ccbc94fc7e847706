"""One training step of the cfg-1 model (enc 3-3-4-4 / dec 4-4-3-3, 'min&max' latent, MLP 6 x 6, chamfer + 1e-8 L1, fp64) on
150-particle jets through the module API (forward, chamfer and L1, autograd backward), on two paths:
  tiled      the fused forward and the tiled fused adjoint (what LGNEncoder / LGNDecoder run for N > 32);
  composite  the layer-level composite (_forward_generic), forced by marking the tiled adjoint as unavailable.
The composite is timed at the largest power-of-two batch up to --batch that fits in device memory, and says so.

Per path: warm-up, then steps until at least --seconds of measured time, L2 (126 MB) overwritten before every step with a
256 MB write that is not timed; CUDA events around each step.  Also: per-kernel times of the tiled step (lgae_timing_enable),
jets/s, the share of the measured 37.1 TFLOP/s fp64 peak (flop_model.step_flops_per_jet: the reference algorithm's flops), and
parity of both paths against the CPU oracle on two jets with the timed weights.  Prints one JSON document (and writes it to --out).

    python tools/long_jet_bench.py --batch 512 --out long_jet.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CFG = dict(n=150, enc_channels=[3, 3, 4, 4], dec_channels=[4, 4, 3, 3], tau_s=1, tau_v=8, map_to_latent="min&max", num_basis_fn=10,
           mlp_depth=6, mlp_width=6, l1_lambda=1e-8)
FP64_PEAK_TFLOPS = 37.1   # measured with tools/fp64_peak.cu: profiles/fp64_peak_r01.json


def build(dev, seed=0, n=None):
    """The cfg-1 encoder and decoder at CFG["n"] particles (or n)."""
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    n = CFG["n"] if n is None else n
    torch.manual_seed(seed)
    common = dict(maxdim=[2], num_basis_fn=CFG["num_basis_fn"], max_zf=[1], weight_init="randn", level_gain=[1.0], activation="leakyrelu",
                  mlp=True, mlp_depth=CFG["mlp_depth"], mlp_width=CFG["mlp_width"], device=torch.device("cpu"), dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=n, tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=CFG["tau_s"],
                     tau_latent_vectors=CFG["tau_v"], num_channels=CFG["enc_channels"], jet_features=False,
                     map_to_latent=CFG["map_to_latent"], **common)
    dec = LGNDecoder(tau_latent_scalars=2 * CFG["tau_s"], tau_latent_vectors=2 * CFG["tau_v"], num_output_particles=n,
                     tau_output_scalars=1, tau_output_vectors=1, num_channels=CFG["dec_channels"], cg_dict=enc.cg_dict, **common)
    return enc.to(dev), dec.to(dev)


def jets(batch, seed=1):
    from oracle import lgae_oracle as orc
    data = orc.synthetic_jets(batch, CFG["n"], seed=seed, mass_scale=0.05, pad=True)
    pn, _ = orc.normalize_p4_overall_max(data["p4"])
    return {"p4": pn, "labels": data["labels"]}


def set_path(enc, dec, path):
    reason = None if path == "tiled" else "forced composite (benchmark)"
    enc._tiled_reason = dec._tiled_reason = reason


def step(enc, dec, batch):
    from lgn_autoencoder_b200 import fused
    for m in (enc, dec):
        m.zero_grad(set_to_none=True)
    recon = dec(enc(batch))
    loss = fused.chamfer_loss(recon, batch["p4"], "real") + CFG["l1_lambda"] * (enc.l1_norm() + dec.l1_norm())
    loss.backward()
    return loss


def time_path(enc, dec, batch, seconds, warmup):
    flush = torch.empty(32 * 1024 * 1024, dtype=torch.float64, device=batch["p4"].device)   # 256 MB > 126 MB of L2
    for _ in range(warmup):
        step(enc, dec, batch)
    torch.cuda.synchronize()
    times = []
    while sum(times) < seconds * 1e3 or len(times) < 3:
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step(enc, dec, batch)
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return {"steps": len(times), "median_ms": times[len(times) // 2], "min_ms": times[0], "max_ms": times[-1], "total_ms": sum(times)}


def parity(enc, dec, path, dev):
    """Both paths' loss and gradients on two jets against one oracle step with the same weights."""
    from oracle import lgae_oracle as orc
    data = jets(2, seed=7)
    enc_sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in enc.state_dict().items()}
    dec_sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in dec.state_dict().items()}
    ecfg = dict(num_channels=CFG["enc_channels"], maxdim=[2], max_zf=[1], map_to_latent=CFG["map_to_latent"])
    dcfg = dict(num_channels=CFG["dec_channels"], maxdim=[2], max_zf=[1])
    recon = orc.decoder_forward(dec_sd, dcfg, orc.encoder_forward(enc_sd, ecfg, data))
    ref = orc.chamfer_loss(orc.get_real(recon, "real"), data["p4"]) + CFG["l1_lambda"] * (orc.l1_norm(enc_sd) + orc.l1_norm(dec_sd))
    ref.backward()
    set_path(enc, dec, path)
    loss = step(enc, dec, {k: v.to(dev) for k, v in data.items()})
    gmax = max(v.grad.abs().max().item() for sd in (enc_sd, dec_sd) for v in sd.values())
    worst = 0.0
    for m, sd in ((enc, enc_sd), (dec, dec_sd)):
        for k, p in m.named_parameters():
            r = sd[k].grad
            worst = max(worst, (p.grad.cpu() - r).abs().max().item() / max(r.abs().max().item(), 1e-4 * gmax))
    return {"loss_rel_err": abs(loss.item() - ref.item()) / abs(ref.item()), "grad_err_worst_scaled": worst}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("long_jet_bench.py measures on a CUDA device; none is visible")
    from lgn_autoencoder_b200 import _lib, flop_model
    dev = torch.device("cuda:0")
    out = {"workload": f"cfg1 train step through the module API, {CFG['n']}-particle jets, fp64", "device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = f"not read: {e}"
    enc, dec = build(dev)
    assert enc.fused and dec.fused and enc._tiled_reason is None and dec._tiled_reason is None
    flops = flop_model.step_flops_per_jet(CFG["n"], CFG["enc_channels"], CFG["dec_channels"], CFG["num_basis_fn"], CFG["mlp_width"],
                                          CFG["mlp_depth"])
    out["flops_per_jet"] = flops
    for path in ("tiled", "composite"):
        set_path(enc, dec, path)
        b = args.batch
        while True:
            try:
                batch = {k: v.to(dev) for k, v in jets(b).items()}
                r = time_path(enc, dec, batch, args.seconds, args.warmup)
                break
            except torch.cuda.OutOfMemoryError:
                batch = None
                torch.cuda.empty_cache()
                if b == 1:
                    raise
                b //= 2
        r["batch"] = b
        if b != args.batch:
            r["note"] = f"{args.batch} jets do not fit in device memory on this path; timed at {b}, the largest power-of-two batch that fits"
        r["jets_per_s"] = b / (r["median_ms"] * 1e-3)
        r["fraction_of_fp64_peak"] = flops * r["jets_per_s"] / (FP64_PEAK_TFLOPS * 1e12)
        if path == "tiled":
            torch.cuda.synchronize()
            r["peak_memory_GB"] = torch.cuda.max_memory_allocated() / 1e9
            kt = _lib.kernel_timings(lambda: step(enc, dec, batch), reps=3)
            r["kernels_ms_per_launch"] = {k: {"launches_per_step": n / 3, "ms": ms} for k, (n, ms) in sorted(kt.items(), key=lambda kv: -kv[1][0] * kv[1][1])}
        out[path] = r
        batch = None
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
    out["speedup_per_jet"] = out["tiled"]["jets_per_s"] / out["composite"]["jets_per_s"]
    out["parity_vs_oracle_2_jets"] = {p: parity(enc, dec, p, dev) for p in ("tiled", "composite")}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
