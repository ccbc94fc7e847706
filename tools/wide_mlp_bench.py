"""Scalar MLPs wider than 48 on the fused path (the streamed-weight CGMLP kernels, DESIGN section 4g).

  - The cfg-4 channel shape, enc 6-6-8-8 / dec 8-8-6-6 (MLP hidden widths 72 and 96), 'min&max' latent with tau = 1/8, MLP 6 x 6,
    fp64, 512 jets of 30 particles, chamfer + 1e-8 L1: FusedTrainStep replayed as one CUDA graph against the layer-level
    composite (the modules' _forward_generic + autograd, where these models ran before), alternated until each has at least
    --seconds of measured time; CUDA events around each step, L2 overwritten before every step (256 MB write, not timed); medians.
  - Per-kernel times of one eager fused step (lgae_timing_enable).
  - The raw MLP entry points on one level at 512 x 30 rows and depth 6, at hidden widths 96 (ntw 12) and 72 (ntw 9, resident
    forward and streamed adjoint), and the resident kernels at width 48 for comparison: per-kernel times, the fp64 rate from the
    layer shapes (forward 2 * rows * sum(n_in * n_out); adjoint twice that: data and weight gradients) against the measured
    37.1 TFLOP/s DMMA peak, and the reduce of the adjoint's partial rows.
Prints one JSON document (and writes it to --out) with the device name and power limit read in the same run.

    python tools/wide_mlp_bench.py --out profiles/r07_wide_mlp_bench.json
"""
import argparse
import ctypes as C
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import FP64_PEAK_TFLOPS  # noqa: E402
from tools.input_grad_bench import _device_info, _kernel_times  # noqa: E402

BATCH, N = 512, 30
MODEL = dict(enc_channels=[6, 6, 8, 8], dec_channels=[8, 8, 6, 6], tau_s=1, tau_v=8, map_to_latent="min&max", num_basis_fn=10, mlp_depth=6,
             mlp_width=6)


def build(dev, enc_channels, dec_channels, mlp_width, mlp_depth, n=N, seed=0):
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    torch.manual_seed(seed)
    common = dict(maxdim=[2], num_basis_fn=MODEL["num_basis_fn"], max_zf=[1], weight_init="randn", level_gain=[1.0], activation="leakyrelu",
                  mlp=True, mlp_depth=mlp_depth, mlp_width=mlp_width, device=torch.device("cpu"), dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=n, tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=MODEL["tau_s"],
                     tau_latent_vectors=MODEL["tau_v"], num_channels=enc_channels, jet_features=False, map_to_latent=MODEL["map_to_latent"],
                     **common)
    dec = LGNDecoder(tau_latent_scalars=2 * MODEL["tau_s"], tau_latent_vectors=2 * MODEL["tau_v"], num_output_particles=n,
                     tau_output_scalars=1, tau_output_vectors=1, num_channels=dec_channels, cg_dict=enc.cg_dict, **common)
    return enc.to(dev), dec.to(dev)


def jets(batch, seed=1):
    from oracle import lgae_oracle as orc
    data = orc.synthetic_jets(batch, N, seed=seed, mass_scale=0.05, pad=True)
    pn, _ = orc.normalize_p4_overall_max(data["p4"])
    return {"p4": pn, "labels": data["labels"]}


def train_step(seconds, dev):
    from lgn_autoencoder_b200 import fused
    from lgn_autoencoder_b200.train import FusedTrainStep
    enc, dec = build(dev, MODEL["enc_channels"], MODEL["dec_channels"], MODEL["mlp_width"], MODEL["mlp_depth"])
    assert enc.fused and dec.fused, (enc._fused_reason, dec._fused_reason)
    batch = {k: v.to(dev) for k, v in jets(BATCH).items()}
    flush = torch.empty(32 * 1024 * 1024, dtype=torch.float64, device=dev)
    step = FusedTrainStep(enc, dec, BATCH, l1_lambda=1e-8, normalize=False, use_labels=True, use_graph=True, get_real="real")

    def fused_step():
        step.step(batch["p4"], batch["labels"])

    def composite_step():
        enc.zero_grad(set_to_none=True)
        dec.zero_grad(set_to_none=True)
        latent = enc._forward_generic(batch, batch["p4"], False)
        recon = dec._forward_generic(latent, False, None)
        loss = fused.chamfer_loss(recon, batch["p4"], "real") + 1e-8 * (enc.l1_norm() + dec.l1_norm())
        loss.backward()

    def timed(fn):
        flush.fill_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    for _ in range(3):
        fused_step()
        composite_step()
    torch.cuda.synchronize()
    t = {"fused": [], "composite": []}
    while min(sum(t["fused"]), sum(t["composite"])) < 1000 * seconds:
        t["fused"].append(timed(fused_step))
        t["composite"].append(timed(composite_step))
    eager = FusedTrainStep(enc, dec, BATCH, l1_lambda=1e-8, normalize=False, use_labels=True, use_graph=False, get_real="real")
    eager.step(batch["p4"], batch["labels"])
    kern = _kernel_times(lambda: (eager.step(batch["p4"], batch["labels"]), torch.cuda.synchronize()))
    med = {k: sorted(v)[len(v) // 2] for k, v in t.items()}
    return {"workload": f"enc {MODEL['enc_channels']} / dec {MODEL['dec_channels']}, min&max tau 1/8, MLP 6 x 6, {BATCH} x {N} particles",
            "steps_each": len(t["fused"]), "fused_graph_median_ms": med["fused"], "composite_median_ms": med["composite"],
            "fused_jets_per_s": BATCH / med["fused"] * 1e3, "composite_over_fused": med["composite"] / med["fused"],
            "kernels_fused_eager_step": kern}


def raw_level(c_out, mlp_width, depth, reps, dev):
    """lgae_mlp_forward + lgae_mlp_backward on one level with c_out output channels, 512 x 30 rows."""
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200._lib import ptr
    lib = _lib.load()
    enc, _ = build(dev, [2, c_out], [2, 2], mlp_width, depth)
    assert enc.fused, enc._fused_reason
    desc = enc._plan.desc
    theta, _ = enc._flat_params()
    lin = [m.weight for m in enc.lgn_cg.mlp_levels[0].linear]
    rows = BATCH * N
    nin, width = lin[0].shape[1], lin[0].shape[0]
    x = torch.randn(rows, nin, dtype=torch.float64, device=dev)
    g_y = torch.randn(rows, nin, dtype=torch.float64, device=dev)
    wpack = torch.empty(lib.lgae_mlp_pack_doubles(C.byref(desc), 0), dtype=torch.float64, device=dev)
    acts = torch.empty(len(lin) - 1, rows, 8 * ((width + 7) // 8), dtype=torch.float64, device=dev)
    y, g_x, gtheta = torch.empty_like(x), torch.empty_like(x), torch.zeros_like(theta)
    partials = torch.empty(lib.lgae_partials_doubles(C.byref(desc), 1), dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream().cuda_stream

    def run():
        for _ in range(reps):
            _lib.check(lib.lgae_mlp_forward(C.byref(desc), 0, ptr(theta), ptr(x), rows, ptr(wpack), ptr(acts), ptr(y), st), "mlp_forward")
            _lib.check(lib.lgae_mlp_backward(C.byref(desc), 0, ptr(theta), ptr(x), rows, ptr(wpack), ptr(acts), ptr(g_y), ptr(g_x), ptr(gtheta),
                                             ptr(partials), st), "mlp_backward")
        torch.cuda.synchronize()

    run()
    times = _lib.kernel_timings(run)
    fwd_flop = 2 * rows * sum(w.shape[0] * w.shape[1] for w in lin)
    out = {"c_out": c_out, "hidden_width": width, "depth": depth, "rows": rows, "reps": reps,
           "part_row_mb": lib.lgae_partials_doubles(C.byref(desc), 1) * 8 / 1e6, "fwd_gflop": fwd_flop / 1e9, "bwd_gflop": 2 * fwd_flop / 1e9,
           "kernels_ms_per_launch": {k: v[1] for k, v in times.items()}}
    for name, t in times.items():
        if name.startswith("mlp_fwd") or name.startswith("mlp_bwd"):
            flop = fwd_flop if name.startswith("mlp_fwd") else 2 * fwd_flop
            tf = flop / (t[1] * 1e-3) / 1e12
            out[name] = {"ms": t[1], "tflops": tf, "share_of_dmma_peak": tf / FP64_PEAK_TFLOPS}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=3.0)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("wide_mlp_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"device": _device_info(), "fp64_dmma_peak_tflops": FP64_PEAK_TFLOPS,
           "train_step": train_step(args.seconds, dev),
           "raw_mlp": [raw_level(8, 6, 6, args.reps, dev),    # width 96: (12, 2), both streamed
                       raw_level(6, 6, 6, args.reps, dev),    # width 72: (9, 2), resident forward, streamed adjoint
                       raw_level(4, 6, 6, args.reps, dev)]}   # width 48: (6, 1), resident
    doc = json.dumps(res, indent=1)
    print(doc)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
