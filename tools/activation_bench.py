"""Cost of the CGMLP activation: the cfg-1 training step (enc 3-3-4-4 / dec 4-4-3-3, 'min&max' latent, MLP 6 x 6, fp64, 512 jets
of 30 particles, chamfer + 1e-8 L1) for each activation of the reference's table,
  - as FusedTrainStep replayed as one CUDA graph (the fused path every activation now takes), and
  - through the layer-level composite (the modules' _forward_generic + autograd), which is how every activation other than
    leakyrelu ran before the fused MLP kernels took them,
alternated in one run: per activation, warm-up, then alternating steps of the two until each has at least --seconds of measured
time; CUDA events around each step, L2 overwritten before every step (256 MB write, not timed).  Also the per-kernel times of one
fused step (lgae_timing_enable), of which mlp_fwd / mlp_bwd are the kernels the activation changes.  Prints one JSON document
(and writes it to --out) with the device name and power limit read in the same run.

    python tools/activation_bench.py --out profiles/r06_activation_bench.json
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import CFG  # noqa: E402   (the cfg-1 model at 30 particles)
from tools.input_grad_bench import _device_info, _kernel_times  # noqa: E402

ACTIVATIONS = ("leakyrelu", "relu", "elu", "sigmoid", "logsigmoid", "tanh", "atan")
BATCH = 512


def build(dev, activation):
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    torch.manual_seed(0)
    common = dict(maxdim=[2], num_basis_fn=CFG["num_basis_fn"], max_zf=[1], weight_init="randn", level_gain=[1.0], activation=activation,
                  mlp=True, mlp_depth=CFG["mlp_depth"], mlp_width=CFG["mlp_width"], device=torch.device("cpu"), dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=CFG["n"], tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=CFG["tau_s"],
                     tau_latent_vectors=CFG["tau_v"], num_channels=CFG["enc_channels"], jet_features=False,
                     map_to_latent=CFG["map_to_latent"], **common)
    dec = LGNDecoder(tau_latent_scalars=2 * CFG["tau_s"], tau_latent_vectors=2 * CFG["tau_v"], num_output_particles=CFG["n"],
                     tau_output_scalars=1, tau_output_vectors=1, num_channels=CFG["dec_channels"], cg_dict=enc.cg_dict, **common)
    assert enc.fused and dec.fused, (enc._fused_reason, dec._fused_reason)
    return enc.to(dev), dec.to(dev)


def jets(batch, seed=1):
    from oracle import lgae_oracle as orc
    data = orc.synthetic_jets(batch, CFG["n"], seed=seed, mass_scale=0.05, pad=True)
    pn, _ = orc.normalize_p4_overall_max(data["p4"])
    return {"p4": pn, "labels": data["labels"]}


def run_activation(activation, seconds, dev):
    from lgn_autoencoder_b200 import fused
    from lgn_autoencoder_b200.train import FusedTrainStep
    enc, dec = build(dev, activation)
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
    kern = _kernel_times(lambda: (eager.step(batch["p4"], batch["labels"]), torch.cuda.synchronize()))
    med = {k: sorted(v)[len(v) // 2] for k, v in t.items()}
    return {"activation": activation, "steps_each": len(t["fused"]), "fused_graph_median_ms": med["fused"],
            "composite_median_ms": med["composite"], "fused_jets_per_s": BATCH / med["fused"] * 1e3,
            "composite_over_fused": med["composite"] / med["fused"],
            "mlp_fwd_ms": kernel_ms(kern, "mlp_fwd"), "mlp_bwd_ms": kernel_ms(kern, "mlp_bwd"), "kernels_fused_eager_step": kern}


def kernel_ms(kern, name):
    return kern[name]["ms"] if name in kern else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--activations", default=",".join(ACTIVATIONS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("activation_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"device": _device_info(),
           "workload": f"cfg-1 training step, {BATCH} x {CFG['n']} particles, FusedTrainStep (one CUDA graph) vs layer-level composite",
           "cases": [run_activation(a, args.seconds, dev) for a in args.activations.split(",")]}
    doc = json.dumps(res, indent=1)
    print(doc)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
