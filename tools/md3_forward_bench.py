"""The fused maxdim-3 forward (csrc/lgae_md3.cu, DESIGN section 4h) against the layer-level composite it replaces for forward-only calls.

  - Model: the cfg-4 shape, enc 6-6-8-8 / dec 8-8-6-6, 'mix' latent with tau = 1 / 8, MLP 6 x 6, fp64.
  - Anomaly scoring at N = 30 (B = 1024) and N = 150 (B = 1024, or the largest of 512 / 256 / 128 the composite fits; the JSON says
    which): FusedInference replayed as one CUDA graph against the composite's no-grad forward plus the per-jet chamfer score,
    alternated, CUDA events around each pass, L2 overwritten before every pass (256 MB write, not timed); medians.
  - Per-kernel times of one eager FusedInference pass (lgae_timing_enable), and the fraction of the measured 37.1 TFLOP/s fp64
    peak from the reference-faithful count (flop_model.md3_forward_flops_per_jet).
  - Wall time of the equivariance harness (26 boosts + 26 rotations, models/autotest covariance_test) on the cfg-4 shape, fused
    forward against the composite: one warm-up run each, then five timed runs each, alternated; medians and the largest deviations.
Prints one JSON document (and writes it to --out) with the device name, power limit and max SM clock read in the same run.

    python tools/md3_forward_bench.py --out profiles/r08_md3_forward_bench.json
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import FP64_PEAK_TFLOPS  # noqa: E402
from tools.input_grad_bench import _device_info, _kernel_times  # noqa: E402

ENC, DEC = [6, 6, 8, 8], [8, 8, 6, 6]


def build(dev, n, seed=0):
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    torch.manual_seed(seed)
    common = dict(maxdim=[3], num_basis_fn=10, max_zf=[1], weight_init="randn", level_gain=[1.0], activation="leakyrelu", mlp=True,
                  mlp_depth=6, mlp_width=6, device=dev, dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=n, tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=1, tau_latent_vectors=8,
                     num_channels=ENC, jet_features=False, map_to_latent="mix", **common)
    dec = LGNDecoder(tau_latent_scalars=1, tau_latent_vectors=8, num_output_particles=n, tau_output_scalars=1, tau_output_vectors=1,
                     num_channels=DEC, cg_dict=enc.cg_dict, **common)
    assert enc.fused_forward and dec.fused_forward and not enc.fused
    return enc, dec


def composite(model, on):
    model._forward_reason = "composite (benchmark)" if on else None


def scoring(dev, n, batches, reps):
    from lgn_autoencoder_b200 import fused
    from lgn_autoencoder_b200.train import FusedInference
    from oracle import lgae_oracle as orc
    enc, dec = build(dev, n)
    flush = torch.empty(32 * 1024 * 1024, dtype=torch.float64, device=dev)
    for b in batches:
        data = orc.synthetic_jets(b, n, seed=1, mass_scale=0.05, pad=n > 30)
        p4 = data["p4"].to(dev)
        pn, _ = orc.normalize_p4_overall_max(p4)
        batch = {"p4": pn, "labels": data["labels"].to(dev)} if "labels" in data else {"p4": pn}

        def comp():
            with torch.no_grad():
                recon = dec(enc(batch))
                return fused.chamfer_per_jet(recon, pn, "sum")
        composite(enc, True), composite(dec, True)
        try:
            ref = comp()
            torch.cuda.synchronize()
        except torch.OutOfMemoryError:
            torch.cuda.empty_cache()
            continue
        finally:
            composite(enc, False), composite(dec, False)
        inf = FusedInference(enc, dec, b, get_real="sum", use_labels="labels" in batch, normalize=False)
        got = inf.score(pn, batch.get("labels")).clone()
        err = ((got - ref).abs().max() / ref.abs().max()).item()
        times = {"fused_graph": [], "composite": []}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for r in range(reps + 1):
            for name in ("fused_graph", "composite"):
                flush.fill_(1.0)
                if name == "composite":
                    composite(enc, True), composite(dec, True)
                ev[0].record()
                if name == "fused_graph":
                    inf.score(pn, batch.get("labels"))
                else:
                    comp()
                ev[1].record()
                torch.cuda.synchronize()
                composite(enc, False), composite(dec, False)
                if r:
                    times[name].append(ev[0].elapsed_time(ev[1]))
        eager = FusedInference(enc, dec, b, get_real="sum", use_labels="labels" in batch, normalize=False, use_graph=False)
        eager.p4_in.copy_(pn)
        if eager.mask is not None:
            eager.mask.copy_(batch["labels"].to(torch.uint8))
        eager.run()
        kernels = _kernel_times(eager.run)
        from lgn_autoencoder_b200.flop_model import md3_forward_flops_per_jet
        mflop = sum(md3_forward_flops_per_jet(n, ENC, DEC).values()) / 1e6
        med = {k: statistics.median(v) for k, v in times.items()}
        tflops = b * mflop * 1e6 / (med["fused_graph"] * 1e-3) / 1e12
        return {"n": n, "batch": b, "batch_note": "largest of %s the composite fits" % (batches,), "rel_err_scores_vs_composite": err,
                "ms_median": med, "ms_all": times, "speedup": med["composite"] / med["fused_graph"], "mflop_per_jet_forward": mflop,
                "fused_tflops": tflops, "frac_of_fp64_peak": tflops / FP64_PEAK_TFLOPS, "kernels_eager_pass": kernels,
                "peak_mem_gib": torch.cuda.max_memory_allocated() / 2 ** 30}
    return {"n": n, "error": "the composite did not fit at any batch of %s" % (batches,)}


def _max_dev(x):
    """Largest entry of a nested deviation table (dicts / lists of tensors or numbers)."""
    if torch.is_tensor(x):
        return x.abs().max().item()
    if isinstance(x, dict):
        return max((_max_dev(v) for v in x.values()), default=0.0)
    if isinstance(x, (list, tuple)):
        return max((_max_dev(v) for v in x), default=0.0)
    try:
        return abs(float(x))
    except (TypeError, ValueError):
        return 0.0


def harness(dev, jets, reps):
    """Boosts + rotations of covariance_test on both paths: one warm-up run each, then `reps` timed runs each, alternated;
    medians, and the largest output / internal deviations of each path."""
    from lgn_autoencoder_b200.models.autotest import covariance_test
    from oracle import lgae_oracle as orc
    enc, dec = build(dev, 30)
    data = orc.synthetic_jets(jets, 30, seed=3, mass_scale=0.05)
    data = {"p4": data["p4"].to(dev) * 1e3}
    times = {"fused": [], "composite": []}
    devs = {}
    for r in range(reps + 1):
        for label, on in (("fused", False), ("composite", True)):
            composite(enc, on), composite(dec, on)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with torch.no_grad():
                res = [covariance_test(enc, dec, data, t) for t in ("boost", "rotation")]
            torch.cuda.synchronize()
            if r:
                times[label].append(time.perf_counter() - t0)
            else:
                devs[label] = {k: _max_dev(v) for part in res for k, v in part.items() if "dev" in k}
    composite(enc, False), composite(dec, False)
    return {"jets": jets, "timed_runs": reps, "s_median": {k: statistics.median(v) for k, v in times.items()}, "s_all": times,
            "max_deviation": devs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    res = {"device": _device_info(), "model": "enc 6-6-8-8 / dec 8-8-6-6, maxdim 3, 'mix' latent tau 1/8, MLP 6 x 6, fp64",
           "fp64_peak_tflops": FP64_PEAK_TFLOPS}
    res["scoring_n30"] = scoring(dev, 30, [1024], args.reps)
    torch.cuda.empty_cache()
    res["scoring_n150"] = scoring(dev, 150, [1024, 512, 256, 128], max(3, args.reps // 2))
    torch.cuda.empty_cache()
    res["equivariance_harness"] = harness(dev, 8, 5)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
