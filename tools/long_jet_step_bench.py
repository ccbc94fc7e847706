"""The cfg-1 training step on 150-particle jets (tools/long_jet_bench.py's model and jets, 'real' get_real, chamfer + 1e-8 L1,
fp64), timed three ways:
  module          the module API (forward, chamfer and L1, autograd backward): the fused forward and the tiled adjoints as
                  separate calls, the `tiled` row of long_jet_bench.py;
  fused_step      FusedTrainStep(adjoint="tiled") replayed as one CUDA graph (lgae_train_step_tiled);
  module_adam     the module step followed by two torch.optim.Adam steps (one per model), as a training loop runs it;
  fused_step_adam FusedTrainStep(adjoint="tiled") with FlatAdam attached: step and parameter update in one graph.

Per way: warm-up, then steps until at least --seconds of measured time, L2 (126 MB) overwritten before every step with a 256 MB
write that is not timed; CUDA events around each step; peak device memory of that way alone.  Also: the per-kernel times of the
fused step (lgae_timing_enable, eager launches) and the fused step's loss against the module step's on the timed jets.  Prints
one JSON document (and writes it to --out).

    python tools/long_jet_step_bench.py --batch 512 --out long_jet_step.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from long_jet_bench import CFG, build, jets  # noqa: E402

GET_REAL = "real"


def module_step(enc, dec, batch, opts=()):
    from lgn_autoencoder_b200 import fused
    for m in (enc, dec):
        m.zero_grad(set_to_none=True)
    recon = dec(enc(batch))
    loss = fused.chamfer_loss(recon, batch["p4"], GET_REAL) + CFG["l1_lambda"] * (enc.l1_norm() + dec.l1_norm())
    loss.backward()
    for o in opts:
        o.step()
    return loss


def timed(fn, dev, seconds, warmup):
    flush = torch.empty(32 * 1024 * 1024, dtype=torch.float64, device=dev)   # 256 MB > 126 MB of L2
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    while sum(times) < seconds * 1e3 or len(times) < 3:
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return {"steps": len(times), "median_ms": times[len(times) // 2], "min_ms": times[0], "max_ms": times[-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("long_jet_step_bench.py measures on a CUDA device; none is visible")
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200.train import FlatAdam, FusedTrainStep
    dev = torch.device("cuda:0")
    B = args.batch
    out = {"workload": f"cfg1 train step, {CFG['n']}-particle padded jets, batch {B}, fp64", "device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = f"not read: {e}"
    batch = {k: v.to(dev) for k, v in jets(B).items()}

    def run(name, make):
        """make() -> the step function; timed with its own peak memory (models, buffers and jets included)."""
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        fn, keep = make()
        r = timed(fn, dev, args.seconds, args.warmup)
        torch.cuda.synchronize()
        r["peak_memory_GB"] = torch.cuda.max_memory_allocated() / 1e9
        r["jets_per_s"] = B / (r["median_ms"] * 1e-3)
        out[name] = r
        return keep

    def make_module():
        enc, dec = build(dev)
        return (lambda: module_step(enc, dec, batch)), (enc, dec)

    enc_m, dec_m = run("module", make_module)
    loss_module = module_step(enc_m, dec_m, batch).item()
    del enc_m, dec_m

    def make_fused():
        enc, dec = build(dev)
        fs = FusedTrainStep(enc, dec, B, l1_lambda=CFG["l1_lambda"], normalize=False, use_labels=True, get_real=GET_REAL, adjoint="tiled")
        fs.load(batch["p4"], batch["labels"])
        return fs.run, fs

    fs = run("fused_step", make_fused)
    out["fused_step"]["loss_rel_diff_vs_module"] = abs(fs.run().item() - loss_module) / abs(loss_module)
    fs.use_graph = False   # per-kernel events need eager launches
    kt = _lib.kernel_timings(fs.run, reps=3)
    out["fused_step"]["kernels_ms_per_launch"] = {k: {"launches_per_step": n / 3, "ms": ms}
                                                  for k, (n, ms) in sorted(kt.items(), key=lambda kv: -kv[1][0] * kv[1][1])}
    out["fused_step"]["kernels_sum_ms"] = sum(n / 3 * ms for n, ms in kt.values())
    del fs

    def make_module_adam():
        enc, dec = build(dev)
        opts = [torch.optim.Adam(enc.parameters(), 1e-4), torch.optim.Adam(dec.parameters(), 1e-4)]
        return (lambda: module_step(enc, dec, batch, opts)), (enc, dec, opts)

    run("module_adam", make_module_adam)

    def make_fused_adam():
        enc, dec = build(dev)
        fs = FusedTrainStep(enc, dec, B, l1_lambda=CFG["l1_lambda"], normalize=False, use_labels=True, get_real=GET_REAL, adjoint="tiled")
        fs.attach_optimizer(FlatAdam(fs, lr=1e-4))
        fs.load(batch["p4"], batch["labels"])
        return fs.run, fs

    run("fused_step_adam", make_fused_adam)
    out["speedup_fused_step_vs_module"] = out["module"]["median_ms"] / out["fused_step"]["median_ms"]
    out["speedup_fused_step_adam_vs_module_adam"] = out["module_adam"]["median_ms"] / out["fused_step_adam"]["median_ms"]
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
