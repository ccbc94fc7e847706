"""Cost of the input gradient: the cfg-1 model (enc 3-3-4-4 / dec 4-4-3-3, 'min&max' latent, MLP 6 x 6, fp64) through the module
API -- encoder, decoder, fused chamfer against the jets, autograd backward -- with and without p4.requires_grad, at 512 x 30
particles (per-lane adjoint) and 512 x 150 (tiled adjoint).  Per case: warm-up, then alternating steps of the two variants until
each has at least --seconds of measured time, CUDA events around each step, L2 overwritten before every step (256 MB write, not
timed).  Also the per-kernel times of one step with the input gradient (lgae_timing_enable).  Prints one JSON document (and writes
it to --out) with the device name and power limit.

    python tools/input_grad_bench.py --out profiles/r05_input_grad_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.long_jet_bench import build  # noqa: E402


def _device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        out = f"nvidia-smi unavailable: {e}"
    return out


def _kernel_times(fn):
    from lgn_autoencoder_b200 import _lib
    lib = _lib.load()
    lib.lgae_timing_enable(1)
    fn()
    buf = __import__("ctypes").create_string_buffer(1 << 16)
    lib.lgae_timing_report(buf, len(buf))
    lib.lgae_timing_enable(0)
    rows = {}
    for line in buf.value.decode().splitlines():
        name, count, ms = line.split()
        rows[name] = {"count": int(count), "ms": float(ms)}
    return rows


def run_case(n, batch, seconds, dev):
    from lgn_autoencoder_b200 import fused
    from oracle import lgae_oracle as orc
    enc, dec = build(dev, n=n)
    data = orc.synthetic_jets(batch, n, seed=3, mass_scale=0.05, pad=n > 32)
    p4 = orc.normalize_p4_overall_max(data["p4"])[0].to(dev)
    labels = data["labels"].to(dev) if "labels" in data else None
    flush = torch.empty(32 * 1024 * 1024, dtype=torch.float64, device=dev)

    def step(with_grad):
        enc.zero_grad(set_to_none=True)
        dec.zero_grad(set_to_none=True)
        x = p4.clone().requires_grad_(with_grad)
        d = {"p4": x} if labels is None else {"p4": x, "labels": labels}
        fused.chamfer_loss(dec(enc(d)), x, "real").backward()

    def timed(with_grad):
        flush.fill_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step(with_grad)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    for _ in range(3):
        step(False)
        step(True)
    torch.cuda.synchronize()
    t = {False: [], True: []}
    while min(sum(t[False]), sum(t[True])) < 1000 * seconds:
        for w in (False, True):
            t[w].append(timed(w))
    kern = _kernel_times(lambda: (step(True), torch.cuda.synchronize()))
    med = {w: sorted(v)[len(v) // 2] for w, v in t.items()}
    input_ms = sum(r["ms"] for k, r in kern.items() if k.startswith("pgrad") or k == "chamfer_target_grad")
    return {"n": n, "batch": batch, "adjoint": "per-lane" if n <= 32 else "tiled", "steps_each": len(t[False]),
            "median_ms_without_p4_grad": med[False], "median_ms_with_p4_grad": med[True], "overhead_ms": med[True] - med[False],
            "input_grad_kernels_ms": input_ms, "kernels_with_p4_grad": kern}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=3.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("input_grad_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"device": _device_info(), "workload": "cfg-1 model, module API forward + chamfer + backward, with / without p4.requires_grad",
           "cases": [run_case(30, 512, args.seconds, dev), run_case(150, 512, args.seconds, dev)]}
    doc = json.dumps(res, indent=1)
    print(doc)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
