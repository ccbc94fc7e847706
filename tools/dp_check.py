"""Developer / GPU-box check of the data-parallel gradient exchange (run under torchrun with 2+ ranks):
the peer-memory all-reduce (lgae_peer_allreduce) against NCCL's, bit-identity of the result across ranks, graph replay, and
the step time of the three exchange variants.
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/dp_check.py
--particles N runs the same cross-check on the cfg-1 model of tools/long_jet_bench.py at N particles per jet, through
FusedTrainStep(adjoint="tiled") (any N), at --batch jets per rank (default 512, or 64 with --particles)."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from bench import CFG, build_models, synthetic_jets
from lgn_autoencoder_b200.train import FusedTrainStep

ap = argparse.ArgumentParser()
ap.add_argument("--particles", type=int, default=None)
ap.add_argument("--batch", type=int, default=None)
args = ap.parse_args()
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
kw = dict(l1_lambda=1e-8, l1_scale=1.0 / world, normalize=True, get_real="sum")
if args.particles is None:
    enc, dec = build_models(dev)
    N, B = CFG["n"], args.batch or 512
else:
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from long_jet_bench import build
    enc, dec = build(dev, n=args.particles)
    N, B = args.particles, args.batch or 64
    kw["adjoint"] = "tiled"
p4 = synthetic_jets(B, N, seed=100 + rank).to(dev)
res = {}
os.environ["LGAE_PEER_MULTICAST"] = "1"
for name, opts in (("peer_multicast", dict(peer_allreduce=True)), ("peer", dict(peer_allreduce=True)), ("nccl_split", dict(peer_allreduce=False, overlap_allreduce=True)),
                   ("nccl_single", dict(peer_allreduce=False, overlap_allreduce=False))):
    if name == "peer":
        os.environ["LGAE_PEER_MULTICAST"] = "0"
    st = FusedTrainStep(enc, dec, B, **kw, **opts)
    if name.startswith("peer"):
        assert st._peer is not None, "peer path not active"
        if rank == 0:
            print(name, "multicast pointer:", hex(st._peer[7]))
    for _ in range(5):
        loss = st.step(p4)
    torch.cuda.synchronize()
    dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(200):
        st.run()
    b.record()
    torch.cuda.synchronize()
    t = torch.tensor([a.elapsed_time(b) / 200], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res[name] = (st.g_all.clone(), loss.item(), t.item())
    if name.startswith("peer"):
        assert not st.peer_error(), "peer hand-shake timed out"
    st.graph = None
    del st
# no exchange at all (every rank steps on its own shard, no synchronisation): what the exchange + rank skew cost
st = FusedTrainStep(enc, dec, B, **kw, peer_allreduce=False)
st._distributed = lambda: False
for _ in range(5):
    st.step(p4)
torch.cuda.synchronize()
dist.barrier()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(200):
    st.run()
b.record()
torch.cuda.synchronize()
t = torch.tensor([a.elapsed_time(b) / 200], device=dev, dtype=torch.float64)
dist.all_reduce(t, op=dist.ReduceOp.MAX)
res["no_exchange"] = (None, 0.0, t.item())
st.graph = None
del st
g_peer, g_ref = res["peer"][0], res["nccl_single"][0]
scale = g_ref.abs().max().item()
err = max((g_peer - g_ref).abs().max().item(), (res["peer_multicast"][0] - g_ref).abs().max().item()) / scale
err_split = (res["nccl_split"][0] - g_ref).abs().max().item() / scale
gathered = [torch.empty_like(g_peer) for _ in range(world)]
dist.all_gather(gathered, g_peer)
identical = all(torch.equal(gathered[0], g) for g in gathered)
if rank == 0:
    print(f"world {world}, {N} particles: peer vs nccl rel err {err:.2e}; split vs single {err_split:.2e}; peer result bit-identical on all ranks: {identical}")
    print("ms/step (max over ranks): " + ", ".join(f"{k} {v[2]:.4f}" for k, v in res.items()))
    assert err < 1e-13 and err_split < 1e-13 and identical
dist.barrier()
dist.destroy_process_group()
os._exit(0)
