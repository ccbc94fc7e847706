"""Build liblgae_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so must travel with the repo)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SOURCES = ["lgae_api.cu", "lgae_glue.cu", "lgae_level.cu", "lgae_radial.cu", "lgae_mlp.cu", "lgae_cg.cu", "lgae_layers.cu", "lgae_optim.cu", "lgae_collective.cu",
           "lgae_input_grad.cu", "lgae_md3.cu", "lgae_mlp_act_relu.cu", "lgae_mlp_act_sigmoid.cu", "lgae_mlp_act_tanh.cu",
           *[f"lgae_mlp_streamed_{a}.cu" for a in ("leakyrelu", "relu", "elu", "sigmoid", "logsigmoid", "tanh", "atan")]]
LIB = os.path.join(HERE, "liblgae_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "lgae_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source into one shared library (objects in parallel, then link)."""
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    objs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {src}")
    subprocess.check_call([nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
