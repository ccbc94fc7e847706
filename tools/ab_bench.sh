#!/bin/bash
# Developer: A/B of library builds on the bench step (tools/build_variant.sh builds them).
# usage: tools/ab_bench.sh "LGAE_B200_LIB=tools/variants/a.so" "LGAE_B200_LIB=tools/variants/b.so" ...
for cfg in "$@"; do
  out=$(env $cfg python bench.py --no-extras --no-cpu-baseline --steps 200 2>/dev/null | tail -1)
  python - "$cfg" <<PY
import json,sys
d=json.loads('''$out''')
k=d["kernels"]
print(sys.argv[1], "| ms/step %.4f e2e %.4f |" % (d["ms_per_step"], d["e2e"]["ms_per_step"]), " ".join("%s %.1f" % (n, k[n]["ms_per_launch"]*1e3) for n in ("mlp_fwd","mlp_bwd","level_fwd","level_bwd","radial_fwd","radial_bwd","reduce_partials") if n in k))
PY
done
