"""The drop-in ``lgn`` package (SURVEY.md section 8(b)): every import the reference's callers make resolves to this
repository's implementation, and the regular package shadows the reference's namespace package when both are visible."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

IMPORTS = r"""
import lgn, lgn_autoencoder_b200 as impl
from lgn.models import LGNEncoder, LGNDecoder                       # utils/initialize.py
from lgn.cg_lib.zonal_functions import p_cplx_to_rep, repdot         # utils/losses/chamfer_loss/distance_sq.py:3
from lgn.cg_lib import CGProduct, CGDict, cg_product
from lgn.cg_lib.cg_ops_tau import cg_product_tau
from lgn.g_lib import rotations, GVec, GScalar, GTau                 # lgn/models/autotest/lgn_tests.py
from lgn.g_lib.g_vec import GVec as GVec2
from lgn.nn import MixReps, CatMixReps, RadialFilters
from lgn.models.lgn_cg import LGNCG
from lgn.models.lgn_levels import LGNNodeLevel, CGMLP
from lgn.models.autotest import lgn_tests
import lgn_autoencoder_b200.models as m
assert LGNEncoder is m.LGNEncoder and LGNDecoder is m.LGNDecoder and GVec is GVec2
assert os.path.dirname(os.path.abspath(lgn.__file__)) == os.path.join(ROOT, "lgn"), lgn.__file__
print("shim ok")
"""


def _run(cwd):
    env = dict(os.environ, PYTHONPATH=ROOT)
    code = f"import os\nROOT = {ROOT!r}\n" + IMPORTS
    return subprocess.run([sys.executable, "-c", code], cwd=cwd, env=env, capture_output=True, text=True, timeout=300)


def test_reference_import_paths_resolve_to_this_package():
    r = _run(ROOT)
    assert r.returncode == 0 and "shim ok" in r.stdout, r.stderr[-2000:]


def test_shim_shadows_the_reference_namespace_package(tmp_path):
    """cwd = a reference checkout (its own lgn/ has no __init__.py): PYTHONPATH=<repo> must still win.  The checkout is a
    stand-in of the reference's layout whose sub-packages fail on import, so any of them being picked up fails the run."""
    for sub in ("cg_lib", "g_lib", "models", "nn"):
        d = tmp_path / "lgn" / sub
        d.mkdir(parents=True)
        (d / "__init__.py").write_text(f"raise ImportError('the reference checkout shadowed the shim: lgn.{sub}')\n")
    assert not (tmp_path / "lgn" / "__init__.py").exists()
    r = _run(str(tmp_path))
    assert r.returncode == 0 and "shim ok" in r.stdout, r.stderr[-2000:]
