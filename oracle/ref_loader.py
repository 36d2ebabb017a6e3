"""TEST INFRASTRUCTURE -- imports the unmodified reference (zju3dv/ENeRF) on CPU.

Only usable where a reference tree exists (see find_reference), so no test, smoke() or bench.py calls this.
It is used by `oracle/make_golden.py` to mint tests/golden/*.pt and tests/golden/boundary_*.json.

What it does (SURVEY.md section 8c): puts two shims on sys.path (kornia.utils.create_meshgrid,
imp.load_source), sets $workspace (lib/config/config.py:10), fakes argv before `import lib.config`
(argparse runs at import, config.py:191-201), chdirs to the reference root (relative yaml paths).
"""
import contextlib
import io
import os
import sys
import tempfile

_HERE = os.path.dirname(os.path.abspath(__file__))


def find_reference():
    for cand in (os.environ.get("ENERF_REF"), "/root/reference"):
        if cand and os.path.isfile(os.path.join(cand, "lib", "networks", "enerf", "network.py")):
            return cand
    return None


def load_reference(cfg_file="configs/enerf/dtu_pretrain.yaml", opts=()):
    """Returns (cfg, module_dict).  Can be called once per process (cfg is a global built at import)."""
    root = find_reference()
    if root is None:
        raise RuntimeError("reference tree not found (set ENERF_REF)")
    sys.dont_write_bytecode = True
    shims = os.path.join(_HERE, "shims")
    for p in (shims, root):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ.setdefault("workspace", tempfile.mkdtemp(prefix="enerf_ws_"))
    old_argv, old_cwd = sys.argv, os.getcwd()
    sys.argv = ["run.py", "--type", "evaluate", "--cfg_file", cfg_file, "gpus", "-1,"] + [str(o) for o in opts]
    os.chdir(root)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            from lib.config import cfg
            import lib.networks.enerf.network as network
            import lib.networks.enerf.utils as utils
            import lib.datasets.enerf_utils as enerf_utils
    finally:
        sys.argv = old_argv
        os.chdir(old_cwd)
    return cfg, {"network": network, "utils": utils, "enerf_utils": enerf_utils}
