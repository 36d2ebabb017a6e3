"""The drop-in seam, exercised the way the reference itself does it (SURVEY.md section 8b, VERDICT r1 item 7):
``lib/networks/make_network.py:5-9`` executes the file named by ``cfg.network_path`` with
``imp.load_source(cfg.network_module, cfg.network_path)`` and calls ``Network()`` with no arguments.  Pointing it at
enerf_b200/network{,_human,_composite}.py must yield a module whose state_dict is key-for-key / shape-for-shape the
reference's own, with the same initial values under the same seed, that loads a state_dict of the reference's layout
with strict=True, and that reads the same global ``lib.config.cfg``.

What the reference produced for each variant (its merged cfg keys and the digest of its Network's initial
state_dict) is stored in tests/golden/boundary_<variant>.json, minted by ``oracle/make_golden.py boundary_<variant>``.
One subprocess per variant because the plugin reads the process-global ``lib.config.cfg``."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

VARIANTS = ["network", "network_composite", "network_human"]

CHILD = r'''
import json, os, sys, types, torch
sys.path.insert(0, {root!r})
sys.path.insert(0, os.path.join({root!r}, "oracle", "shims"))
from enerf_b200.config import Node
from oracle.make_golden import state_dict_digest
fx = json.load(open(os.path.join({root!r}, "tests", "golden", "boundary_" + {variant!r} + ".json")))

def node(v):
    return Node({{k: node(x) for k, x in v.items()}}) if isinstance(v, dict) else v

ours = os.path.join({root!r}, "enerf_b200", {variant!r})
cfg = node(fx["cfg"])
cfg.network_module, cfg.network_path = ours, ours + ".py"
lib_config = types.ModuleType("lib.config")                # the reference's global cfg, as its run.py leaves it
lib_config.cfg = cfg
sys.modules["lib.config"] = lib_config
import imp
torch.manual_seed(0)
net = imp.load_source(cfg.network_module, cfg.network_path).Network()   # the reference's factory (lib/networks/make_network.py)
assert type(net).__module__ == ours and os.path.samefile(sys.modules[ours].__file__, ours + ".py"), type(net)
a = net.state_dict()
got, want = state_dict_digest(a), fx["state_dict"]
assert [g[0] for g in got] == [w[0] for w in want], set(g[0] for g in got) ^ set(w[0] for w in want)
for g, w in zip(got, want):
    assert g[1:3] == w[1:3], (g[:3], w[:3])
    assert g[3] == w[3], "same seed -> same initial weights: " + g[0]
ref_sd = {{k: torch.zeros(shape, dtype=getattr(torch, dtype)) for k, shape, dtype, _ in want}}
net.load_state_dict(ref_sd, strict=True)                   # what lib/utils/net_utils.py:load_network does with latest.pth
assert all(not v.any() for v in net.state_dict().values())
import enerf_b200.config as bcfg
assert bcfg.get_cfg() is cfg                               # the plugin reads the reference's global cfg, not a private copy
assert next(net.parameters()).device.type == "cpu" and callable(getattr(net, "forward"))
try:
    net.eval()({{"src_inps": torch.zeros(1, 3, 3, 64, 96)}})   # CPU tensors: the plugin must refuse loudly (no CPU fallback)
except ValueError as e:
    assert "CUDA" in str(e)
else:
    raise AssertionError("CPU batch was accepted")
print("BOUNDARY_OK", len(a))
'''


@pytest.mark.parametrize("variant", VARIANTS)
def test_reference_make_network_loads_the_plugin(variant):
    code = CHILD.format(root=ROOT, variant=variant)
    env = dict(os.environ)
    env.pop("ENERF_B200_PRECISION", None)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and "BOUNDARY_OK" in r.stdout, r.stdout[-2000:] + "\n" + r.stderr[-4000:]
