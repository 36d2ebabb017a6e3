"""TEST INFRASTRUCTURE -- mint tests/golden/*.pt and tests/golden/boundary_*.json by running the UNMODIFIED reference on CPU.

Usage (authoring container only; needs /root/reference or $ENERF_REF):
    python oracle/make_golden.py            # writes every case listed in CASES
    python oracle/make_golden.py c1_nocascade

The reference's cfg is a process-global built at import (lib/config/config.py:191-201), hence one
subprocess per case.  Each fixture holds: the cfg overrides, the weights (state_dict of the
reference's own Network under torch.manual_seed(0) + randomised BN), the synthetic batch, the
reference outputs (Network.forward, network.py:76-113) and a few per-stage intermediates obtained
by calling the reference's own functions in the order forward() does.
"""
import os
import subprocess
import sys

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, _ROOT)

# name -> (yaml, cfg opts, make_cfg kind + overrides, H, W, S)
CASES = {
    # BASELINE.json configs[0]: 64x80 crop, 2 src views, 8 planes, 1 cascade level
    "c1_nocascade": dict(yaml="configs/enerf/dtu_pretrain_nocascade.yaml",
                         opts=["enerf.cas_config.volume_planes", "8,"],
                         kind="nocascade", over=dict(volume_planes=[8]), H=64, W=80, S=2),
    # reduced configs[1]: 2-level cascade, both levels rendered (exercises nerf_0 with Ns=8, fc=35)
    "c2_small_cascade": dict(yaml="configs/enerf/dtu_pretrain.yaml",
                             opts=["enerf.cas_config.volume_planes", "8,8"],
                             kind="cascade", over=dict(volume_planes=[8, 8]), H=64, W=96, S=3),
    # reduced headline run (README.md:114: render_if False,True), 4 source views
    "c2_headline_small": dict(yaml="configs/enerf/dtu_pretrain.yaml",
                              opts=["enerf.cas_config.volume_planes", "16,8", "enerf.cas_config.render_if", "False,True"],
                              kind="cascade", over=dict(volume_planes=[16, 8], render_if=[False, True]), H=96, W=64, S=4),
    # network_human (ZJU-MoCap / interactive variant): rays masked by mask_at_box at the last level
    "c4_human_small": dict(yaml="configs/enerf/dtu_pretrain.yaml",
                           opts=["enerf.cas_config.volume_planes", "8,8", "enerf.cas_config.render_if", "False,True"],
                           kind="cascade", over=dict(volume_planes=[8, 8], render_if=[False, True]), H=64, W=96, S=2, human=True),
    # network_composite (configs/enerf/enerf_outdoor/actor1.yaml): one bbox-cropped foreground layer + background
    "c5_composite_1fg": dict(yaml="configs/enerf/enerf_outdoor/actor1.yaml",
                             opts=["enerf.cas_config.volume_planes", "8,8"],
                             kind="composite", over=dict(volume_planes=[8, 8]), H=64, W=96, S=3, composite=1),
    # two overlapping foreground layers (exercises the per-pixel z-sort), level 0 not rendered, 2 samples
    "c5_composite_2fg": dict(yaml="configs/enerf/enerf_outdoor/actor1.yaml",
                             opts=["num_fg_layers", "2", "enerf.cas_config.volume_planes", "8,8", "enerf.cas_config.num_samples", "2,2",
                                   "enerf.cas_config.render_if", "False,True"],
                             kind="composite", over=dict(volume_planes=[8, 8], num_samples=[2, 2], render_if=[False, True]),
                             H=64, W=96, S=2, composite=2),
    # oracle branches the other cases leave unpinned (VERDICT r1): white background (utils.py:596-599) ...
    "c2_white_bkgd": dict(yaml="configs/enerf/dtu_pretrain.yaml",
                          opts=["enerf.cas_config.volume_planes", "8,8", "enerf.cas_config.render_if", "False,True", "enerf.white_bkgd", "True"],
                          kind="cascade", over=dict(volume_planes=[8, 8], render_if=[False, True], white_bkgd=True), H=64, W=96, S=3),
    # ... Agg without the view-direction MLP (nerf.py:74-78) ...
    "c2_no_viewdir": dict(yaml="configs/enerf/dtu_pretrain.yaml",
                          opts=["enerf.cas_config.volume_planes", "8,8", "enerf.cas_config.render_if", "False,True", "enerf.viewdir_agg", "False"],
                          kind="cascade", over=dict(volume_planes=[8, 8], render_if=[False, True], viewdir_agg=False), H=64, W=96, S=3),
    # ... and five source views (beyond the tensor-core ray kernel's former S <= 4 limit)
    "c2_five_views": dict(yaml="configs/enerf/dtu_pretrain.yaml",
                          opts=["enerf.cas_config.volume_planes", "8,8", "enerf.cas_config.render_if", "False,True"],
                          kind="cascade", over=dict(volume_planes=[8, 8], render_if=[False, True]), H=64, W=96, S=5),
    # BASELINE.json configs[4] in miniature: 6 source views, 3 foreground layers + background
    "c5_composite_3fg_s6": dict(yaml="configs/enerf/enerf_outdoor/actor1.yaml",
                                opts=["num_fg_layers", "3", "enerf.cas_config.volume_planes", "8,8", "enerf.cas_config.render_if", "False,True"],
                                kind="composite", over=dict(volume_planes=[8, 8], render_if=[False, True]),
                                H=64, W=128, S=6, composite=3),
}


# the plugin seam (tests/test_reference_boundary.py): variant -> (yaml, cfg opts, the reference's own module for that cfg)
BOUNDARY = {
    "network": ("configs/enerf/dtu_pretrain.yaml", [], "lib.networks.enerf.network"),
    "network_human": ("configs/enerf/zjumocap_eval.yaml", [], "lib.networks.enerf.network_human"),
    "network_composite": ("configs/enerf/enerf_outdoor/actor1.yaml", ["num_fg_layers", "2"], "lib.networks.enerf.network_composite"),
}


def state_dict_digest(sd):
    """[key, shape, dtype, sha256 of the raw bytes] per entry, in state_dict order."""
    import hashlib
    return [[k, list(v.shape), str(v.dtype).replace("torch.", ""), hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest()]
            for k, v in sd.items()]


def run_boundary_case(variant):
    """The cfg keys the reference's Network reads after its yaml is merged (``enerf``, and ``num_fg_layers`` where the
    yaml sets it) and the digest of the reference Network's initial state_dict under torch.manual_seed(0)."""
    import importlib
    import json
    import torch
    from oracle.ref_loader import load_reference

    yaml, opts, module = BOUNDARY[variant]
    cfg, _ = load_reference(yaml, opts)

    def plain(node):
        return {k: plain(v) for k, v in node.items()} if isinstance(node, dict) else (list(node) if isinstance(node, tuple) else node)

    keep = {"enerf": plain(cfg.enerf)}
    if "num_fg_layers" in cfg:
        keep["num_fg_layers"] = int(cfg.num_fg_layers)
    torch.manual_seed(0)
    net = importlib.import_module(module).Network()
    fixture = {"variant": variant, "yaml": yaml, "opts": opts, "reference_module": module, "reference_commit": "5a084e9",
               "torch": torch.__version__, "cfg": keep, "state_dict": state_dict_digest(net.state_dict())}
    path = os.path.join(_ROOT, "tests", "golden", f"boundary_{variant}.json")
    entries = fixture.pop("state_dict")
    with open(path, "w") as f:               # one state_dict entry per line
        f.write(json.dumps(fixture)[:-1] + ', "state_dict": [\n' + ",\n".join(json.dumps(e) for e in entries) + "\n]}\n")
    fixture["state_dict"] = entries
    print(variant, "->", path, os.path.getsize(path) // 1024, "KiB;", len(fixture["state_dict"]), "state_dict entries")


def run_composite_case(name):
    """network_composite has no per-stage hooks worth stashing: outputs + a few layer intermediates
    recomputed with the reference's own functions."""
    import torch
    from oracle.ref_loader import load_reference
    from enerf_b200 import config as bcfg
    from enerf_b200 import synthetic

    case = CASES[name]
    cfg, mods = load_reference(case["yaml"], case["opts"])
    assert cfg.num_fg_layers == case["composite"]
    import lib.networks.enerf.network_composite as network_composite
    torch.manual_seed(0)
    net = network_composite.Network().eval()
    synthetic.randomize_bn_(net, seed=1)
    my_cfg = bcfg.composite_cfg(num_fg_layers=case["composite"], **case["over"])
    batch = synthetic.make_composite_batch(case["H"], case["W"], case["S"], my_cfg, seed=2)
    torch.set_num_threads(os.cpu_count())
    with torch.no_grad():
        out = net({k: v.clone() for k, v in batch.items()})
    fixture = {
        "case": name, "composite": case["composite"], "cfg_kind": case["kind"], "cfg_over": case["over"],
        "H": case["H"], "W": case["W"], "S": case["S"],
        "state_dict": {k: v.clone() for k, v in net.state_dict().items()},
        "batch": batch,
        "out": {k: (v.clone() if torch.is_tensor(v) else v) for k, v in out.items()},
        "mid": {},
        "reference_commit": "5a084e9", "torch": torch.__version__,
    }
    path = os.path.join(_ROOT, "tests", "golden", name + ".pt")
    torch.save(fixture, path)
    print(name, "->", path, os.path.getsize(path) // 1024, "KiB;", {k: (tuple(v.shape) if torch.is_tensor(v) else v) for k, v in out.items()})


def run_case(name):
    if name.startswith("boundary_"):
        return run_boundary_case(name[len("boundary_"):])
    if CASES[name].get("composite"):
        return run_composite_case(name)
    import torch
    from oracle.ref_loader import load_reference
    from enerf_b200 import config as bcfg
    from enerf_b200 import synthetic

    case = CASES[name]
    cfg, mods = load_reference(case["yaml"], case["opts"])
    utils = mods["utils"]
    torch.manual_seed(0)
    if case.get("human"):
        import lib.networks.enerf.network_human as network_human
        net = network_human.Network().eval()
    else:
        net = mods["network"].Network().eval()
    synthetic.randomize_bn_(net, seed=1)
    my_cfg = (bcfg.nocascade_cfg if case["kind"] == "nocascade" else bcfg.make_cfg)(**case["over"])
    batch = synthetic.make_batch(case["H"], case["W"], case["S"], my_cfg, seed=2)
    if case.get("human"):
        batch["mask_at_box"] = synthetic.make_mask_at_box(case["H"], case["W"])
    # cross-check the ray generator against the reference's own (lib/datasets/enerf_utils.py:25-71)
    import numpy as np
    for i in range(cfg.enerf.cas_config.num):
        r, _, _ = mods["enerf_utils"].build_rays(np.zeros((case["H"], case["W"], 3), np.float32),
                                                 batch["tar_ext"][0].numpy().astype(np.float64),
                                                 batch["tar_ixt"][0].numpy().astype(np.float64),
                                                 np.ones((case["H"], case["W"]), np.uint8), i, "test")
        assert np.abs(r - batch[f"rays_{i}"][0].numpy()).max() < 1e-5, "ray generator mismatch"
    torch.set_num_threads(os.cpu_count())
    with torch.no_grad():
        out = net({k: v.clone() for k, v in batch.items()})
        mid = {}
        feats = net.forward_feat(batch["src_inps"])
        mid["feat_level_0"] = feats["level_0"]
        depth = std = nf = None
        for i in range(cfg.enerf.cas_config.num):
            var, dv, nf = utils.build_feature_volume(feats[f"level_{i}"], batch, D=cfg.enerf.cas_config.volume_planes[i],
                                                     depth=depth, std=std, near_far=nf, level=i)
            vol, prob = getattr(net, f"cost_reg_{i}")(var)
            depth, std = utils.depth_regression(prob, dv, i, batch)
            if i == 0:
                mid["variance_0"] = var
            mid.update({f"near_far_{i}": nf, f"depth_prob_{i}": prob, f"depth_{i}": depth, f"std_{i}": std})
            if i == cfg.enerf.cas_config.num - 1:
                mid[f"feat_volume_{i}"] = vol
    fixture = {
        "case": name, "human": bool(case.get("human")), "cfg_kind": case["kind"], "cfg_over": case["over"], "H": case["H"], "W": case["W"], "S": case["S"],
        "state_dict": {k: v.clone() for k, v in net.state_dict().items()},
        "batch": batch,
        "out": {k: v.clone() for k, v in out.items()},
        "mid": {k: v.clone() for k, v in mid.items()},
        "reference_commit": "5a084e9", "torch": torch.__version__,
    }
    path = os.path.join(_ROOT, "tests", "golden", name + ".pt")
    torch.save(fixture, path)
    print(name, "->", path, os.path.getsize(path) // 1024, "KiB;", {k: tuple(v.shape) for k, v in out.items()})


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--one":
        run_case(sys.argv[2])
    else:
        for n in (sys.argv[1:] or list(CASES) + [f"boundary_{v}" for v in BOUNDARY]):
            subprocess.check_call([sys.executable, os.path.abspath(__file__), "--one", n])
