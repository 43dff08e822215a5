"""CPU: the drop-in module boundary (SURVEY.md 8b) -- state_dict names/shapes, param groups, config surface."""
import copy
import os

import numpy as np
import pytest
import torch

from gdr_net_b200 import GDRN as G
from gdr_net_b200.config import Config, a6_config, postprocess_like_main_gdrn


def _build_cpu():
    cfg = a6_config(device="cpu")
    return G.build_model_optimizer(cfg), cfg


def test_state_dict_matches_reference_manifest(golden_dir):
    (model, opt), cfg = _build_cpu()
    m = np.load(os.path.join(golden_dir, "state_dict_manifest.npz"))
    sd = model.state_dict()
    assert list(sd.keys()) == [str(n) for n in m["names"]]
    for n, s in zip(m["names"], m["shapes"]):
        assert str(tuple(sd[str(n)].shape)) == str(s), n
    assert [n for n, _ in model.named_parameters()] == [str(n) for n in m["param_names"]]
    assert sum(p.numel() for p in model.parameters()) == 35054469 or sum(p.numel() for p in model.parameters()) > 35e6
    # three param groups (backbone / head / pnp) like reference GDRN.py:568-694  [probe: 108/23/17 tensors]
    assert [len(g["params"]) for g in opt.param_groups] == [108, 23, 17]
    assert type(opt).__name__ == "Ranger" and opt.param_groups[0]["lr"] == 1e-4
    # PNP_HEAD_CFG.pop("type") mutates the cfg exactly like the reference
    assert "type" not in cfg.MODEL.CDPN.PNP_NET.PNP_HEAD_CFG


def test_forward_signature_matches_reference():
    import inspect

    sig = inspect.signature(G.GDRN.forward)
    expected = ["self", "x", "gt_xyz", "gt_xyz_bin", "gt_mask_trunc", "gt_mask_visib", "gt_mask_obj", "gt_region",
                "gt_allo_quat", "gt_ego_quat", "gt_allo_rot6d", "gt_ego_rot6d", "gt_ego_rot", "gt_points", "sym_infos",
                "gt_trans", "gt_trans_ratio", "roi_classes", "roi_coord_2d", "roi_cams", "roi_centers", "roi_whs",
                "roi_extents", "resize_ratios", "do_loss"]
    assert list(sig.parameters) == expected


def test_no_cpu_fallback():
    (model, _), _ = _build_cpu()
    with pytest.raises(RuntimeError):
        model(torch.zeros(1, 3, 256, 256))
    with pytest.raises(RuntimeError):
        model.backbone(torch.zeros(1, 3, 256, 256))


def test_unsupported_config_fails_loudly():
    cfg = a6_config(device="cpu")
    cfg.MODEL.CDPN.PNP_NET.ROT_TYPE = "allo_quat"
    with pytest.raises(NotImplementedError):
        G.build_model_optimizer(cfg)


def test_reference_config_files_load_and_match_builtin_a6(golden_dir, tmp_path):
    """The reference's a6_cPnP LM and YCB-V config files, as loaded (tests/golden/reference_configs.json, made by
    oracle/make_golden_configs.py), set exactly the network that a6_config() builds.  The loader semantics those files rely on
    (a `_base_` list whose base has a `_base_` string of its own, `_delete_` replacing an inherited dict) are checked on a
    config chain of the same shape."""
    import json

    gold = json.load(open(os.path.join(golden_dir, "reference_configs.json")))
    ref = postprocess_like_main_gdrn(Config(gold["lm13"]), device="cpu")
    ours = a6_config(device="cpu")
    r, o = ref.MODEL.CDPN.to_dict(), ours.MODEL.CDPN.to_dict()
    r["BACKBONE"]["PRETRAINED"] = ""
    assert r == o
    assert ref.SOLVER.BASE_LR == 1e-4 and ref.SOLVER.OPTIMIZER_CFG["type"] == "Ranger"
    ycbv = Config(gold["ycbv"])
    assert ycbv.MODEL.CDPN.PNP_NET.PM_LOSS_SYM is True
    # _delete_ semantics: OPTIMIZER_CFG replaced, not merged with the base's
    assert set(ref.SOLVER.OPTIMIZER_CFG.keys()) == {"type", "lr", "weight_decay"}

    (tmp_path / "_base_").mkdir()
    (tmp_path / "exp").mkdir()
    (tmp_path / "_base_" / "common.py").write_text(
        "SOLVER = dict(IMS_PER_BATCH=24, OPTIMIZER_CFG=dict(type='RMSprop', lr=1e-4, momentum=0.0, weight_decay=0))\n"
        "MODEL = dict(CDPN=dict(NAME='GDRN', PNP_NET=dict(PM_LOSS_SYM=False, PM_LW=1.0)))\n")
    (tmp_path / "_base_" / "model.py").write_text("_base_ = './common.py'\nMODEL = dict(CDPN=dict(TASK='rot'))\n")
    (tmp_path / "exp" / "a6.py").write_text(
        "_base_ = ['../_base_/model.py']\n"
        "SOLVER = dict(OPTIMIZER_CFG=dict(_delete_=True, type='Ranger', lr=1e-4, weight_decay=0))\n"
        "MODEL = dict(CDPN=dict(PNP_NET=dict(PM_LOSS_SYM=True)))\n")
    cfg = postprocess_like_main_gdrn(Config.fromfile(str(tmp_path / "exp" / "a6.py")), device="cpu")
    assert cfg.SOLVER.OPTIMIZER_CFG.to_dict() == {"type": "Ranger", "lr": 1e-4, "weight_decay": 0}
    assert cfg.SOLVER.IMS_PER_BATCH == 24 and cfg.SOLVER.BASE_LR == 1e-4
    assert cfg.MODEL.CDPN.to_dict() == {"NAME": "GDRN", "TASK": "rot", "PNP_NET": {"PM_LOSS_SYM": True, "PM_LW": 1.0}}


def test_ranger_matches_reference_algorithm():
    """Our multi-tensor Ranger against a literal per-parameter restatement of ranger.py:100-200."""
    import math

    from gdr_net_b200.solver import Ranger

    torch.manual_seed(0)
    ps = [torch.randn(8, 4, 3, 3), torch.randn(16, 8), torch.randn(5)]
    a = [p.clone().requires_grad_(True) for p in ps]
    b = [p.clone() for p in ps]
    opt = Ranger(a, lr=1e-2)
    st = [dict(step=0, m=torch.zeros_like(p), v=torch.zeros_like(p), slow=p.clone()) for p in b]
    for it in range(14):
        grads = [torch.randn_like(p) for p in ps]
        for p, g in zip(a, grads):
            p.grad = g.clone()
        opt.step()
        for p, g, s in zip(b, grads, st):
            g = g.clone()
            if g.dim() > 1:
                g -= g.mean(dim=tuple(range(1, g.dim())), keepdim=True)
            s["step"] += 1
            s["v"].mul_(0.999).addcmul_(g, g, value=0.001)
            s["m"].mul_(0.95).add_(g, alpha=0.05)
            b2t = 0.999 ** s["step"]
            nmax = 2 / 0.001 - 1
            nsma = nmax - 2 * s["step"] * b2t / (1 - b2t)
            if nsma > 5:
                ss = math.sqrt((1 - b2t) * (nsma - 4) / (nmax - 4) * (nsma - 2) / nsma * nmax / (nmax - 2)) / (1 - 0.95 ** s["step"])
                p.addcdiv_(s["m"], s["v"].sqrt().add_(1e-5), value=-ss * 1e-2)
            else:
                p.add_(s["m"], alpha=-1e-2 / (1 - 0.95 ** s["step"]))
            if s["step"] % 6 == 0:
                s["slow"].add_(p - s["slow"], alpha=0.5)
                p.copy_(s["slow"])
    for x, y in zip(a, b):
        assert torch.allclose(x.detach(), y, rtol=1e-5, atol=1e-6)


def test_batch_data_matches_reference_collate_keys():
    """train_harness.batch_data = the reference's collate (engine_utils.py:6-60): same keys, dtypes and shapes."""
    from gdr_net_b200 import synth
    from gdr_net_b200.train_harness import batch_data, forward_kwargs

    b = synth.make_batch(3, seed=4, with_sym=True)
    data = []
    for i in range(3):  # per-sample dicts as the reference's dataset emits them (data_loader.py:617-632)
        d = dict(roi_img=b["roi_img"][i], roi_cls=int(b["roi_cls"][i]), roi_coord_2d=b["roi_coord_2d"][i], cam=b["roi_cam"][i],
                 bbox_center=b["roi_center"][i].double(), roi_wh=b["roi_wh"][i], resize_ratio=float(b["resize_ratio"][i]),
                 roi_extent=b["roi_extent"][i], trans_ratio=b["roi_trans_ratio"][i], roi_xyz=b["roi_xyz"][i],
                 roi_mask_trunc=b["roi_mask_trunc"][i], roi_mask_visib=b["roi_mask_visib"][i], roi_mask_obj=b["roi_mask_obj"][i],
                 roi_region=b["roi_region"][i].int(), ego_rot=b["ego_rot"][i], trans=b["trans"][i], roi_points=b["roi_points"][i],
                 sym_info=b["sym_info"][i])
        data.append(d)
    out = batch_data(None, data, device="cpu")
    for k in ("roi_img", "roi_coord_2d", "roi_cam", "roi_center", "roi_wh", "resize_ratio", "roi_extent", "roi_trans_ratio", "roi_xyz",
              "roi_mask_trunc", "roi_mask_visib", "roi_mask_obj", "ego_rot", "trans", "roi_points"):
        assert out[k].dtype == torch.float32 and torch.allclose(out[k], b[k].float()), k
    assert out["roi_region"].dtype == torch.long and torch.equal(out["roi_region"], b["roi_region"])
    assert out["roi_cls"].dtype == torch.long and len(out["sym_info"]) == 3
    kw = forward_kwargs(out, train=True)
    import inspect

    assert set(kw) <= set(inspect.signature(G.GDRN.forward).parameters)
    test = batch_data(None, data, device="cpu", phase="test")
    assert "roi_xyz" not in test and "roi_cam" in test


def test_ranger_matches_reference_golden(golden_dir):
    """solver.Ranger against the UNMODIFIED reference optimizer (lib/torch_utils/solver/ranger.py), whose parameters after 14 steps
    on seeded gradients are stored in tests/golden/ranger_14steps.npz (oracle/make_golden_ranger.py)."""
    import os

    import numpy as np

    from gdr_net_b200.solver import Ranger

    g = np.load(os.path.join(golden_dir, "ranger_14steps.npz"))
    for tag, wd in (("wd0", 0.0), ("wd1e-2", 1e-2)):
        ps = [torch.from_numpy(g[f"p0_{i}"]).clone().requires_grad_(True) for i in range(3)]
        opt = Ranger(ps, lr=1e-2, weight_decay=wd)
        for t in range(14):
            for i, p in enumerate(ps):
                p.grad = torch.from_numpy(g[f"g{t}_{i}"]).clone()
            opt.step()
        for i, p in enumerate(ps):
            assert torch.allclose(p.detach(), torch.from_numpy(g[f"{tag}_p{i}"]), rtol=1e-5, atol=1e-6), (tag, i)


def test_batch_data_matches_reference_golden(golden_dir):
    """train_harness.batch_data against the UNMODIFIED reference collate (engine_utils.py:6-60): identical key set, dtypes, shapes and
    tensor bytes (tests/golden/batch_data_b3.json, made by oracle/make_golden_batch_data.py on the same seeded per-sample dicts)."""
    import hashlib
    import json
    import os

    from gdr_net_b200.train_harness import batch_data
    from oracle.make_golden_batch_data import per_sample_dicts

    gold = json.load(open(os.path.join(golden_dir, "batch_data_b3.json")))["train"]
    out = batch_data(None, per_sample_dicts(), device="cpu")
    assert set(out) == set(gold), (sorted(out), sorted(gold))
    for k, want in gold.items():
        v = out[k]
        if "dtype" in want:
            assert str(v.dtype) == want["dtype"] and list(v.shape) == want["shape"], (k, v.dtype, tuple(v.shape), want)
            assert hashlib.sha1(v.contiguous().numpy().tobytes()).hexdigest() == want["sha1"], k
        else:
            assert type(v).__name__ == want["type"] and len(v) == want["len"], k
