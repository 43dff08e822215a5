"""TEST INFRASTRUCTURE ONLY -- golden values of the reference's own experiment configs: the MODEL and SOLVER sections that
`configs/gdrn/lm/a6_cPnP_lm13.py` and `configs/gdrn/ycbv/a6_cPnP_AugAAETrunc_BG0.5_Rsym_ycbv_real_pbr_visib20_10e.py` load to
(with their `_base_` chains and `_delete_` overrides).  The files are read from the reference tree by this project's own loader,
`gdr_net_b200.config.Config.fromfile` (the reference loads them with mmcv, which is not a dependency here), so the fixture records
this loader's reading of the reference's files.  Output: tests/golden/reference_configs.json.  Usage: python -m oracle.make_golden_configs"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gdr_net_b200.config import Config  # noqa: E402
from oracle import ref_shim  # noqa: E402

CONFIGS = {
    "lm13": "configs/gdrn/lm/a6_cPnP_lm13.py",
    "ycbv": "configs/gdrn/ycbv/a6_cPnP_AugAAETrunc_BG0.5_Rsym_ycbv_real_pbr_visib20_10e.py",
}


def main():
    if not os.path.isdir(ref_shim.REFERENCE_ROOT):
        raise RuntimeError(f"reference not found at {ref_shim.REFERENCE_ROOT}")
    gold = {}
    for tag, rel in CONFIGS.items():
        cfg = Config.fromfile(os.path.join(ref_shim.REFERENCE_ROOT, rel)).to_dict()
        gold[tag] = dict(file=rel, MODEL=cfg["MODEL"], SOLVER=cfg["SOLVER"])
    path = os.path.join(ROOT, "tests", "golden", "reference_configs.json")
    with open(path, "w") as f:
        json.dump(gold, f, indent=1, sort_keys=True)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
