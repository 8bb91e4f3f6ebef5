"""tools/make_golden_vit_gather.py -- needs a checkout of the reference SAM-6D repository.

Pins oracle/vit_oracle.chosen_pixel_feats against the reference's own get_chosen_pixel_feats
(Pose_Estimation_Model/utils/model_utils.py:69-81), imported unmodified, on the seeded inputs of
tests/test_oracle_vit.py.  Writes tests/golden/vit_gather.pt.

Usage: python tools/make_golden_vit_gather.py <path of the SAM-6D directory of the reference>"""
import builtins
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from test_oracle_vit import gather_inputs  # noqa: E402


def main():
    pem = os.path.join(sys.argv[1], "Pose_Estimation_Model")
    builtins.__POINTNET2_SETUP__ = True              # model_utils imports pointnet2_utils, which then skips its CUDA extension
    sys.path[:0] = [os.path.join(pem, "utils"), os.path.join(pem, "model", "pointnet2")]
    import model_utils as mu
    img, choose = gather_inputs()
    gold = dict(meta=dict(source="get_chosen_pixel_feats of Pose_Estimation_Model/utils/model_utils.py (CPU)", torch=torch.__version__),
                feats=mu.get_chosen_pixel_feats(img, choose))
    out = os.path.join(ROOT, "tests", "golden", "vit_gather.pt")
    torch.save(gold, out)
    print(f"wrote {out}")


if __name__ == "__main__":
    main()
