"""tools/make_golden_pn2_ref.py -- needs a GPU and oracle/_ref/ (the reference's pointnet2._ext, compiled by
oracle/build_ref_ext.py).

Runs the reference's own FPS / ball-query / gather / group CUDA kernels on every case of tests/test_gpu_pn2_ref.py and writes
what they returned, summarised by that test's summarize() (SHA-256 of the full output + a fixed sample of rows), together
with the SHA-256 of the inputs, to tests/golden/pn2_ref.pt or the path given.

Usage: python tools/make_golden_pn2_ref.py [OUT]"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import build_ref_ext  # noqa: E402
import test_gpu_pn2_ref as t  # noqa: E402


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "pn2_ref.pt")
    ref = build_ref_ext.load_module()
    assert ref is not None, "oracle/_ref/ not built: run oracle/build_ref_ext.py where the reference sources are"
    gold = dict(meta=dict(source="reference pointnet2._ext kernels (oracle/_ref) on " + torch.cuda.get_device_name(0),
                          torch=torch.__version__))

    def put(key, got, *inputs):
        gold[key] = dict(t.summarize(got), input_sha256=[t.sha256(x) for x in inputs])

    for b, n, m, dup in t.FPS_CASES:
        x = t._clouds(b, n, n + m, dup)
        put(f"fps_{b}_{n}_{m}_{int(dup)}", ref.furthest_point_sampling(x.cuda(), m), x)
    for b, n, m in t.CLUSTER_CASES:
        x = t._clouds(b, n, n + m, dup=(n == 50000))
        put(f"fps_cluster_{b}_{n}_{m}", ref.furthest_point_sampling(x.cuda(), m), x)
    for n, r, ns in t.BALL_QUERY_CASES:
        x = t._clouds(3, n, n + ns)
        put(f"ball_query_{n}_{r}_{ns}", ref.ball_query(x.cuda(), x.cuda(), r, ns), x)
    pts, idx, gi = t.gather_group_inputs()
    put("gather_points", ref.gather_points(pts.cuda(), idx.cuda()), pts, idx)
    put("group_points", ref.group_points(pts.cuda(), gi.cuda()), pts, gi)
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    torch.save(gold, out)
    print(f"wrote {out}: {len(gold) - 1} outputs")


if __name__ == "__main__":
    main()
