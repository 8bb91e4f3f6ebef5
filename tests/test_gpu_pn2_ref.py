"""GPU: pins the point-cloud ops against the outputs of the REFERENCE's own CUDA kernels.

tests/golden/pn2_ref.pt holds what the reference's pointnet2._ext kernels returned on a B200 for every case below
(tools/make_golden_pn2_ref.py runs them from oracle/_ref/, the extension oracle/build_ref_ext.py compiles from the reference
sources): per output its SHA-256 and a fixed sample of its rows, which makes a mismatch readable.  Both the C restatement
(oracle/pn2_oracle.c) and the sam6d_b200 kernels must reproduce those index outputs bit for bit."""
import hashlib
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import pn2     # noqa: E402

FPS_CASES = [(4, 2048, 196, False), (2, 2048, 196, True), (2, 1000, 100, False), (1, 5000, 64, False), (2, 300, 40, True)]
CLUSTER_CASES = [(1, 210000, 2048), (2, 50000, 512), (3, 4097, 100), (1, 106496, 300), (1, 106497, 300)]
BALL_QUERY_CASES = [(2048, 0.1, 32), (2048, 0.2, 64), (700, 0.3, 16)]


@pytest.fixture(scope="module")
def gold(golden_dir):
    return torch.load(os.path.join(golden_dir, "pn2_ref.pt"), weights_only=False)


def _clouds(b, n, seed, dup=False):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(b, n, 3, generator=g)
    x = x / x.norm(dim=2, keepdim=True) * (0.5 + 0.5 * torch.rand(b, n, 1, generator=g))
    if dup:
        pick = torch.randint(0, n // 6, (b, n), generator=g)
        x = torch.gather(x, 1, pick.unsqueeze(2).expand(b, n, 3))
    return x.contiguous()


def gather_group_inputs():
    g = torch.Generator().manual_seed(3)
    pts = torch.randn(2, 9, 500, generator=g)
    idx = torch.randint(0, 500, (2, 77), generator=g, dtype=torch.int32)
    gi = torch.randint(0, 500, (2, 77, 8), generator=g, dtype=torch.int32)
    return pts, idx, gi


def sha256(t):
    return hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).hexdigest()


def summarize(t, n_rows=32):
    """SHA-256, dtype and shape of a whole output, and a fixed sample of its rows (a row = the last axis)"""
    t = t.detach().cpu().contiguous()
    rows = t.reshape(-1, t.shape[-1])
    pick = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:n_rows].sort()[0]
    return dict(sha256=sha256(t), dtype=str(t.dtype), shape=tuple(t.shape), rows=pick, sample=rows[pick].clone())


def _assert_inputs(gold, key, *inputs):
    assert [sha256(x) for x in inputs] == gold[key]["input_sha256"], f"{key}: inputs differ from those the golden was made from"


def _assert_reference(got, gold, key, what):
    want, have = gold[key], summarize(got)
    assert (have["dtype"], have["shape"]) == (want["dtype"], want["shape"]), f"{what}: {key}"
    assert torch.equal(have["sample"], want["sample"]), f"{what} != reference CUDA kernel: {key}, sampled rows {want['rows'].tolist()}"
    assert have["sha256"] == want["sha256"], f"{what} != reference CUDA kernel: {key}"


@pytest.mark.parametrize("b,n,m,dup", FPS_CASES)
def test_fps_matches_reference_kernel(gold, b, n, m, dup):
    from sam6d_b200 import ops
    key = f"fps_{b}_{n}_{m}_{int(dup)}"
    x = _clouds(b, n, n + m, dup)
    _assert_inputs(gold, key, x)
    _assert_reference(pn2.furthest_point_sampling(x, m), gold, key, "C restatement")
    _assert_reference(ops.furthest_point_sampling(x.cuda(), m), gold, key, "sam6d_b200 kernel")


@pytest.mark.parametrize("b,n,m", CLUSTER_CASES)
def test_fps_cluster_kernel_matches_reference_kernel(gold, b, n, m):
    """large clouds: the thread-block-cluster FPS (8 / 16 CTAs per cloud, points in distributed shared memory) against the
    reference's own kernel and the one-CTA kernel; 210 000 -> 2048 is the template bank of get_obj_feats
    (PEM/model/feature_extraction.py:170-181).  The two kernels' times are printed next to each other."""
    from sam6d_b200 import ops
    key = f"fps_cluster_{b}_{n}_{m}"
    x = _clouds(b, n, n + m, dup=(n == 50000))
    _assert_inputs(gold, key, x)
    x = x.cuda()
    _assert_reference(ops.furthest_point_sampling(x, m), gold, key, "cluster FPS")
    _assert_reference(ops.furthest_point_sampling_single_cta(x, m), gold, key, "single-CTA FPS")

    def t_ms(fn):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1)
    print("FPS", dict(b=b, n=n, m=m, cluster_ms=t_ms(lambda: ops.furthest_point_sampling(x, m)),
                      single_cta_ms=t_ms(lambda: ops.furthest_point_sampling_single_cta(x, m))))


@pytest.mark.parametrize("n,r,ns", BALL_QUERY_CASES)
def test_ball_query_matches_reference_kernel(gold, n, r, ns):
    from sam6d_b200 import ops
    key = f"ball_query_{n}_{r}_{ns}"
    x = _clouds(3, n, n + ns)
    _assert_inputs(gold, key, x)
    _assert_reference(pn2.ball_query(x, x, r, ns), gold, key, "C restatement")
    _assert_reference(ops.ball_query(x.cuda(), x.cuda(), r, ns), gold, key, "sam6d_b200 kernel")


def test_gather_group_match_reference_kernel(gold):
    from sam6d_b200 import ops
    pts, idx, gi = gather_group_inputs()
    _assert_inputs(gold, "gather_points", pts, idx)
    _assert_inputs(gold, "group_points", pts, gi)
    _assert_reference(ops.gather_points(pts.cuda(), idx.cuda()), gold, "gather_points", "sam6d_b200 kernel")
    _assert_reference(ops.group_points(pts.cuda(), gi.cuda()), gold, "group_points", "sam6d_b200 kernel")
