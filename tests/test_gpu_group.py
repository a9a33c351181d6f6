"""GPU parity: grouping family through the C ABI / the drop-in Python modules, against the oracle, the
reference-generated fixtures (the oracle itself is pinned to the reference's own pointnet2 CUDA kernels by
tests/test_oracle_group.py::test_reference_cuda_kernels_agree_with_oracle)."""
import numpy as np
import pytest
import torch

from oracle import group as og

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.fixture(scope="module")
def g(golden_dir):
    return np.load(f"{golden_dir}/group.npz")


# ---- torch-semantics helpers vs the real reference's outputs ---------------------------------
def test_query_ball_point_golden(g):
    from learning3d_b200.utils import model_common_utils as mcu, pointconv_util as pcu, ppfnet_util as ppu
    xyz, new_xyz = T(g["xyz"]), T(g["new_xyz"])
    idx, cnt = mcu.query_ball_point(0.25, 16, xyz, new_xyz, get_cnt=True)
    assert np.array_equal(idx.cpu().numpy(), g["qbp_idx"]) and np.array_equal(cnt.cpu().numpy(), g["qbp_cnt"])
    assert np.array_equal(pcu.query_ball_point(0.05, 8, xyz, new_xyz).cpu().numpy(), g["qbp_small_r"])
    itself = torch.arange(0, 300, 3)[None].repeat(2, 1).to(DEV)
    assert np.array_equal(ppu.query_ball_point(0.25, 16, xyz, new_xyz, itself).cpu().numpy(), g["qbp_itself"])


def test_fps_golden(g):
    from learning3d_b200.utils import model_common_utils as mcu, pointconv_util as pcu, ppfnet_util as ppu
    xyz = T(g["xyz"])
    assert np.array_equal(mcu.farthest_point_sample(xyz, 64, start_with_first_point=True).cpu().numpy(), g["fps_first"])
    assert np.array_equal(pcu.farthest_point_sample(xyz, 50).cpu().numpy(), g["fps_pointconv"])
    torch.manual_seed(7)     # same CPU generator call as the reference -> same random start
    assert np.array_equal(mcu.farthest_point_sample(xyz, 40).cpu().numpy(), g["fps_random_seed7"])
    torch.manual_seed(8)
    assert np.array_equal(ppu.farthest_point_sample(xyz, 40).cpu().numpy(), g["fps_ppf_seed8"])


def test_index_points_density_square_distance_golden(g, golden_dir):
    from learning3d_b200.utils import index_points, square_distance
    from learning3d_b200.utils.pointconv_util import compute_density
    feats = T(g["feats"]).requires_grad_(True)
    out = index_points(feats, T(g["qbp_idx"]))
    assert np.array_equal(out.detach().cpu().numpy(), g["index_points"])
    go = torch.randn_like(out)
    out.backward(go)
    want = torch.zeros_like(feats)
    want.index_put_((torch.arange(2, device=DEV)[:, None, None].expand_as(T(g["qbp_idx"])), T(g["qbp_idx"])), go, accumulate=True)
    np.testing.assert_allclose(feats.grad.cpu().numpy(), want.detach().cpu().numpy(), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(compute_density(T(g["xyz"]), 0.1).cpu().numpy(), g["density"], rtol=1e-5)
    kp = np.load(f"{golden_dir}/knn_point.npz")
    assert np.array_equal(square_distance(T(kp["query"]), T(kp["data"])).cpu().numpy(), kp["sqdist"])


def test_sample_and_group_compositions_golden(g):
    from learning3d_b200.utils import pointconv_util as pcu, ppfnet_util as ppu
    xyz, feats, normals = T(g["xyz"]), T(g["feats"]), T(g["normals"])
    nx, npts, gnorm, gidx = pcu.sample_and_group(32, 8, xyz, feats)
    assert np.array_equal(nx.cpu().numpy(), g["pc_sg_new_xyz"])
    # reference kNN is topk(sorted=False): same neighbour SET per row
    assert np.array_equal(np.sort(gidx.cpu().numpy(), -1), np.sort(g["pc_sg_idx"], -1))
    torch.manual_seed(11)
    res, gxyz, fidx = ppu.sample_and_group_multi(20, 0.3, 12, xyz, normals, returnfps=True)
    assert np.array_equal(fidx.cpu().numpy(), g["ppf_fps"])
    assert np.array_equal(res["xyz"].cpu().numpy(), g["ppf_xyz"])
    assert np.array_equal(res["dxyz"].cpu().numpy(), g["ppf_dxyz"])
    np.testing.assert_allclose(res["ppf"].cpu().numpy(), g["ppf_ppf"], rtol=1e-5, atol=1e-6)
    res_all = ppu.sample_and_group_multi(-1, 0.3, 12, xyz, normals)
    np.testing.assert_allclose(res_all["ppf"].cpu().numpy(), g["ppf_all_ppf"], rtol=1e-5, atol=1e-6)


# ---- larger seeded cases vs the oracle ---------------------------------------------------------
@pytest.mark.parametrize("B,N,S,r,ns", [(16, 2048, 1024, 0.5, 16), (2, 1000, 333, 0.12, 64), (1, 50, 50, 0.01, 8)])
def test_ball_query_both_semantics_vs_oracle(B, N, S, r, ns):
    from learning3d_b200.utils.lib import pointnet2_utils as pu
    from learning3d_b200.utils import query_ball_point
    rng = np.random.default_rng(N + S)
    xyz = (rng.random((B, N, 3), dtype=np.float32) * 4 - 2).astype(np.float32)
    new_xyz = np.ascontiguousarray(xyz[:, :S])
    got = pu.ball_query(r, ns, T(xyz), T(new_xyz)).cpu().numpy()
    assert got.dtype == np.int32 and np.array_equal(got, og.pn2_ball_query(r, ns, xyz, new_xyz))
    idx, cnt = query_ball_point(r, ns, T(xyz), T(new_xyz), get_cnt=True)
    oi, oc = og.query_ball_point(r, ns, xyz, new_xyz, want_cnt=True)
    assert np.array_equal(idx.cpu().numpy(), oi) and np.array_equal(cnt.cpu().numpy(), oc)
    far = np.full((B, 3, 3), 100.0, np.float32)      # rows with no hit: 0 (pointnet2) / N (torch)
    assert (pu.ball_query(r, ns, T(xyz), T(far)).cpu().numpy() == 0).all()
    assert (query_ball_point(r, ns, T(xyz), T(far)).cpu().numpy() == N).all()


@pytest.mark.parametrize("B,N,M", [(16, 2048, 1024), (3, 1000, 256), (2, 513, 64), (1, 5000, 100), (2, 64, 64), (1, 8192, 32)])
def test_fps_vs_oracle(B, N, M):
    from learning3d_b200.utils.lib import pointnet2_utils as pu
    from learning3d_b200.utils.pointconv_util import farthest_point_sample
    rng = np.random.default_rng(N * 7 + M)
    xyz = rng.standard_normal((B, N, 3)).astype(np.float32)
    got = pu.furthest_point_sample(T(xyz), M).cpu().numpy()
    want, _ = og.pn2_fps(xyz, M)
    assert got.dtype == np.int32 and np.array_equal(got, want)
    got_t = farthest_point_sample(T(xyz), M).cpu().numpy()
    assert np.array_equal(got_t, og.farthest_point_sample(xyz, M))


def test_fps_tie_rules_on_duplicates():
    from learning3d_b200.utils.lib import pointnet2_utils as pu
    from learning3d_b200.utils.pointconv_util import farthest_point_sample
    rng = np.random.default_rng(5)
    base = rng.random((2, 150, 3), dtype=np.float32)
    xyz = np.tile(base, (1, 5, 1))                   # every point 5 times: constant ties
    assert np.array_equal(pu.furthest_point_sample(T(xyz), 100).cpu().numpy(), og.pn2_fps(xyz, 100)[0])
    assert np.array_equal(farthest_point_sample(T(xyz), 100).cpu().numpy(), og.farthest_point_sample(xyz, 100))


def test_group_gather_interpolate_vs_oracle():
    from learning3d_b200.utils.lib import pointnet2_utils as pu
    rng = np.random.default_rng(2)
    feats = rng.standard_normal((3, 67, 500)).astype(np.float32)
    idx = rng.integers(0, 500, (3, 128, 16)).astype(np.int32)
    f = T(feats).requires_grad_(True)
    out = pu.grouping_operation(f, T(idx))
    assert np.array_equal(out.detach().cpu().numpy(), og.pn2_group_points(feats, idx))
    go = torch.randn_like(out)
    out.backward(go)
    np.testing.assert_allclose(f.grad.cpu().numpy(), og.pn2_group_points_grad(go.cpu().numpy(), idx, 500), rtol=1e-4, atol=1e-4)
    gi = rng.integers(0, 500, (3, 77)).astype(np.int32)
    f2 = T(feats).requires_grad_(True)
    o2 = pu.gather_operation(f2, T(gi))
    assert np.array_equal(o2.detach().cpu().numpy(), og.pn2_group_points(feats, gi))
    o2.sum().backward()
    np.testing.assert_allclose(f2.grad.cpu().numpy(), og.pn2_group_points_grad(np.ones(o2.shape, np.float32), gi, 500), rtol=1e-5, atol=1e-5)
    i3 = rng.integers(0, 500, (3, 900, 3)).astype(np.int32)
    w = rng.random((3, 900, 3)).astype(np.float32)
    f3 = T(feats).requires_grad_(True)
    o3 = pu.three_interpolate(f3, T(i3), T(w))
    assert np.array_equal(o3.detach().cpu().numpy(), og.pn2_three_interpolate(feats, i3, w))
    g3 = torch.randn_like(o3)
    o3.backward(g3)
    np.testing.assert_allclose(f3.grad.cpu().numpy(), og.pn2_three_interpolate_grad(g3.cpu().numpy(), i3, w, 500), rtol=1e-4, atol=1e-4)


def test_pn2_knn_and_three_nn_api(oracle_mod):
    from learning3d_b200.utils.lib import pointnet2_utils as pu
    rng = np.random.default_rng(4)
    q = rng.random((2, 256, 3), dtype=np.float32); d = rng.random((2, 300, 3), dtype=np.float32)
    dist, idx = pu.knn(64, T(q), T(d))
    od2, oi = oracle_mod.pn2_knn(64, q, d)
    assert idx.dtype == torch.int32 and np.array_equal(idx.cpu().numpy(), oi)
    assert np.array_equal(dist.cpu().numpy(), np.sqrt(od2))
    dist3, idx3 = pu.three_nn(T(q), T(d))
    od3, oi3 = oracle_mod.pn2_knn(3, q, d)
    assert np.array_equal(idx3.cpu().numpy(), oi3) and np.array_equal(dist3.cpu().numpy(), np.sqrt(od3))


def test_query_and_group_module():
    from learning3d_b200.utils.lib import pointnet2_utils as pu
    rng = np.random.default_rng(6)
    xyz = rng.random((2, 400, 3), dtype=np.float32)
    feats = rng.standard_normal((2, 9, 400)).astype(np.float32)
    new_xyz = np.ascontiguousarray(xyz[:, :64])
    out = pu.QueryAndGroup(0.3, 16)(T(xyz), T(new_xyz), T(feats))
    idx = og.pn2_ball_query(0.3, 16, xyz, new_xyz)
    gx = og.pn2_group_points(np.ascontiguousarray(xyz.transpose(0, 2, 1)), idx) - new_xyz.transpose(0, 2, 1)[..., None]
    want = np.concatenate([gx, og.pn2_group_points(feats, idx)], 1)
    assert out.shape == (2, 12, 64, 16) and np.array_equal(out.cpu().numpy(), want)
    assert pu.GroupAll()(T(xyz), None, T(feats)).shape == (2, 12, 1, 400)
