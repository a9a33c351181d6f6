"""RPMNet's matching tail on the GPU (l3d_feature_square_distance, l3d_sinkhorn, l3d_rpm_match_tail,
l3d_weighted_rigid_transform) against the real-reference fixture, the numpy oracle at RPMNet's sizes and — where
the staged reference package exists — the reference's own functions run on this GPU."""
import numpy as np
import pytest
import torch

from oracle import rpm as orpm

pytestmark = pytest.mark.gpu
DEV = "cuda"
T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def test_tail_against_reference_fixture(golden_dir):
    from learning3d_b200.models import rpmnet as R
    g = np.load(f"{golden_dir}/rpm_tail.npz")
    fs, fr = T(g["feat_src"]), T(g["feat_ref"])
    d = R.match_features(fs, fr)
    np.testing.assert_allclose(d.cpu().numpy(), g["dist"], atol=3e-5)
    from learning3d_b200.utils._ops import feature_square_distance
    aff = feature_square_distance(fs, fr, T(g["beta"]), T(g["alpha"]))
    np.testing.assert_allclose(aff.cpu().numpy(), g["affinity"], atol=2e-4)
    affr = T(g["affinity"])
    np.testing.assert_allclose(R.sinkhorn(affr, 5, True).cpu().numpy(), g["log_perm"], rtol=3e-6, atol=3e-5)
    np.testing.assert_allclose(R.sinkhorn(affr, 3, False).cpu().numpy(), g["log_noslack"], rtol=3e-6, atol=3e-5)
    perm, weighted, rs = R.match_tail(affr, T(g["xyz_ref"]), 5, True)
    np.testing.assert_allclose(perm.cpu().numpy(), g["perm"], rtol=2e-4, atol=1e-7)
    np.testing.assert_allclose(weighted.cpu().numpy(), g["weighted"], atol=1e-5)
    np.testing.assert_allclose(rs.cpu().numpy(), g["rowsum"], rtol=2e-4, atol=1e-12)
    Tm = R.compute_rigid_transform(T(g["xyz_src"]), T(g["weighted"]), T(g["rowsum"]))
    np.testing.assert_allclose(Tm.cpu().numpy(), g["T"], atol=1e-5)
    T2 = R.compute_rigid_transform(T(g["a2"]), T(g["b2"]), T(g["w2"]))
    np.testing.assert_allclose(T2.cpu().numpy(), g["T2"], atol=1e-5)


@pytest.mark.parametrize("B,J,K,C", [(8, 717, 717, 96), (2, 1024, 1000, 96), (1, 33, 257, 13), (3, 128, 64, 200)])
def test_tail_against_oracle_at_size(B, J, K, C):
    """RPMNet's own sizes (717 points after its crop, 96-d PPFNet features) and ragged ones."""
    from learning3d_b200.models import rpmnet as R
    from learning3d_b200.utils._ops import feature_square_distance
    rng = np.random.default_rng(B * J + K)
    fs = (0.3 * rng.standard_normal((B, J, C))).astype(np.float32)
    fr = (0.3 * rng.standard_normal((B, K, C))).astype(np.float32)
    n = min(J, K) // 2
    fr[:, :n] = fs[:, :n] + 0.03 * rng.standard_normal((B, n, C)).astype(np.float32)     # true matches
    d = R.match_features(T(fs), T(fr)).cpu().numpy()
    want = orpm.square_distance(fs, fr)
    mag = (fs.astype(np.float64) ** 2).sum(-1)[:, :, None] + (fr.astype(np.float64) ** 2).sum(-1)[:, None, :]
    assert (np.abs(d - want) / (mag + 1e-6)).max() < 4e-6
    beta = (1.0 + rng.random(B)).astype(np.float32); alpha = rng.random(B).astype(np.float32)
    aff = feature_square_distance(T(fs), T(fr), T(beta), T(alpha))
    np.testing.assert_allclose(aff.cpu().numpy(), -beta[:, None, None] * (want - alpha[:, None, None]), atol=3e-4)
    affn = aff.cpu().numpy()
    for slack, it in ((True, 5), (False, 2)):
        got = R.sinkhorn(aff, it, slack).cpu().numpy()
        np.testing.assert_allclose(got, orpm.sinkhorn(affn, it, slack), rtol=3e-6, atol=5e-5)
    xyz = (rng.random((B, K, 3)) - 0.5).astype(np.float32)
    perm, weighted, rs = R.match_tail(aff, T(xyz), 5, True)
    op, ow, ors = orpm.match_tail(affn, xyz, 5, True)
    np.testing.assert_allclose(perm.cpu().numpy(), op, rtol=3e-4, atol=1e-7)
    np.testing.assert_allclose(weighted.cpu().numpy(), ow, atol=2e-5)
    np.testing.assert_allclose(rs.cpu().numpy(), ors, rtol=2e-4, atol=1e-12)
    src = (rng.random((B, J, 3)) - 0.5).astype(np.float32)
    Tm = R.compute_rigid_transform(T(src), weighted, rs).cpu().numpy()
    np.testing.assert_allclose(Tm, orpm.compute_rigid_transform(src, weighted.cpu().numpy(), rs.cpu().numpy()), atol=2e-5)


def test_tail_gradients_take_the_torch_path():
    from learning3d_b200.models import rpmnet as R
    torch.manual_seed(0)
    fs = torch.randn(2, 50, 16, device=DEV, requires_grad=True)
    fr = torch.randn(2, 60, 16, device=DEV)
    d = R.match_features(fs, fr)
    lp = R.sinkhorn(-d, 3, True)
    w = torch.exp(lp).sum(2)
    Tm = R.compute_rigid_transform(torch.rand(2, 50, 3, device=DEV), torch.rand(2, 50, 3, device=DEV), w)
    Tm.sum().backward()
    assert fs.grad is not None and torch.isfinite(fs.grad).all()
    # and the forward values of both paths agree
    with torch.no_grad():
        np.testing.assert_allclose(R.match_features(fs, fr).cpu().numpy(), d.detach().cpu().numpy(), atol=1e-4)
        np.testing.assert_allclose(R.sinkhorn(-d.detach(), 3, True).cpu().numpy(), lp.detach().cpu().numpy(), atol=5e-5)


def _check_rpm_tail(R, golden_dir):
    """RPMNet's matching tail through the rpmnet module `R` against what the reference's own rpmnet functions,
    unmodified, returned on a B200 (tests/golden/make_golden_gpu.py, seeded samples)."""
    from oracle import seeded
    g = np.load(f"{golden_dir}/ref_gpu.npz")
    with torch.no_grad():
        d, lp, T = seeded.rpm_tail(R, *[t.to(DEV) for t in seeded.rpm_inputs()])
    np.testing.assert_allclose(d.cpu().numpy().reshape(-1)[seeded.sample_index(d.numel(), 1024, "rpm_d")], g["rpm_d"], atol=1e-4)
    np.testing.assert_allclose(lp.cpu().numpy().reshape(-1)[seeded.sample_index(lp.numel(), 1024, "rpm_lp")], g["rpm_lp"], atol=2e-4)
    np.testing.assert_allclose(T.cpu().numpy(), g["rpm_T"], atol=2e-5)


def test_rpmnet_tail_matches_reference_fixture(golden_dir):
    """Our rpmnet functions (learning3d_b200.models.rpmnet) return what the reference's returned."""
    from learning3d_b200.models import rpmnet as ours
    _check_rpm_tail(ours, golden_dir)


def test_square_distance_dispatch_and_reference_rpmnet_rebound(golden_dir):
    """learning3d_b200.utils.square_distance accepts C != 3 now; the reference's own rpmnet functions, rebound to
    libl3d_b200.so (learning3d_b200.bind), return what the unmodified ones returned."""
    from learning3d_b200.utils import square_distance
    from oracle import ref_pkg
    x = torch.randn(2, 40, 7, device=DEV); y = torch.randn(2, 30, 7, device=DEV)
    np.testing.assert_allclose(square_distance(x, y).cpu().numpy(), orpm.square_distance(x.cpu().numpy(), y.cpu().numpy()), atol=1e-4)
    if ref_pkg.reference_root() is None:
        pytest.skip("reference package not staged")
    from learning3d_b200 import bind
    ref = ref_pkg.import_reference()
    bind.bind(ref)
    try:
        _check_rpm_tail(ref.models.rpmnet, golden_dir)
    finally:
        bind.unbind(ref)


def test_knn_point_on_features():
    """knn_point (model_common_utils.py:84-100) with C != 3: Gram matrix + selection; values sqrt(d2) within the GEMM
    tolerance, indices equal the fp64 top-k wherever the k / k+1 gap exceeds it."""
    from learning3d_b200.utils import knn_point
    torch.manual_seed(2)
    B, N, M, C, k = 2, 300, 120, 32, 9
    data = torch.randn(B, N, C, device=DEV); query = torch.randn(B, M, C, device=DEV)
    val, idx = knn_point(k, data, query)
    d2 = ((query.double()[:, :, None, :] - data.double()[:, None, :, :]) ** 2).sum(-1)           # [B, M, N]
    top = torch.topk(d2, k + 1, dim=-1, largest=False)
    np.testing.assert_allclose(val.double().cpu().numpy(), top.values[..., :k].sqrt().cpu().numpy(), atol=2e-4)
    clear = (top.values[..., k] - top.values[..., k - 1]) > 1e-3
    same = (idx.sort(-1)[0] == top.indices[..., :k].sort(-1)[0]).all(-1)
    assert same[clear].all() and clear.float().mean() > 0.9
