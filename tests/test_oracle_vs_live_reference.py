"""CPU: the oracle against what the UNMODIFIED reference's pure-torch helpers (utils/model_common_utils.py,
pointconv_util.py, ppfnet_util.py) returned on these seeded inputs, beyond the other fixtures.  The reference's
outputs were recorded by tests/golden/make_golden.py (gen_live) into tests/golden/live_reference.npz; large
outputs as a seeded sample."""
import numpy as np
import pytest
import torch

from oracle import group as og


@pytest.fixture(scope="module")
def ref(golden_dir):
    return np.load(f"{golden_dir}/live_reference.npz")


@pytest.mark.parametrize("seed", range(4))
def test_knn_and_graph_feature_live(oracle_mod, ref, seed):
    rng = np.random.default_rng(500 + seed)
    B, N, k = int(rng.integers(1, 4)), int(rng.integers(40, 400)), int(rng.integers(1, 30))
    x = rng.random((B, 3, N), dtype=np.float32)
    xt = torch.from_numpy(x)
    rows = ref["knn%d_rows" % seed]
    want = ref["knn%d_idx" % seed].astype(np.int64)
    got = oracle_mod.knn_expansion(x, k)
    # torch.topk leaves the order of exactly tied keys unspecified: rows must agree unless their keys tie
    xx = (xt ** 2).sum(1, keepdim=True)
    pd = (-xx - (-2 * torch.matmul(xt.transpose(2, 1).contiguous(), xt)) - xx.transpose(2, 1).contiguous()).numpy()[:, rows]
    diff = np.argwhere(want != got[:, rows])
    for b, i, r in diff:
        assert pd[b, i, want[b, i, r]] == pd[b, i, got[b, rows[i], r]], (b, i, r)
    assert len(diff) <= 0.01 * want.size
    if len(diff) == 0:
        flat = ref["knn%d_feat_flat" % seed]
        assert np.array_equal(oracle_mod.graph_feature(x, got).reshape(-1)[flat], ref["knn%d_feat" % seed])


@pytest.mark.parametrize("seed", range(3))
def test_grouping_functions_live(oracle_mod, ref, seed):
    rng = np.random.default_rng(700 + seed)
    B, N, S = 2, int(rng.integers(50, 300)), int(rng.integers(5, 40))
    xyz = rng.random((B, N, 3), dtype=np.float32)
    new_xyz = np.ascontiguousarray(xyz[:, :S])
    flat = ref["group%d_sqdist_flat" % seed]
    assert np.array_equal(oracle_mod.square_distance(new_xyz, xyz).reshape(-1)[flat], ref["group%d_sqdist" % seed])
    r, ns = 0.25, int(rng.integers(2, 20))
    oi, oc = og.query_ball_point(r, ns, xyz, new_xyz, want_cnt=True)
    assert np.array_equal(oi, ref["group%d_ball_idx" % seed]) and np.array_equal(oc, ref["group%d_ball_cnt" % seed])
    assert np.array_equal(og.farthest_point_sample(xyz, S), ref["group%d_fps" % seed])
    k = int(rng.integers(1, 12))
    val, kidx = ref["group%d_knn_val" % seed], ref["group%d_knn_idx" % seed]
    ov, oi2 = oracle_mod.knn_point(k, xyz, new_xyz)
    same = oi2 == kidx
    assert same.mean() > 0.99                       # exact distance ties may order differently
    np.testing.assert_allclose(ov[same], val[same], rtol=2e-7, atol=1e-7)


@pytest.mark.parametrize("seed", range(2))
def test_pointconv_and_ppfnet_variants_live(oracle_mod, ref, seed):
    rng = np.random.default_rng(900 + seed)
    B, N, S = 2, int(rng.integers(64, 200)), int(rng.integers(8, 32))
    xyz = rng.random((B, N, 3), dtype=np.float32)
    new_xyz = np.ascontiguousarray(xyz[:, :S])
    # pointconv knn_point: topk(sorted=False) -> compare as sets per row (pointconv_util.py:107-118)
    ns = int(rng.integers(2, 16))
    want = np.sort(ref["pc%d_knn" % seed], axis=-1)
    got = np.sort(oracle_mod.knn_sqdist(xyz, new_xyz, ns), axis=-1)
    assert (want == got).mean() > 0.995
    # start-0 FPS (pointconv_util.py:60-83) and density (:199-209)
    assert np.array_equal(og.farthest_point_sample(xyz, S), ref["pc%d_fps" % seed])
    np.testing.assert_allclose(og.compute_density(xyz, 0.2), ref["pc%d_density" % seed], rtol=2e-6)
    # ppfnet ball query with the query's own index masked out (ppfnet_util.py:96-131)
    itself = np.tile(np.arange(S), (B, 1))
    want = ref["pc%d_ppf_ball" % seed]
    got = og.query_ball_point(0.3, 12, xyz, new_xyz, itself=itself)
    assert np.array_equal(want, got)
