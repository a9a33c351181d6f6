"""CPU: grouping-family restatements (oracle/l3d_oracle_group.c) against fixtures produced by the
real reference's pure-torch helpers (tests/golden/make_golden.py gen_group)."""
import numpy as np
import pytest

from oracle import group as og


@pytest.fixture(scope="module")
def g(golden_dir):
    return np.load(f"{golden_dir}/group.npz")


def test_query_ball_point_variants(oracle_mod, g):
    idx, cnt = og.query_ball_point(0.25, 16, g["xyz"], g["new_xyz"], want_cnt=True)
    assert np.array_equal(idx, g["qbp_idx"]) and np.array_equal(cnt, g["qbp_cnt"])
    assert np.array_equal(og.query_ball_point(0.05, 8, g["xyz"], g["new_xyz"]), g["qbp_small_r"])
    itself = np.tile(np.arange(0, 300, 3)[None], (2, 1))
    assert np.array_equal(og.query_ball_point(0.25, 16, g["xyz"], g["new_xyz"], itself=itself), g["qbp_itself"])


def test_query_ball_point_no_hit_row_is_N(oracle_mod):
    xyz = np.zeros((1, 10, 3), np.float32)
    q = np.full((1, 2, 3), 5.0, np.float32)
    assert (og.query_ball_point(0.1, 4, xyz, q) == 10).all()       # what the reference's sort leaves
    assert (og.pn2_ball_query(0.1, 4, xyz, q) == 0).all()          # pointnet2: pre-zeroed idx


def test_fps_torch_variants(oracle_mod, g):
    assert np.array_equal(og.farthest_point_sample(g["xyz"], 64), g["fps_first"])
    assert np.array_equal(og.farthest_point_sample(g["xyz"], 50), g["fps_pointconv"])
    for key in ("fps_random_seed7", "fps_ppf_seed8"):
        ref = g[key]
        assert np.array_equal(og.farthest_point_sample(g["xyz"], 40, start=ref[:, 0].copy()), ref)


def test_fps_pointnet2_simulation_properties(oracle_mod):
    rng = np.random.default_rng(0)
    x = rng.random((2, 1000, 3), dtype=np.float32)
    idx, temp = og.pn2_fps(x, 128)
    assert (idx[:, 0] == 0).all()
    assert all(len(set(r)) == 128 for r in idx)
    # each pick is an arg-max of the running min-distance: recompute with the same fma distance
    d = np.full((2, 1000), 1e10, np.float32)
    for j in range(1, 128):
        c = x[np.arange(2), idx[:, j - 1]]
        dx, dy, dz = [(x[..., a] - c[:, None, a]).astype(np.float32) for a in range(3)]
        dd = np.float32(dy * dy)
        dd = (dx.astype(np.float64) * dx + dd).astype(np.float32)
        dd = (dz.astype(np.float64) * dz + dd).astype(np.float32)
        d = np.minimum(d, dd)
        assert np.array_equal(d[np.arange(2), idx[:, j]], d.max(-1))
    # tie rule on duplicated points: deterministic and distinct picks
    xd = np.tile(x[:, :100], (1, 4, 1))
    i2, _ = og.pn2_fps(xd, 50)
    assert np.array_equal(i2, og.pn2_fps(xd, 50)[0])


def test_index_points_density_and_compositions(oracle_mod, g):
    assert np.array_equal(og.index_points(g["feats"], g["qbp_idx"]), g["index_points"])
    np.testing.assert_allclose(og.compute_density(g["xyz"], 0.1), g["density"], rtol=2e-6)
    # pointconv sample_and_group = FPS(start 0) -> kNN(sqdist) -> gather; compare the pieces
    fps = og.farthest_point_sample(g["xyz"], 32)
    new_xyz = og.index_points(g["xyz"], fps)
    assert np.array_equal(new_xyz, g["pc_sg_new_xyz"])
    idx = oracle_mod.knn_sqdist(g["xyz"], new_xyz, 8)
    assert np.array_equal(np.sort(idx, -1), np.sort(g["pc_sg_idx"], -1))


def test_group_gather_interpolate_adjoints(oracle_mod):
    rng = np.random.default_rng(1)
    pts = rng.standard_normal((2, 7, 50)).astype(np.float32)
    idx = rng.integers(0, 50, (2, 11, 4)).astype(np.int32)
    out = og.pn2_group_points(pts, idx)
    assert out.shape == (2, 7, 11, 4)
    assert np.array_equal(out[1, 3, 5, 2], pts[1, 3, idx[1, 5, 2]])
    go = rng.standard_normal(out.shape).astype(np.float32)
    gp = og.pn2_group_points_grad(go, idx, 50)
    assert abs(float((out.astype(np.float64) * go).sum()) - float((pts.astype(np.float64) * gp).sum())) < 1e-3
    i3 = rng.integers(0, 50, (2, 30, 3)).astype(np.int32)
    w = rng.random((2, 30, 3)).astype(np.float32)
    o3 = og.pn2_three_interpolate(pts, i3, w)
    g3 = rng.standard_normal(o3.shape).astype(np.float32)
    gp3 = og.pn2_three_interpolate_grad(g3, i3, w, 50)
    assert abs(float((o3.astype(np.float64) * g3).sum()) - float((pts.astype(np.float64) * gp3).sum())) < 1e-3


# ---- the reference's own CUDA kernels pin the oracle ---------------------------------------------------
def test_reference_cuda_kernels_agree_with_oracle(oracle_mod, golden_dir):
    """Outputs of the reference's pointnet2 kernels on a B200, recorded by tests/golden/make_golden_gpu.py as one
    SHA-256 digest per cloud (every query row), bit-exact against the oracle."""
    from oracle import seeded
    D = seeded.array_digest
    g = np.load(f"{golden_dir}/ref_gpu.npz")
    rng = np.random.default_rng(12)
    B, N, S = 4, 2048, 512
    xyz = (rng.random((B, N, 3), dtype=np.float32) * 2 - 1).astype(np.float32)
    new_xyz = np.ascontiguousarray(xyz[:, :S])
    # ball query (K7)
    assert np.array_equal(g["pn2_ball"], D(og.pn2_ball_query(0.2, 16, xyz, new_xyz)))
    # kNN (K11) and three_nn (K12)
    for k in (8, 64):
        od2, oi = oracle_mod.pn2_knn(k, new_xyz, xyz)
        assert np.array_equal(g["pn2_knn%d_idx" % k], D(oi)) and np.array_equal(g["pn2_knn%d_dist2" % k], D(od2))
    od3, oi3 = oracle_mod.pn2_knn(3, new_xyz, xyz)
    assert np.array_equal(g["pn2_three_nn_idx"], D(oi3)) and np.array_equal(g["pn2_three_nn_dist2"], D(od3))
    # FPS (K10), including a duplicated cloud (tie rule of the shared-memory tree)
    for tag, cloud in (("", xyz), ("_dup", np.tile(xyz[:, :256], (1, 4, 1)))):
        want, wtemp = og.pn2_fps(cloud, 300)
        assert np.array_equal(g["pn2_fps%s_idx" % tag], want)
        assert np.array_equal(g["pn2_fps%s_temp" % tag], D(wtemp))
    # group / interpolate
    feats = rng.standard_normal((B, 10, N)).astype(np.float32)
    gi = rng.integers(0, N, (B, 64, 8)).astype(np.int32)
    w = rng.random((B, S, 3)).astype(np.float32); ti = rng.integers(0, N, (B, S, 3)).astype(np.int32)
    assert np.array_equal(g["pn2_group"], D(og.pn2_group_points(feats, gi)))
    assert np.array_equal(g["pn2_interp"], D(og.pn2_three_interpolate(feats, ti, w)))
