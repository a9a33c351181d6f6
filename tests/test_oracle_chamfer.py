"""CPU: Chamfer restatement in the C oracle against fixtures made by the reference's own
extension (cd.forward / cd.backward on CPU)."""
import numpy as np
import pytest


@pytest.mark.parametrize("tag", ["c1", "ragged"])
def test_chamfer_forward_backward_bit_exact(oracle_mod, golden_dir, tag):
    g = np.load(f"{golden_dir}/chamfer_{tag}.npz")
    d1, d2, i1, i2 = oracle_mod.chamfer_forward(g["xyz1"], g["xyz2"])
    assert np.array_equal(d1, g["dist1"]) and np.array_equal(d2, g["dist2"])
    assert np.array_equal(i1, g["idx1"]) and np.array_equal(i2, g["idx2"])
    gx1, gx2 = oracle_mod.chamfer_backward(g["xyz1"], g["xyz2"], g["graddist1"], g["graddist2"], i1, i2)
    assert np.array_equal(gx1, g["gradxyz1"]) and np.array_equal(gx2, g["gradxyz2"])


@pytest.mark.parametrize("tag", ["c1", "ragged"])
def test_chamfer_loss_and_grads(oracle_mod, golden_dir, tag):
    g = np.load(f"{golden_dir}/chamfer_{tag}.npz")
    loss = oracle_mod.chamfer_loss(g["xyz1"], g["xyz2"])
    assert abs(loss - float(g["loss"])) < 1e-6
    assert abs(loss - float(g["loss_torch"])) < 1e-6      # pure-torch fallback gives the same value
    l1, l2 = oracle_mod.chamfer_loss_grads(g["xyz1"], g["xyz2"])
    np.testing.assert_allclose(l1, g["loss_grad1"], rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(l2, g["loss_grad2"], rtol=1e-5, atol=1e-9)


def test_chamfer_against_compiled_reference(oracle_mod, golden_dir):
    """The reference's compiled extension (cd.forward, its CPU nnsearch) on a ragged pair, recorded by
    tests/golden/make_golden.py (gen_compiled_chamfer): bit-exact."""
    g = np.load(f"{golden_dir}/chamfer_compiled.npz")
    rng = np.random.default_rng(7)
    a, b = rng.random((2, 257, 3), dtype=np.float32), rng.random((2, 130, 3), dtype=np.float32)
    o = oracle_mod.chamfer_forward(a, b)
    for name, y in zip(("dist1", "dist2", "idx1", "idx2"), o):
        assert np.array_equal(g[name], y), name


def test_identical_clouds_give_nonfinite_grads(oracle_mod):
    # sqrt(0) -> inf * 0 -> NaN in the reference (SURVEY.md App. A): reproduced, not "fixed"
    a = np.random.default_rng(0).random((1, 16, 3), dtype=np.float32)
    g1, _ = oracle_mod.chamfer_loss_grads(a, a.copy())
    assert not np.isfinite(g1).all()
