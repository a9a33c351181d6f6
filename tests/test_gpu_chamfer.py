"""GPU parity: Chamfer kernels (through the C ABI) against the oracle, the golden fixtures made by
the reference's extension, and the outputs of the reference's CUDA kernels."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _fwd(a_np, b_np):
    from learning3d_b200.losses.cuda.chamfer_distance import ChamferDistanceFunction
    a = torch.from_numpy(a_np).to(DEV).requires_grad_(True)
    b = torch.from_numpy(b_np).to(DEV).requires_grad_(True)
    d1, d2 = ChamferDistanceFunction.apply(a, b)
    return a, b, d1, d2


@pytest.mark.parametrize("tag", ["c1", "ragged"])
def test_chamfer_golden_bit_exact(golden_dir, tag):
    g = np.load(f"{golden_dir}/chamfer_{tag}.npz")
    a, b, d1, d2 = _fwd(g["xyz1"], g["xyz2"])
    assert np.array_equal(d1.detach().cpu().numpy(), g["dist1"])
    assert np.array_equal(d2.detach().cpu().numpy(), g["dist2"])
    ga, gb = torch.autograd.grad([d1, d2], [a, b], [torch.from_numpy(g["graddist1"]).to(DEV),
                                                    torch.from_numpy(g["graddist2"]).to(DEV)])
    assert np.array_equal(ga.cpu().numpy(), g["gradxyz1"])      # gather backward == CPU loop order
    assert np.array_equal(gb.cpu().numpy(), g["gradxyz2"])


@pytest.mark.parametrize("B,n,m", [(4, 1024, 1024), (2, 1, 7), (1, 5000, 1031), (3, 2048, 2048),
                                   (1, 33, 4500), (32, 1024, 1024)])
def test_chamfer_matches_oracle(oracle_mod, B, n, m):
    from learning3d_b200 import _C
    rng = np.random.default_rng(B * 1000 + n + m)
    a_np = rng.standard_normal((B, n, 3)).astype(np.float32)
    b_np = rng.standard_normal((B, m, 3)).astype(np.float32)
    a, b = torch.from_numpy(a_np).to(DEV), torch.from_numpy(b_np).to(DEV)
    d1 = torch.empty(B, n, device=DEV); d2 = torch.empty(B, m, device=DEV)
    i1 = torch.empty(B, n, dtype=torch.int, device=DEV); i2 = torch.empty(B, m, dtype=torch.int, device=DEV)
    _C.check(_C.lib().l3d_chamfer_forward(_C.ptr(a), _C.ptr(b), B, n, m, _C.ptr(d1), _C.ptr(d2),
                                          _C.ptr(i1), _C.ptr(i2), _C.stream()))
    od1, od2, oi1, oi2 = oracle_mod.chamfer_forward(a_np, b_np)
    assert np.array_equal(i1.cpu().numpy(), oi1) and np.array_equal(i2.cpu().numpy(), oi2)
    assert np.array_equal(d1.cpu().numpy(), od1) and np.array_equal(d2.cpu().numpy(), od2)
    g1 = torch.randn(B, n, device=DEV); g2 = torch.randn(B, m, device=DEV)
    ga = torch.empty_like(a); gb = torch.empty_like(b)
    _C.check(_C.lib().l3d_chamfer_backward(_C.ptr(a), _C.ptr(b), B, n, m, _C.ptr(g1), _C.ptr(g2),
                                           _C.ptr(i1), _C.ptr(i2), _C.ptr(ga), _C.ptr(gb), _C.stream()))
    oa, ob = oracle_mod.chamfer_backward(a_np, b_np, g1.cpu().numpy(), g2.cpu().numpy(), oi1, oi2)
    assert np.array_equal(ga.cpu().numpy(), oa) and np.array_equal(gb.cpu().numpy(), ob)


def test_chamfer_ties_lowest_index(oracle_mod):
    a_np = np.zeros((1, 40, 3), np.float32)
    b_np = np.zeros((1, 50, 3), np.float32)          # every distance ties at 0
    _, _, d1, d2 = _fwd(a_np, b_np)
    from learning3d_b200 import _C  # noqa: F401
    od1, od2, oi1, oi2 = oracle_mod.chamfer_forward(a_np, b_np)
    assert (oi1 == 0).all() and (oi2 == 0).all()
    assert np.array_equal(d1.detach().cpu().numpy(), od1)


@pytest.mark.parametrize("tag", ["c1", "ragged"])
def test_chamfer_loss_module(oracle_mod, golden_dir, tag):
    """ChamferDistanceLoss (fused loss + fused backward) vs the reference's loss value and autograd
    gradients; tolerance 1e-5 (fp32 mean/sqrt chain, BASELINE.json north_star)."""
    from learning3d_b200.losses import ChamferDistanceLoss
    g = np.load(f"{golden_dir}/chamfer_{tag}.npz")
    a = torch.from_numpy(g["xyz1"]).to(DEV).requires_grad_(True)
    b = torch.from_numpy(g["xyz2"]).to(DEV).requires_grad_(True)
    crit = ChamferDistanceLoss()
    for _ in range(3):            # repeated calls: the self-resetting workspace must stay valid
        a.grad = b.grad = None
        loss = crit(a, b)
        (loss * 3.0).backward()   # non-unit upstream gradient
    assert abs(loss.item() - float(g["loss"])) <= 1e-5 * abs(float(g["loss"]))
    np.testing.assert_allclose(a.grad.cpu().numpy() / 3.0, g["loss_grad1"], rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(b.grad.cpu().numpy() / 3.0, g["loss_grad2"], rtol=1e-5, atol=1e-9)
    assert abs(loss.item() - oracle_mod.chamfer_loss(g["xyz1"], g["xyz2"])) < 1e-6


def test_chamfer_loss_deterministic_and_nan_on_shared_points():
    from learning3d_b200.losses import chamfer_distance
    torch.manual_seed(0)
    a = torch.rand(8, 1024, 3, device=DEV, requires_grad=True)
    b = torch.rand(8, 1024, 3, device=DEV, requires_grad=True)
    outs = []
    for _ in range(3):
        a.grad = b.grad = None
        l = chamfer_distance(a, b); l.backward()
        outs.append((l.item(), a.grad.clone(), b.grad.clone()))
    assert outs[0][0] == outs[1][0] == outs[2][0]
    assert torch.equal(outs[0][1], outs[2][1]) and torch.equal(outs[0][2], outs[2][2])
    c = a.detach().clone().requires_grad_(True)
    l = chamfer_distance(c, a.detach()); l.backward()
    assert not torch.isfinite(c.grad).all()      # sqrt(0) gradient, as in the reference


def test_chamfer_vs_reference_cuda_kernels(oracle_mod, golden_dir):
    """The reference's own CUDA kernels (recorded on a B200 by tests/golden/make_golden_gpu.py, a seeded
    sample of rows).  They are built with nvcc's default fma contraction, so distances may differ in the last ulp
    from the reference's CPU path that we reproduce; arg-mins must agree except at such near-ties."""
    from oracle import seeded
    g = np.load(f"{golden_dir}/ref_gpu.npz")
    rng = np.random.default_rng(3)
    a, b = rng.random((4, 1024, 3), dtype=np.float32), rng.random((4, 1024, 3), dtype=np.float32)
    rows = seeded.sample_index(1024, 256, "cd_rows")
    _, _, m1, m2 = _fwd(a, b)
    np.testing.assert_allclose(m1.detach().cpu().numpy()[:, rows], g["cd_dist1"], rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(m2.detach().cpu().numpy()[:, rows], g["cd_dist2"], rtol=1e-5, atol=1e-9)
    od1, od2, oi1, oi2 = oracle_mod.chamfer_forward(a, b)
    agree = (g["cd_idx1"] == oi1[:, rows]).mean()
    print("arg-min agreement with the reference CUDA kernel: %.6f" % agree)
    assert agree > 0.999