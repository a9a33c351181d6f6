"""GPU parity: EMD (approxmatch/matchcost/grads) and the SVD-head tail against the oracle; tolerance 1e-5
relative on cost / R / t as BASELINE.json's north_star states (match entries: absolute 1e-5 of unit mass)."""
import numpy as np
import pytest
import torch

from oracle import emd as oe

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _emd(a_np, b_np):
    from learning3d_b200.losses.cuda.emd_torch.pkg.layer import EMDFunction
    a = T(a_np).requires_grad_(True)
    b = T(b_np).requires_grad_(True)
    cost = EMDFunction.apply(a, b)
    return a, b, cost


@pytest.mark.parametrize("B,n,m", [(8, 1024, 1024), (2, 256, 256), (3, 100, 333), (1, 512, 128), (1, 1500, 1500)])
def test_emd_forward_backward_vs_oracle(B, n, m):
    rng = np.random.default_rng(n + m)
    a_np = rng.random((B, n, 3), dtype=np.float32)
    b_np = rng.random((B, m, 3), dtype=np.float32)
    a, b, cost = _emd(a_np, b_np)
    ocost, omatch = oe.emd_forward(a_np, b_np)
    np.testing.assert_allclose(cost.detach().cpu().numpy(), ocost, rtol=1e-5)
    # the saved matching itself
    from learning3d_b200 import _C
    lib = _C.lib()
    match = torch.empty((B, n, m), device=DEV)
    c2 = torch.empty((B,), device=DEV)
    ws = torch.empty(int(lib.l3d_emd_forward_ws_bytes(B, n, m)), dtype=torch.uint8, device=DEV)
    _C.check(lib.l3d_emd_forward(_C.ptr(a.detach()), _C.ptr(b.detach()), B, n, m, _C.ptr(c2), _C.ptr(match),
                                 _C.ptr(ws), _C.stream()))
    # The soft matching amplifies last-bit differences of exp() where two candidates nearly tie
    # (__expf/ex2.approx on the GPU, libm expf in the oracle): single entries move by up to ~2e-3 of a
    # unit-mass row while row/column masses and the cost agree to 1e-6 (profiles/diag_emd.py).
    mm = match.cpu().numpy()
    np.testing.assert_allclose(mm, omatch, atol=5e-3)
    np.testing.assert_allclose(mm.reshape(B, m, n).sum(1), omatch.reshape(B, m, n).sum(1), atol=2e-5)
    assert torch.equal(c2, cost.detach())                       # deterministic
    # gradient kernels on the SAME matching: 1e-5
    g1 = torch.empty_like(a); g2 = torch.empty_like(b)
    ws2 = torch.empty(int(lib.l3d_emd_backward_ws_bytes(B, n, m)), dtype=torch.uint8, device=DEV)
    om_d = T(omatch)
    _C.check(lib.l3d_emd_backward(_C.ptr(a.detach()), _C.ptr(b.detach()), _C.ptr(om_d), B, n, m, _C.ptr(g1),
                                  _C.ptr(g2), _C.ptr(ws2), _C.stream()))
    og1, og2 = oe.grads(a_np, b_np, omatch)
    np.testing.assert_allclose(g1.cpu().numpy(), og1, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(g2.cpu().numpy(), og2, rtol=1e-5, atol=1e-5)
    # autograd path (own matching; grad_output ignored exactly like the reference)
    (cost * 7.0).sum().backward()
    np.testing.assert_allclose(a.grad.cpu().numpy(), og1, atol=3e-3)
    np.testing.assert_allclose(b.grad.cpu().numpy(), og2, atol=3e-3)


def test_emd_loss_module_intended_semantics():
    from learning3d_b200.losses import EMDLoss
    rng = np.random.default_rng(3)
    a_np = rng.random((8, 1024, 3), dtype=np.float32)        # BASELINE config C5 shape
    b_np = rng.random((8, 1024, 3), dtype=np.float32)
    a = T(a_np).requires_grad_(True)
    loss = EMDLoss()(a, T(b_np))
    ocost, omatch = oe.emd_forward(a_np, b_np)
    want = ocost.mean() / 1024
    assert abs(loss.item() - want) <= 1e-5 * abs(want)
    loss.backward()
    og1, _ = oe.grads(a_np, b_np, omatch)
    np.testing.assert_allclose(a.grad.cpu().numpy(), og1 / (8 * 1024), atol=3e-3 / (8 * 1024))


def test_emd_input_checks():
    from learning3d_b200.losses.cuda.emd_torch.pkg.layer import EMDLoss
    with pytest.raises(RuntimeError):
        EMDLoss()(torch.rand(1, 8, 3), torch.rand(1, 8, 3))            # CPU tensors (CHECK_CUDA)
    x = torch.rand(1, 3, 8, device=DEV).transpose(1, 2)
    with pytest.raises(RuntimeError):
        EMDLoss()(x, x)                                                # non-contiguous (CHECK_CONTIGUOUS)


def test_svd_head_golden(golden_dir):
    from learning3d_b200.utils import SVDHead
    g = np.load(f"{golden_dir}/svd_head.npz")
    head = SVDHead(64).to(DEV)
    assert "reflect" in head.state_dict()
    with torch.no_grad():
        R, t = head(T(g["src_emb"]), T(g["tgt_emb"]), T(g["src"]), T(g["tgt"]))
    np.testing.assert_allclose(R.cpu().numpy(), g["R"], atol=1e-5)     # includes two det<0 items
    np.testing.assert_allclose(t.cpu().numpy(), g["t"], atol=1e-5)


def test_svd_tail_vs_oracle_and_kabsch_entry():
    from learning3d_b200 import _C
    rng = np.random.default_rng(8)
    B, N = 32, 1024                                           # BASELINE config C3 shape
    src = rng.standard_normal((B, 3, N)).astype(np.float32)
    A = rng.standard_normal((B, 3, 3)).astype(np.float32)     # general linear maps: both det signs
    corr = (A @ src + rng.standard_normal((B, 3, 1)).astype(np.float32) +
            0.01 * rng.standard_normal((B, 3, N)).astype(np.float32)).astype(np.float32)
    R = torch.empty((B, 3, 3), device=DEV); t = torch.empty((B, 3), device=DEV)
    sd, cd_ = T(src), T(corr)      # keep alive: a freed temporary's block is handed to the next T()
    _C.check(_C.lib().l3d_svd_head_tail(_C.ptr(sd), _C.ptr(cd_), B, N, _C.ptr(R), _C.ptr(t), _C.stream()))
    torch.cuda.synchronize()
    oR, ot = oe.svd_head_tail(src, corr)
    np.testing.assert_allclose(R.cpu().numpy(), oR, atol=1e-5)
    np.testing.assert_allclose(t.cpu().numpy(), ot, atol=2e-5)
    Rn = R.cpu().numpy()
    np.testing.assert_allclose(Rn @ Rn.transpose(0, 2, 1), np.tile(np.eye(3), (B, 1, 1)), atol=1e-6)
    assert np.allclose(np.linalg.det(Rn), 1.0, atol=1e-5)
    # the H-level entry point gives the same rotation
    mu_s = src.mean(2); mu_c = corr.mean(2)
    H = ((src - mu_s[..., None]) @ (corr - mu_c[..., None]).transpose(0, 2, 1)).astype(np.float32)
    R2 = torch.empty((B, 3, 3), device=DEV); t2 = torch.empty((B, 3), device=DEV)
    Hd, ms, mc = T(H), T(mu_s), T(mu_c)
    _C.check(_C.lib().l3d_kabsch3x3_batched(_C.ptr(Hd), _C.ptr(ms), _C.ptr(mc), B, _C.ptr(R2), _C.ptr(t2), _C.stream()))
    torch.cuda.synchronize()
    np.testing.assert_allclose(R2.cpu().numpy(), oR, atol=1e-5)


def _torch_tail(src, corr):
    """utils/svd.py:29-58 in differentiable torch (fp64): the formulation autograd differentiates in the
    reference's training scripts."""
    B = src.shape[0]
    sc = src - src.mean(dim=2, keepdim=True)
    cc = corr - corr.mean(dim=2, keepdim=True)
    H = torch.matmul(sc, cc.transpose(2, 1))
    Rs = []
    reflect = torch.eye(3, dtype=src.dtype, device=src.device); reflect[2, 2] = -1
    for i in range(B):
        u, s, vh = torch.linalg.svd(H[i])
        v = vh.transpose(0, 1)
        r = v @ u.transpose(0, 1)
        if torch.det(r) < 0:
            r = (v @ reflect) @ u.transpose(0, 1)
        Rs.append(r)
    R = torch.stack(Rs)
    t = torch.matmul(-R, src.mean(dim=2, keepdim=True)) + corr.mean(dim=2, keepdim=True)
    return R, t.view(B, 3)


def test_svd_tail_backward_matches_autograd():
    from learning3d_b200.utils.svd import svd_head_tail
    rng = np.random.default_rng(21)
    B, N = 6, 300
    src = rng.standard_normal((B, 3, N)).astype(np.float32)
    A = rng.standard_normal((B, 3, 3)).astype(np.float32)
    A[3:] *= np.sign(np.linalg.det(A[3:]))[:, None, None] * -1      # items 3..5: reflections -> det fix branch
    corr = (A @ src + 0.05 * rng.standard_normal((B, 3, N)).astype(np.float32)).astype(np.float32)
    s = T(src).requires_grad_(True); c = T(corr).requires_grad_(True)
    R, t = svd_head_tail(s, c)
    wR = torch.randn_like(R); wt = torch.randn_like(t)
    ((R * wR).sum() + (t * wt).sum()).backward()
    # reference gradients on the CPU (fp64 LAPACK): torch.linalg.svd on the GPU drags cuSOLVER/MAGMA
    # initialisation (minutes on a cold box) into the suite
    s64 = torch.from_numpy(src).double().requires_grad_(True); c64 = torch.from_numpy(corr).double().requires_grad_(True)
    R64, t64 = _torch_tail(s64, c64)
    ((R64 * wR.double().cpu()).sum() + (t64 * wt.double().cpu()).sum()).backward()
    np.testing.assert_allclose(R.detach().cpu().numpy(), R64.detach().cpu().numpy(), atol=1e-5)
    scale = s64.grad.abs().max().item()
    np.testing.assert_allclose(s.grad.cpu().numpy(), s64.grad.cpu().numpy(), atol=2e-5 * scale + 1e-7)
    np.testing.assert_allclose(c.grad.cpu().numpy(), c64.grad.cpu().numpy(), atol=2e-5 * scale + 1e-7)
    assert (np.linalg.det(A[3:]) < 0).all()


def test_svd_head_module_is_trainable(golden_dir):
    from learning3d_b200.utils import SVDHead
    g = np.load(f"{golden_dir}/svd_head.npz")
    head = SVDHead(64).to(DEV)
    e1 = T(g["src_emb"]).requires_grad_(True); e2 = T(g["tgt_emb"]).requires_grad_(True)
    R, t = head(e1, e2, T(g["src"]), T(g["tgt"]))
    np.testing.assert_allclose(R.detach().cpu().numpy(), g["R"], atol=1e-5)
    (R.sum() + t.sum()).backward()
    assert torch.isfinite(e1.grad).all() and e1.grad.abs().sum() > 0


@pytest.mark.parametrize("B,n,m", [(8, 1024, 1024), (2, 300, 700)])
def test_emd_against_reference_cuda_kernels(B, n, m, golden_dir):
    """The reference's OWN approxmatch / matchcost / matchcostgrad kernels (emd.cuh), recorded on a B200 by
    tests/golden/make_golden_gpu.py (seeded samples of the large outputs): pins the EMD path against the
    reference.  cost 1e-5 relative; row/column masses 2e-5; single match entries within the soft-assignment jitter."""
    from learning3d_b200 import _C
    from oracle import seeded
    g = np.load(f"{golden_dir}/ref_gpu.npz")
    tag = "emd_%d_%d_%d_" % (B, n, m)
    cols, rows = seeded.sample_index(n, 64, tag + "cols"), seeded.sample_index(m, 64, tag + "rows")
    lib = _C.lib()
    rng = np.random.default_rng(B + n)
    a = T(rng.random((B, n, 3), dtype=np.float32)); b = T(rng.random((B, m, 3), dtype=np.float32))
    cost = torch.empty((B,), device=DEV); match = torch.empty((B, n, m), device=DEV)
    ws = torch.empty(int(lib.l3d_emd_forward_ws_bytes(B, n, m)), dtype=torch.uint8, device=DEV)
    _C.check(lib.l3d_emd_forward(_C.ptr(a), _C.ptr(b), B, n, m, _C.ptr(cost), _C.ptr(match), _C.ptr(ws), _C.stream()))
    torch.cuda.synchronize()
    np.testing.assert_allclose(cost.cpu().numpy(), g[tag + "cost"], rtol=1e-5)
    mm = match.cpu().numpy().reshape(B, m, n)
    np.testing.assert_allclose(mm.sum(1)[:, cols], g[tag + "colsum"], atol=2e-5)
    np.testing.assert_allclose(mm.sum(2)[:, rows], g[tag + "rowsum"], atol=1e-3)
    np.testing.assert_allclose(mm.reshape(-1)[seeded.sample_index(mm.size, 1024, tag + "flat")], g[tag + "entries"], atol=5e-3)
    # gradients on the same fixed matching the reference's backward was given
    fixed = T(np.random.default_rng(B + n + 1).random((B, m, n), dtype=np.float32) * np.float32(2.0 / (n + m)))
    g1 = torch.empty_like(a); g2 = torch.empty_like(b)
    ws2 = torch.empty(int(lib.l3d_emd_backward_ws_bytes(B, n, m)), dtype=torch.uint8, device=DEV)
    _C.check(lib.l3d_emd_backward(_C.ptr(a), _C.ptr(b), _C.ptr(fixed), B, n, m, _C.ptr(g1), _C.ptr(g2), _C.ptr(ws2), _C.stream()))
    torch.cuda.synchronize()
    np.testing.assert_allclose(g1.cpu().numpy()[:, cols], g[tag + "grad1"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(g2.cpu().numpy()[:, rows], g[tag + "grad2"], rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("B,n,m", [(8, 1024, 1024), (3, 300, 700), (20, 512, 256), (1, 50, 33)])
def test_emd_single_launch_paths_match_multilaunch(B, n, m):
    """The single-launch forwards — cooperative persistent (default) and cluster-per-item with 16 / 8 CTAs (hardware
    cluster barriers, clouds resident in shared memory) — against the 21-launch path: same arithmetic per pair, only
    the partial-sum order inside a row differs."""
    from learning3d_b200 import _C
    lib = _C.lib()
    rng = np.random.default_rng(B * 7 + n)
    a = T(rng.random((B, n, 3), dtype=np.float32)); b = T(rng.random((B, m, 3), dtype=np.float32))
    outs = []
    for force in (0, 1, 3, 4):
        lib.l3d_debug_emd_force_multilaunch(force)
        try:
            cost = torch.empty((B,), device=DEV); match = torch.empty((B, n, m), device=DEV)
            ws = torch.empty(int(lib.l3d_emd_forward_ws_bytes(B, n, m)), dtype=torch.uint8, device=DEV)
            n0 = _C.launch_count()
            _C.check(lib.l3d_emd_forward(_C.ptr(a), _C.ptr(b), B, n, m, _C.ptr(cost), _C.ptr(match), _C.ptr(ws), _C.stream()))
            torch.cuda.synchronize()
            outs.append((cost.cpu().numpy(), match.cpu().numpy(), _C.launch_count() - n0))
        finally:
            lib.l3d_debug_emd_force_multilaunch(0)
    assert outs[0][2] == 2 and outs[1][2] == 22            # sweeps + final  vs  fill + 20 sweeps + final
    assert outs[2][2] == 2 and outs[3][2] == 2              # cluster kernels: sweeps + final
    for o in (outs[0], outs[2], outs[3]):
        np.testing.assert_allclose(o[0], outs[1][0], rtol=2e-6)
        np.testing.assert_allclose(o[1].sum(1), outs[1][1].sum(1), atol=2e-5)
        np.testing.assert_allclose(o[1], outs[1][1], atol=5e-3)
