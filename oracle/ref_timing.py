"""TEST INFRASTRUCTURE ONLY — times of the reference's own CUDA kernels (oracle/_ref/*.so, built by
oracle/build_ref.py) at the shapes tests/test_gpu_vs_reference_kernels.py times ours.  GPU only."""
import ctypes

import torch

import oracle
from oracle import emd as oemd
from oracle import group as og

DEV = "cuda:0"


def available():
    """True when the reference's Chamfer, pointnet2 and EMD kernels have been built under oracle/_ref/."""
    return bool(og.ref_pn2() and oracle.ref_cd() and oemd.ref_emd())


def time_us(fn, iters=50, warm=5):
    """Microseconds per call: CUDA events around `iters` calls after `warm` untimed ones."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3


def reference_kernel_times():
    """{row name: microseconds per call} for the reference's kernels on the current GPU."""
    ref, cd, remd = og.ref_pn2(), oracle.ref_cd(), oemd.ref_emd()
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rows = {}
    torch.manual_seed(0)
    B, N, S = 16, 2048, 1024
    pc = (torch.rand(B, N, 3, device=DEV) * 4 - 2).contiguous()
    temp = torch.full((B, N), 1e10, device=DEV); fi = torch.empty((B, S), dtype=torch.int32, device=DEV)

    def ref_fps():
        temp.fill_(1e10)
        ref.ref_fps(B, N, S, P(pc), P(temp), P(fi), s)
    rows["FPS B16 2048->1024"] = time_us(ref_fps, 10, 2)
    new_xyz = pc[:, :S].contiguous()
    bi = torch.zeros((B, S, 16), dtype=torch.int32, device=DEV)
    rows["ball_query B16 N2048 S1024 ns16"] = time_us(
        lambda: ref.ref_ball_query(B, N, S, ctypes.c_float(0.5), 16, P(new_xyz), P(pc), P(bi), s))
    p1 = torch.rand(16, 256, 3, device=DEV); p2 = torch.rand(16, 256, 3, device=DEV)
    d2 = torch.empty(16, 256, 64, device=DEV); ki = torch.zeros(16, 256, 64, dtype=torch.int32, device=DEV)
    rows["knn B16 256x256 k64"] = time_us(lambda: ref.ref_knn(16, 256, 256, 64, P(p1), P(p2), P(d2), P(ki), s))
    feat = torch.rand(16, 128, 256, device=DEV); gout = torch.empty(16, 128, 256, 64, device=DEV)
    rows["group_points B16 C128 256x64"] = time_us(
        lambda: ref.ref_group_points(16, 128, 256, 256, 64, P(feat), P(ki), P(gout), s))
    q = torch.rand(16, 2048, 3, device=DEV); kn = torch.rand(16, 1024, 3, device=DEV)
    d3 = torch.empty(16, 2048, 3, device=DEV); i3 = torch.empty(16, 2048, 3, dtype=torch.int32, device=DEV)
    rows["three_nn B16 2048<-1024"] = time_us(lambda: ref.ref_three_nn(16, 2048, 1024, P(q), P(kn), P(d3), P(i3), s))
    for Bc in (4, 32):
        a = torch.rand(Bc, 1024, 3, device=DEV); b = torch.rand(Bc, 1024, 3, device=DEV)
        c1 = torch.zeros(Bc, 1024, device=DEV); c2 = torch.zeros(Bc, 1024, device=DEV)
        j1 = torch.zeros(Bc, 1024, dtype=torch.int, device=DEV); j2 = torch.zeros(Bc, 1024, dtype=torch.int, device=DEV)
        ga = torch.zeros_like(a); gb = torch.zeros_like(b); g1 = torch.rand(Bc, 1024, device=DEV); g2 = torch.rand(Bc, 1024, device=DEV)
        rows["chamfer forward B%d N1024" % Bc] = time_us(lambda: cd.forward_cuda(a, b, c1, c2, j1, j2))
        rows["chamfer backward B%d N1024" % Bc] = time_us(lambda: cd.backward_cuda(a, b, ga, gb, g1, g2, j1, j2))
    Be, ne = 8, 1024
    a = torch.rand(Be, ne, 3, device=DEV); b = torch.rand(Be, ne, 3, device=DEV)
    rm = torch.zeros(Be, ne, ne, device=DEV); rt = torch.zeros(Be, 4 * ne, device=DEV); rc = torch.zeros(Be, device=DEV)
    rows["EMD forward B8 N1024 (approxmatch+matchcost)"] = time_us(
        lambda: remd.ref_emd_forward(Be, ne, ne, P(a), P(b), P(rm), P(rt), P(rc)), 5, 1)
    g1 = torch.empty_like(a); g2 = torch.empty_like(b)
    rows["EMD backward B8 N1024"] = time_us(lambda: remd.ref_emd_backward(Be, ne, ne, P(a), P(b), P(rm), P(g1), P(g2)), 5, 1)
    return rows
