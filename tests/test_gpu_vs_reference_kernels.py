"""GPU: our kernels timed against the REFERENCE'S OWN CUDA kernels at the same shapes, and against the reference's
torch op sequences, on the same GPU.  The reference's kernels are timed in the same run where oracle/build_ref.py has
built them (oracle/_ref/); elsewhere their times on a B200 recorded by tests/golden/make_golden_gpu.py in
tests/golden/ref_kernel_times.json (with the card and its power limit) stand in.  CUDA-event timing after warm-up;
results must match (exactness is asserted elsewhere) and our kernel must not be slower.  The table is printed."""
import ctypes
import json

import pytest
import torch

from oracle import ref_timing
from oracle.ref_timing import time_us as _time

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def test_against_reference_cuda_kernels(golden_dir):
    if ref_timing.available():
        ref_us, source = ref_timing.reference_kernel_times(), "timed in this run"
    else:
        with open(f"{golden_dir}/ref_kernel_times.json") as f:
            rec = json.load(f)
        ref_us, source = rec["reference_us"], "recorded on %s" % rec["device"]
    print("reference kernel times:", source)
    from learning3d_b200 import _C
    from learning3d_b200.utils.lib import pointnet2_utils as pu
    lib = _C.lib()
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rows = []
    torch.manual_seed(0)

    # FlowNet3D sa1 (C4): FPS 2048 -> 1024, ball query r=.5 ns=16, grouping; fe_layer kNN k=64
    B, N, S = 16, 2048, 1024
    pc = (torch.rand(B, N, 3, device=DEV) * 4 - 2).contiguous()
    rows.append(("FPS B16 2048->1024", ref_us["FPS B16 2048->1024"], _time(lambda: pu.furthest_point_sample(pc, S), 10, 2)))
    new_xyz = pc[:, :S].contiguous()
    bi = torch.zeros((B, S, 16), dtype=torch.int32, device=DEV)
    rows.append(("ball_query B16 N2048 S1024 ns16", ref_us["ball_query B16 N2048 S1024 ns16"],
                 _time(lambda: lib.l3d_pn2_ball_query(B, N, S, 0.5, 16, _C.ptr(new_xyz), _C.ptr(pc), _C.ptr(bi), s))))
    p1 = torch.rand(16, 256, 3, device=DEV); p2 = torch.rand(16, 256, 3, device=DEV)
    d2 = torch.empty(16, 256, 64, device=DEV); ki = torch.empty(16, 256, 64, dtype=torch.int32, device=DEV)
    rows.append(("knn B16 256x256 k64", ref_us["knn B16 256x256 k64"],
                 _time(lambda: lib.l3d_pn2_knn(16, 256, 256, 64, _C.ptr(p1), _C.ptr(p2), _C.ptr(d2), _C.ptr(ki), s))))
    feat = torch.rand(16, 128, 256, device=DEV); out = torch.empty(16, 128, 256, 64, device=DEV)
    rows.append(("group_points B16 C128 256x64", ref_us["group_points B16 C128 256x64"],
                 _time(lambda: lib.l3d_pn2_group_points(16, 128, 256, 256, 64, _C.ptr(feat), _C.ptr(ki), _C.ptr(out), s))))
    q = torch.rand(16, 2048, 3, device=DEV); kn = torch.rand(16, 1024, 3, device=DEV)
    d3 = torch.empty(16, 2048, 3, device=DEV); i3 = torch.empty(16, 2048, 3, dtype=torch.int32, device=DEV)
    rows.append(("three_nn B16 2048<-1024", ref_us["three_nn B16 2048<-1024"],
                 _time(lambda: lib.l3d_pn2_three_nn(16, 2048, 1024, _C.ptr(q), _C.ptr(kn), _C.ptr(d3), _C.ptr(i3), s))))

    # Chamfer (C1 and B=32): the reference's CUDA extension kernels
    for Bc in (4, 32):
        a = torch.rand(Bc, 1024, 3, device=DEV); b = torch.rand(Bc, 1024, 3, device=DEV)
        c1 = torch.zeros(Bc, 1024, device=DEV); c2 = torch.zeros(Bc, 1024, device=DEV)
        j1 = torch.zeros(Bc, 1024, dtype=torch.int, device=DEV); j2 = torch.zeros(Bc, 1024, dtype=torch.int, device=DEV)
        ga = torch.zeros_like(a); gb = torch.zeros_like(b); g1 = torch.rand(Bc, 1024, device=DEV); g2 = torch.rand(Bc, 1024, device=DEV)
        rows.append(("chamfer forward B%d N1024" % Bc, ref_us["chamfer forward B%d N1024" % Bc],
                     _time(lambda: lib.l3d_chamfer_forward(_C.ptr(a), _C.ptr(b), Bc, 1024, 1024, _C.ptr(c1), _C.ptr(c2),
                                                           _C.ptr(j1), _C.ptr(j2), s))))
        rows.append(("chamfer backward B%d N1024" % Bc, ref_us["chamfer backward B%d N1024" % Bc],
                     _time(lambda: lib.l3d_chamfer_backward(_C.ptr(a), _C.ptr(b), Bc, 1024, 1024, _C.ptr(g1), _C.ptr(g2),
                                                            _C.ptr(j1), _C.ptr(j2), _C.ptr(ga), _C.ptr(gb), s))))

    # EMD (C5): the reference's approxmatch + matchcost / matchcostgrad kernels
    Be, ne = 8, 1024
    a = torch.rand(Be, ne, 3, device=DEV); b = torch.rand(Be, ne, 3, device=DEV)
    m = torch.empty(Be, ne, ne, device=DEV); c = torch.empty(Be, device=DEV)
    ws = torch.empty(int(lib.l3d_emd_forward_ws_bytes(Be, ne, ne)), dtype=torch.uint8, device=DEV)
    rows.append(("EMD forward B8 N1024 (approxmatch+matchcost)", ref_us["EMD forward B8 N1024 (approxmatch+matchcost)"],
                 _time(lambda: lib.l3d_emd_forward(_C.ptr(a), _C.ptr(b), Be, ne, ne, _C.ptr(c), _C.ptr(m), _C.ptr(ws), s), 5, 1)))
    g1 = torch.empty_like(a); g2 = torch.empty_like(b)
    ws2 = torch.empty(int(lib.l3d_emd_backward_ws_bytes(Be, ne, ne)), dtype=torch.uint8, device=DEV)
    rows.append(("EMD backward B8 N1024", ref_us["EMD backward B8 N1024"],
                 _time(lambda: lib.l3d_emd_backward(_C.ptr(a), _C.ptr(b), _C.ptr(m), Be, ne, ne, _C.ptr(g1), _C.ptr(g2), _C.ptr(ws2), s), 5, 1)))

    # kNN graph (C2): the reference's torch op sequence on the same GPU
    from oracle import ref_torch
    from learning3d_b200.utils import knn
    x = torch.rand(32, 3, 1024, device=DEV)
    rows.append(("knn() C2 B32 N1024 k20 (ref = torch matmul+topk on GPU)", _time(lambda: ref_torch.knn(x, 20), 20, 3),
                 _time(lambda: knn(x, 20), 20, 3)))
    rows.append(("get_graph_feature C2 (ref = torch ops on GPU)", _time(lambda: ref_torch.get_graph_feature(x, 20), 20, 3),
                 _time(lambda: __import__("learning3d_b200").utils.get_graph_feature(x, 20), 20, 3)))

    # feature-space graphs (PRNet's dynamic DGCNN): same torch op sequence, C = 64 / 128
    for C in (64, 128):
        xf = torch.randn(32, C, 1024, device=DEV)
        rows.append(("knn() features B32 C%d N1024 k20 (ref = torch matmul+topk on GPU)" % C,
                     _time(lambda: ref_torch.knn(xf, 20), 10, 2), _time(lambda: knn(xf, 20), 10, 2)))
    # DCP SVD head front half (svd.py:23-28): the reference's three torch ops vs the fused tcgen05 kernel
    import math
    from learning3d_b200.utils.svd import soft_correspondence
    es = torch.randn(32, 512, 1024, device=DEV); et = torch.randn(32, 512, 1024, device=DEV)
    tg = torch.rand(32, 3, 1024, device=DEV)

    def ref_front():
        sc = torch.matmul(es.transpose(2, 1).contiguous(), et) / math.sqrt(512)
        sc = torch.softmax(sc, dim=2)
        return torch.matmul(tg, sc.transpose(2, 1).contiguous())
    rows.append(("SVDHead front C3 B32 d512 N1024 (ref = torch matmul+softmax+matmul on GPU)",
                 _time(ref_front, 10, 2), _time(lambda: soft_correspondence(es, et, tg), 10, 2)))

    table = [{"op": n, "reference_us": round(r, 2), "ours_us": round(o, 2), "speedup": round(r / o, 2)} for n, r, o in rows]
    for t in table:
        print(json.dumps(t))
    slower = [t for t in table if t["speedup"] < 0.9]
    assert not slower, "slower than the reference's own kernel: %s" % slower
