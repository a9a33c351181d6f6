"""Generate tests/golden/ref_gpu.npz and ref_kernel_times.json: what the reference's OWN CUDA kernels and models
return, and how long its kernels take, on a B200.

Needs a GPU and what oracle/build_ref.py makes from the reference's sources under oracle/_ref/ (cd_ref.so: Chamfer;
libpn2_ref.so: pointnet2 grouping; libemd_ref.so: approximate EMD; learning3d/: its Python package):
    python tests/golden/make_golden_gpu.py [OUT_DIR]
Inputs are drawn from seeds the GPU tests draw again, and the models get the weights of
oracle.seeded.seeded_state_dict (the pretrained checkpoints are too large to keep).  Where an output is large, a
seeded sample of it is stored together with the sampled indices, so that the files stay small.
"""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import oracle  # noqa: E402
from oracle import emd as oemd  # noqa: E402
from oracle import group as og  # noqa: E402
from oracle import ref_pkg, ref_timing, seeded  # noqa: E402

DEV = "cuda:0"


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def P(t):
    return ctypes.c_void_p(t.data_ptr())


def chamfer_inputs():
    rng = np.random.default_rng(3)
    return rng.random((4, 1024, 3), dtype=np.float32), rng.random((4, 1024, 3), dtype=np.float32)


def emd_inputs(B, n, m):
    """The clouds of test_emd_against_reference_cuda_kernels and a fixed matching [B, m, n] for the backward."""
    rng = np.random.default_rng(B + n)
    a, b = rng.random((B, n, 3), dtype=np.float32), rng.random((B, m, 3), dtype=np.float32)
    match = (np.random.default_rng(B + n + 1).random((B, m, n), dtype=np.float32) * np.float32(2.0 / (n + m)))
    return a, b, match


EMD_CASES = [(8, 1024, 1024), (2, 300, 700)]


def pn2_inputs():
    rng = np.random.default_rng(12)
    B, N, S = 4, 2048, 512
    xyz = (rng.random((B, N, 3), dtype=np.float32) * 2 - 1).astype(np.float32)
    feats = rng.standard_normal((B, 10, N)).astype(np.float32)
    gi = rng.integers(0, N, (B, 64, 8)).astype(np.int32)
    w = rng.random((B, S, 3)).astype(np.float32)
    ti = rng.integers(0, N, (B, S, 3)).astype(np.int32)
    return xyz, np.ascontiguousarray(xyz[:, :S]), feats, gi, w, ti


def gen_chamfer(out):
    cd = oracle.ref_cd()
    a, b = chamfer_inputs()
    B, n = a.shape[:2]
    d1, d2 = torch.zeros(B, n, device=DEV), torch.zeros(B, n, device=DEV)
    i1, i2 = torch.zeros(B, n, dtype=torch.int, device=DEV), torch.zeros(B, n, dtype=torch.int, device=DEV)
    cd.forward_cuda(T(a), T(b), d1, d2, i1, i2)
    torch.cuda.synchronize()
    rows = seeded.sample_index(n, 256, "cd_rows")
    out.update(cd_dist1=d1.cpu().numpy()[:, rows], cd_dist2=d2.cpu().numpy()[:, rows], cd_idx1=i1.cpu().numpy()[:, rows])


def gen_emd(out):
    ref = oemd.ref_emd()
    for B, n, m in EMD_CASES:
        a, b, fixed = emd_inputs(B, n, m)
        tag = "emd_%d_%d_%d_" % (B, n, m)
        ad, bd = T(a), T(b)
        match = torch.zeros((B, n, m), device=DEV)
        temp = torch.zeros((B, 2 * (n + m)), device=DEV)
        cost = torch.zeros((B,), device=DEV)
        ref.ref_emd_forward(B, n, m, P(ad), P(bd), P(match), P(temp), P(cost))
        torch.cuda.synchronize()
        rm = match.cpu().numpy().reshape(B, m, n)
        cols, rows = seeded.sample_index(n, 64, tag + "cols"), seeded.sample_index(m, 64, tag + "rows")
        flat = seeded.sample_index(rm.size, 1024, tag + "flat")
        g1, g2 = torch.zeros_like(ad), torch.zeros_like(bd)
        fd = T(fixed)
        ref.ref_emd_backward(B, n, m, P(ad), P(bd), P(fd), P(g1), P(g2))
        torch.cuda.synchronize()
        out.update({tag + "cost": cost.cpu().numpy(), tag + "colsum": rm.sum(1)[:, cols], tag + "rowsum": rm.sum(2)[:, rows],
                    tag + "entries": rm.reshape(-1)[flat],
                    tag + "grad1": g1.cpu().numpy()[:, cols], tag + "grad2": g2.cpu().numpy()[:, rows]})


def gen_pn2(out):
    ref = og.ref_pn2()
    xyz, new_xyz, feats, gi, w, ti = pn2_inputs()
    B, N, S = xyz.shape[0], xyz.shape[1], new_xyz.shape[1]
    xd, qd = T(xyz), T(new_xyz)
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    D = seeded.array_digest
    idx = torch.zeros((B, S, 16), dtype=torch.int32, device=DEV)
    ref.ref_ball_query(B, N, S, ctypes.c_float(0.2), 16, P(qd), P(xd), P(idx), s)
    for k in (8, 64):
        d2 = torch.empty((B, S, k), device=DEV); ik = torch.empty((B, S, k), dtype=torch.int32, device=DEV)
        ref.ref_knn(B, S, N, k, P(qd), P(xd), P(d2), P(ik), s)
        torch.cuda.synchronize()
        out["pn2_knn%d_dist2" % k], out["pn2_knn%d_idx" % k] = D(d2.cpu().numpy()), D(ik.cpu().numpy())
    d3 = torch.empty((B, S, 3), device=DEV); i3 = torch.empty((B, S, 3), dtype=torch.int32, device=DEV)
    ref.ref_three_nn(B, S, N, P(qd), P(xd), P(d3), P(i3), s)
    torch.cuda.synchronize()
    out.update(pn2_ball=D(idx.cpu().numpy()), pn2_three_nn_dist2=D(d3.cpu().numpy()), pn2_three_nn_idx=D(i3.cpu().numpy()))
    # FPS, including a duplicated cloud (tie rule of the shared-memory tree)
    for tag, cloud in (("", xyz), ("_dup", np.tile(xyz[:, :256], (1, 4, 1)))):
        n = cloud.shape[1]
        temp = torch.full((B, n), 1e10, device=DEV); fi = torch.empty((B, 300), dtype=torch.int32, device=DEV)
        cd_ = T(cloud)
        ref.ref_fps(B, n, 300, P(cd_), P(temp), P(fi), s)
        torch.cuda.synchronize()
        out.update({"pn2_fps%s_idx" % tag: fi.cpu().numpy(), "pn2_fps%s_temp" % tag: D(temp.cpu().numpy())})
    gout = torch.empty((B, 10, 64, 8), device=DEV)
    fd, gid = T(feats), T(gi)
    ref.ref_group_points(B, 10, N, 64, 8, P(fd), P(gid), P(gout), s)
    o3 = torch.empty((B, 10, S), device=DEV)
    tid, wd = T(ti), T(w)
    ref.ref_three_interpolate(B, 10, N, S, P(fd), P(tid), P(wd), P(o3), s)
    torch.cuda.synchronize()
    out.update(pn2_group=D(gout.cpu().numpy()), pn2_interp=D(o3.cpu().numpy()))


def sample(t, k, key):
    """The values of tensor t at seeded.sample_index(t.numel(), k, key)."""
    return t.detach().cpu().numpy().reshape(-1)[seeded.sample_index(t.numel(), k, key)]


def gen_models(out):
    """The reference's own models, unmodified, on this GPU in fp32 (TF32 off): C3 DCP, C4 FlowNet3D on its own
    pointnet2 kernels, and RPMNet's matching tail."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    ref = ref_pkg.import_reference()
    # C3: DCP (DGCNN-512 + Transformer + SVDHead), B=32, N=1024, eval, cycle=True
    template, source = seeded.dcp_inputs()
    net = ref.models.DCP(feature_model=ref.models.DGCNN(emb_dims=512), cycle=True)
    net.load_state_dict(seeded.seeded_state_dict(net, 3), strict=True)
    net = net.to(DEV).eval()
    template, source = template.to(DEV), source.to(DEV)
    with torch.no_grad():
        want = net(template, source)
        idx = ref.utils.knn(source.permute(0, 2, 1).contiguous(), 20)
    for k in ("est_R", "est_t", "est_R_", "est_t_", "est_T"):
        out["c3_" + k] = want[k].cpu().numpy()
    out["c3_ts"] = sample(want["transformed_source"], 2048, "c3_ts")
    out["c3_r"] = sample(want["r"], 2048, "c3_r")
    out["c3_r_absmax"] = want["r"].abs().max().cpu().numpy()
    # one byte per row of all 32 clouds: the check counts rows whose neighbour set differs
    out["c3_knn_digest"] = (seeded.row_digest(idx.cpu().numpy()) % 256).astype(np.uint8)
    # C4: FlowNet3D, B=16, N=2048, eval, grouping on the reference's own pointnet2 kernels
    net = ref.models.FlowNet3D()
    net.load_state_dict(seeded.seeded_state_dict(net, 4), strict=True)
    net = net.to(DEV).eval()
    pc1, pc2, f1, f2 = [x.to(DEV).contiguous() for x in seeded.flownet_inputs()]
    ref_pkg.set_pointnet2_backend("ref")
    pu = ref.utils.lib.pointnet2_utils
    with torch.no_grad():
        flow = net(pc1, pc2, f1, f2)
        x1 = pc1.permute(0, 2, 1).contiguous()
        x2 = pc2.permute(0, 2, 1).contiguous()
        fps = pu.furthest_point_sample(x1, 1024)
        new = pu.gather_operation(pc1, fps).permute(0, 2, 1).contiguous()
        ball = pu.ball_query(0.5, 16, x1, new)
        _, knn = pu.knn(64, new[:, :256].contiguous(), x2[:, :256].contiguous())
        d3, i3 = pu.three_nn(x1, new)
    torch.cuda.synchronize()
    out["c4_flow"] = sample(flow, 2048, "c4_flow")
    out["c4_flow_absmax"] = flow.abs().max().cpu().numpy()
    for name, t in (("fps", fps), ("ball", ball), ("knn", knn), ("three_nn_idx", i3), ("three_nn_dist2", d3)):
        out["c4_" + name] = seeded.array_digest(t.cpu().numpy())
    # RPMNet matching tail (models/rpmnet.py): match_features, sinkhorn with slack, compute_rigid_transform
    with torch.no_grad():
        d, lp, T = seeded.rpm_tail(ref.models.rpmnet, *[x.to(DEV) for x in seeded.rpm_inputs()])
    out["rpm_d"] = sample(d, 1024, "rpm_d")
    out["rpm_lp"] = sample(lp, 1024, "rpm_lp")
    out["rpm_T"] = T.cpu().numpy()


def gen_times():
    """Times of the reference's own kernels, with the card, its power limit and its top SM clock."""
    rows = ref_timing.reference_kernel_times()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    return {"device": smi or torch.cuda.get_device_name(0), "unit": "us per call, CUDA events after warm-up",
            "reference_us": {k: round(v, 2) for k, v in rows.items()}}


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else HERE
    assert oracle.ref_cd() and og.ref_pn2() and oemd.ref_emd(), "run oracle/build_ref.py first"
    out = {}
    gen_chamfer(out)
    gen_emd(out)
    gen_pn2(out)
    gen_models(out)
    # indices stored as the narrowest of int16 / int32 that holds them (digests keep their unsigned types)
    out = {k: (v.astype(np.int16 if v.max() < 32768 else np.int32) if v.dtype.kind == "i" else v) for k, v in out.items()}
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "ref_gpu.npz")
    np.savez_compressed(path, device=np.array(torch.cuda.get_device_name(0)), **out)
    print("wrote", path, os.path.getsize(path), "bytes")
    times = gen_times()
    path = os.path.join(out_dir, "ref_kernel_times.json")
    with open(path, "w") as f:
        json.dump(times, f, indent=1)
    print("wrote", path, json.dumps(times))


if __name__ == "__main__":
    main()
