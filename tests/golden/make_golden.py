"""Generate the golden fixtures in tests/golden/ by running the REAL reference.

Run in the build container only (needs /root/reference, which does not exist on the GPU box):
    python tests/golden/make_golden.py
The reference is imported unmodified through a symlink package (SURVEY.md App. B); `h5py` is
stubbed because utils/transformer.py:4 imports it.  Inputs are seeded; outputs are what the
reference's own CPU code returns.  The oracle (oracle/l3d_oracle.c) and the CUDA path are
both tested against these files.
"""
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"


def import_reference():
    tmp = tempfile.mkdtemp(prefix="l3dref_")
    os.symlink(REF, os.path.join(tmp, "learning3d"))
    sys.path.insert(0, tmp)
    sys.modules["h5py"] = types.ModuleType("h5py")
    import learning3d  # noqa: F401
    return tmp


def save(name, **arrays):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, {k: v.shape for k, v in arrays.items()})


def gen_knn():
    from learning3d.utils.model_common_utils import knn, get_graph_feature, knn_point, square_distance
    from learning3d.utils import pointconv_util as pcu
    torch.manual_seed(1234)
    # knn / get_graph_feature (utils/model_common_utils.py:3-9,132-155)
    for tag, (B, N, k) in {"a": (2, 256, 20), "b": (1, 300, 33), "c": (2, 128, 8)}.items():
        while True:
            x = torch.rand(B, 3, N)
            idx = knn(x, k)
            xx = (x ** 2).sum(1, keepdim=True)
            pd = -xx - (-2 * torch.matmul(x.transpose(2, 1).contiguous(), x)) - xx.transpose(2, 1).contiguous()
            top = torch.gather(pd, 2, idx)
            # reject draws with exact ties inside the top-(k+1): topk's tie order is unspecified
            top1 = pd.topk(k + 1, dim=-1)[0]
            if (top1[..., 1:] == top1[..., :-1]).any():
                continue
            break
        feat = get_graph_feature(x, k=k, device="cpu")
        save("knn_" + tag, x=x.numpy(), idx=idx.numpy(), pd=top.numpy(), feat=feat.numpy(),
             k=np.array(k))
    # knn_point (:84-100), square_distance (:19-38), pointconv knn_point (pointconv_util.py:107-118)
    data = torch.rand(2, 200, 3)
    query = torch.rand(2, 90, 3)
    val, idx = knn_point(12, data, query)
    sd = square_distance(query, data)
    pc_idx = pcu.knn_point(16, data, query)
    save("knn_point", data=data.numpy(), query=query.numpy(), val=val.numpy(), idx=idx.numpy(),
         sqdist=sd.numpy(), pc_idx=pc_idx.numpy())


def gen_chamfer():
    """Chamfer: the reference's JIT extension (losses/cuda/chamfer_distance) run on CPU
    (cd.forward / cd.backward == nnsearch) + the loss through losses/chamfer_distance.py with
    autograd gradients.  Config C1 shape and a ragged n != m case."""
    import learning3d.losses.cuda.chamfer_distance as ref_cd_pkg   # JIT-builds `cd`
    from learning3d.losses.chamfer_distance import chamfer_distance, chamfer
    torch.manual_seed(4321)
    for tag, (B, n, m) in {"c1": (4, 1024, 1024), "ragged": (3, 200, 333)}.items():
        a = torch.rand(B, n, 3, requires_grad=True)
        b = torch.rand(B, m, 3, requires_grad=True)
        d1, d2 = ref_cd_pkg.ChamferDistance()(a, b)
        idx1 = torch.zeros(B, n, dtype=torch.int); idx2 = torch.zeros(B, m, dtype=torch.int)
        dd1 = torch.zeros(B, n); dd2 = torch.zeros(B, m)
        ref_cd_pkg.chamfer_distance.cd.forward(a.detach(), b.detach(), dd1, dd2, idx1, idx2)
        assert torch.equal(dd1, d1) and torch.equal(dd2, d2)
        g1 = torch.randn(B, n); g2 = torch.randn(B, m)
        ga, gb = torch.autograd.grad([d1, d2], [a, b], [g1, g2])
        loss = chamfer_distance(a, b)                     # native path (ext is importable here)
        la, lb = torch.autograd.grad(loss, [a, b])
        loss_torch = chamfer(a, b)                        # the pure-torch fallback, same value
        save("chamfer_" + tag, xyz1=a.detach().numpy(), xyz2=b.detach().numpy(),
             dist1=d1.detach().numpy(), dist2=d2.detach().numpy(), idx1=idx1.numpy(), idx2=idx2.numpy(),
             graddist1=g1.numpy(), graddist2=g2.numpy(), gradxyz1=ga.numpy(), gradxyz2=gb.numpy(),
             loss=loss.detach().numpy(), loss_torch=loss_torch.detach().numpy(),
             loss_grad1=la.numpy(), loss_grad2=lb.numpy())


def gen_group():
    """Pure-torch grouping helpers on CPU: the three query_ball_point / farthest_point_sample variants,
    index_points, compute_density, and the sample_and_group compositions."""
    from learning3d.utils import model_common_utils as mcu
    from learning3d.utils import pointconv_util as pcu
    from learning3d.utils import ppfnet_util as ppu
    torch.manual_seed(99)
    xyz = torch.rand(2, 300, 3)
    new_xyz = xyz[:, ::3].contiguous()                       # queries are a subset (100 per item)
    normals = torch.nn.functional.normalize(torch.randn(2, 300, 3), dim=-1)
    feats = torch.randn(2, 300, 5)
    out = {"xyz": xyz, "new_xyz": new_xyz, "normals": normals, "feats": feats}
    idx, cnt = mcu.query_ball_point(0.25, 16, xyz, new_xyz, get_cnt=True)
    out["qbp_idx"], out["qbp_cnt"] = idx, cnt
    out["qbp_small_r"] = pcu.query_ball_point(0.05, 8, xyz, new_xyz)       # many rows with 1 hit
    itself = torch.arange(0, 300, 3)[None].repeat(2, 1)
    out["qbp_itself"] = ppu.query_ball_point(0.25, 16, xyz, new_xyz, itself)
    out["fps_first"] = mcu.farthest_point_sample(xyz, 64, start_with_first_point=True)
    out["fps_pointconv"] = pcu.farthest_point_sample(xyz, 50)
    torch.manual_seed(7)
    out["fps_random_seed7"] = mcu.farthest_point_sample(xyz, 40)
    torch.manual_seed(8)
    out["fps_ppf_seed8"] = ppu.farthest_point_sample(xyz, 40)
    out["index_points"] = mcu.index_points(feats, idx)
    out["density"] = pcu.compute_density(xyz, 0.1)
    nx, npts, gnorm, gidx = pcu.sample_and_group(32, 8, xyz, feats)
    out["pc_sg_new_xyz"], out["pc_sg_new_points"], out["pc_sg_idx"] = nx, npts, gidx
    torch.manual_seed(11)
    res, gxyz, fidx = ppu.sample_and_group_multi(20, 0.3, 12, xyz, normals, returnfps=True)
    out["ppf_xyz"], out["ppf_dxyz"], out["ppf_ppf"], out["ppf_fps"] = res["xyz"], res["dxyz"], res["ppf"], fidx
    res_all = ppu.sample_and_group_multi(-1, 0.3, 12, xyz, normals)
    out["ppf_all_ppf"] = res_all["ppf"]
    save("group", **{k: v.numpy() for k, v in out.items()})


def gen_svd():
    """SVDHead (utils/svd.py:5-59) on CPU with matched embeddings (peaky soft correspondences, so H is
    well conditioned): a rigid-motion case and a mirrored case that takes the det < 0 branch."""
    from learning3d.utils.svd import SVDHead
    torch.manual_seed(5)
    B, d, N = 4, 64, 128
    head = SVDHead(d)
    src = torch.rand(B, N, 3) - 0.5
    ang = torch.rand(B) * 1.2
    c, s_ = torch.cos(ang), torch.sin(ang)
    Rz = torch.zeros(B, 3, 3); Rz[:, 0, 0] = c; Rz[:, 0, 1] = -s_; Rz[:, 1, 0] = s_; Rz[:, 1, 1] = c; Rz[:, 2, 2] = 1
    tgt = torch.matmul(src, Rz.transpose(1, 2)) + torch.rand(B, 1, 3)
    tgt[2:, :, 0] *= -1                               # items 2,3: mirrored target -> det(v u^T) < 0
    emb = torch.randn(B, d, N) * 3.0
    perm = torch.stack([torch.randperm(N) for _ in range(B)])
    tgt = torch.gather(tgt, 1, perm[..., None].expand(B, N, 3))          # shuffle the target order
    tgt_emb = torch.gather(emb, 2, perm[:, None, :].expand(B, d, N)) + 0.05 * torch.randn(B, d, N)
    R, t = head(emb, tgt_emb, src, tgt)
    scores = torch.softmax(torch.matmul(emb.transpose(2, 1).contiguous(), tgt_emb) / d ** 0.5, dim=2)
    src_corr = torch.matmul(tgt.permute(0, 2, 1), scores.transpose(2, 1).contiguous())
    save("svd_head", src_emb=emb.numpy(), tgt_emb=tgt_emb.numpy(), src=src.numpy(), tgt=tgt.numpy(),
         src_corr=src_corr.numpy(), R=R.numpy(), t=t.numpy())


def gen_dcp():
    """DCP (models/dcp.py:10-55) = DGCNN + Transformer + SVDHead on CPU, eval mode, small seeded weights
    (emb_dims 32) so the state_dict fits in a fixture; source = rigidly moved template."""
    from learning3d.models import DCP, DGCNN
    best = None
    for seed in range(40):
        torch.manual_seed(1000 + seed)
        net = DCP(feature_model=DGCNN(emb_dims=32), cycle=True).eval()
        template = torch.rand(2, 128, 3) - 0.5
        ang = torch.tensor([0.5, -0.7])
        c, s_ = torch.cos(ang), torch.sin(ang)
        R = torch.zeros(2, 3, 3); R[:, 0, 0] = c; R[:, 0, 1] = -s_; R[:, 1, 0] = s_; R[:, 1, 1] = c; R[:, 2, 2] = 1
        source = torch.matmul(template, R.transpose(1, 2)) + torch.tensor([[0.1, -0.2, 0.05], [0.0, 0.3, -0.1]])[:, None]
        with torch.no_grad():
            out = net(template, source)
            # conditioning of the 3x3 the head decomposes: recompute H as svd.py:23-33 does
            sf, tf = net.emb_nn(source), net.emb_nn(template)
            sp, tp = net.pointer(sf, tf)
            sf, tf = sf + sp, tf + tp
            scores = torch.softmax(torch.matmul(sf.transpose(2, 1).contiguous(), tf) / 32 ** 0.5, dim=2)
            corr = torch.matmul(template.permute(0, 2, 1), scores.transpose(2, 1).contiguous())
            srcT = source.permute(0, 2, 1)
            H = torch.matmul(srcT - srcT.mean(2, keepdim=True), (corr - corr.mean(2, keepdim=True)).transpose(2, 1))
            sv = torch.linalg.svdvals(H)
            cond = (sv[:, 2] / sv[:, 0]).min().item()
        if best is None or cond > best[0]:
            best = (cond, seed, net, template, source, out)
    cond, seed, net, template, source, out = best
    print("dcp fixture: seed", seed, "sigma_min/sigma_max", cond)
    arrays = {"template": template.numpy(), "source": source.numpy()}
    for k in ("est_R", "est_t", "est_R_", "est_t_", "est_T", "transformed_source"):
        arrays["out_" + k] = out[k].numpy()
    for k, v in net.state_dict().items():
        arrays["sd::" + k] = v.numpy()
    save("dcp_small", **arrays)


def gen_rpm():
    """RPMNet's matching tail run by the REAL reference (models/rpmnet.py:130-254): match_features on 96-d
    features, the affinity of RPMNet.compute_affinity (:266-272), sinkhorn with and without slack, the weighted
    template of RPMNet.spam (:283-287) and compute_rigid_transform (incl. one reflected item)."""
    from learning3d.models import rpmnet as R
    torch.manual_seed(99)
    B, J, K, C = 3, 70, 90, 96
    fs = torch.randn(B, J, C) * 0.3
    fr = torch.cat([fs[:, :60] + 0.05 * torch.randn(B, 60, C), torch.randn(B, K - 60, C) * 0.3], dim=1)
    dist = R.match_features(fs, fr)
    beta = torch.tensor([1.5, 4.0, 0.7]); alpha = torch.tensor([0.5, 1.0, 2.0])
    aff = -beta[:, None, None] * (dist - alpha[:, None, None])
    log_perm = R.sinkhorn(aff, n_iters=5, slack=True)
    log_noslack = R.sinkhorn(aff, n_iters=3, slack=False)
    xyz_ref = torch.rand(B, K, 3) - 0.5
    xyz_src = torch.rand(B, J, 3) - 0.5
    perm = torch.exp(log_perm)
    weighted = perm @ xyz_ref / (torch.sum(perm, dim=2, keepdim=True) + R._EPS)
    w = torch.sum(perm, dim=2)
    T = R.compute_rigid_transform(xyz_src, weighted, weights=w)
    # a second, well conditioned rigid-transform case with a reflection: b = mirrored a
    a2 = torch.rand(4, 200, 3) - 0.5
    rot = torch.linalg.qr(torch.randn(4, 3, 3))[0]
    rot[2:] = rot[2:] * torch.tensor([1.0, 1.0, -1.0])          # items 2, 3: improper (det < 0) maps
    b2 = a2 @ rot.transpose(1, 2) + torch.rand(4, 1, 3)
    w2 = torch.rand(4, 200)
    T2 = R.compute_rigid_transform(a2, b2, w2)
    save("rpm_tail", feat_src=fs.numpy(), feat_ref=fr.numpy(), dist=dist.numpy(), beta=beta.numpy(), alpha=alpha.numpy(),
         affinity=aff.numpy(), log_perm=log_perm.numpy(), log_noslack=log_noslack.numpy(), xyz_ref=xyz_ref.numpy(),
         xyz_src=xyz_src.numpy(), perm=perm.numpy(), weighted=weighted.numpy(), rowsum=w.numpy(), T=T.numpy(),
         a2=a2.numpy(), b2=b2.numpy(), w2=w2.numpy(), T2=T2.numpy())


def live_inputs(kind, seed):
    """Seeded inputs of tests/test_oracle_vs_live_reference.py (the test draws them again)."""
    if kind == "knn":
        rng = np.random.default_rng(500 + seed)
        B, N, k = int(rng.integers(1, 4)), int(rng.integers(40, 400)), int(rng.integers(1, 30))
        return rng.random((B, 3, N), dtype=np.float32), k
    rng = np.random.default_rng((700 if kind == "group" else 900) + seed)
    B, N, S = 2, int(rng.integers(50, 300) if kind == "group" else rng.integers(64, 200)), int(
        rng.integers(5, 40) if kind == "group" else rng.integers(8, 32))
    xyz = rng.random((B, N, 3), dtype=np.float32)
    return xyz, np.ascontiguousarray(xyz[:, :S]), rng


def gen_live():
    """The reference's pure-torch kNN / grouping helpers (utils/model_common_utils.py, pointconv_util.py,
    ppfnet_util.py) on the seeded inputs of live_inputs(); large outputs as a seeded sample."""
    from learning3d.utils import model_common_utils as mcu
    from learning3d.utils import pointconv_util as pcu
    from learning3d.utils import ppfnet_util as ppf
    out = {}
    for seed in range(4):
        x, k = live_inputs("knn", seed)
        xt = torch.from_numpy(x)
        feat = mcu.get_graph_feature(xt, k=k, device="cpu").numpy()
        flat = np.sort(np.random.default_rng(seed).choice(feat.size, 512, replace=False))
        rows = np.sort(np.random.default_rng(seed).choice(x.shape[2], min(x.shape[2], 96), replace=False))
        out["knn%d_rows" % seed] = rows.astype(np.int16)
        out["knn%d_idx" % seed] = mcu.knn(xt, k).numpy()[:, rows].astype(np.int16)
        out["knn%d_feat_flat" % seed], out["knn%d_feat" % seed] = flat.astype(np.int32), feat.reshape(-1)[flat]
    for seed in range(3):
        xyz, new_xyz, rng = live_inputs("group", seed)
        t_xyz, t_new = torch.from_numpy(xyz), torch.from_numpy(new_xyz)
        sd = mcu.square_distance(t_new, t_xyz).numpy()
        flat = np.sort(np.random.default_rng(seed).choice(sd.size, 512, replace=False))
        out["group%d_sqdist_flat" % seed], out["group%d_sqdist" % seed] = flat.astype(np.int32), sd.reshape(-1)[flat]
        ns = int(rng.integers(2, 20))
        idx, cnt = mcu.query_ball_point(0.25, ns, t_xyz, t_new, get_cnt=True)
        out["group%d_ball_idx" % seed], out["group%d_ball_cnt" % seed] = idx.numpy().astype(np.int16), cnt.numpy()
        out["group%d_fps" % seed] = mcu.farthest_point_sample(t_xyz, new_xyz.shape[1], start_with_first_point=True).numpy()
        val, kidx = mcu.knn_point(int(rng.integers(1, 12)), t_xyz, t_new)
        out["group%d_knn_val" % seed], out["group%d_knn_idx" % seed] = val.numpy(), kidx.numpy().astype(np.int16)
    for seed in range(2):
        xyz, new_xyz, rng = live_inputs("pointconv", seed)
        t_xyz, t_new = torch.from_numpy(xyz), torch.from_numpy(new_xyz)
        S = new_xyz.shape[1]
        out["pc%d_knn" % seed] = pcu.knn_point(int(rng.integers(2, 16)), t_xyz, t_new).numpy().astype(np.int16)
        out["pc%d_fps" % seed] = pcu.farthest_point_sample(t_xyz, S).numpy()
        out["pc%d_density" % seed] = pcu.compute_density(t_xyz, 0.2).numpy()
        itself = torch.arange(S).view(1, S).repeat(2, 1)
        out["pc%d_ppf_ball" % seed] = ppf.query_ball_point(0.3, 12, t_xyz, t_new, itself).numpy().astype(np.int16)
    save("live_reference", **out)


def gen_compiled_chamfer():
    """The reference's Chamfer extension (cd.forward = nnsearch on CPU) on a ragged pair of clouds."""
    import learning3d.losses.cuda.chamfer_distance as ref_cd_pkg   # JIT-builds `cd`
    rng = np.random.default_rng(7)
    a, b = torch.from_numpy(rng.random((2, 257, 3), dtype=np.float32)), torch.from_numpy(rng.random((2, 130, 3), dtype=np.float32))
    d1, d2 = torch.zeros(2, 257), torch.zeros(2, 130)
    i1, i2 = torch.zeros(2, 257, dtype=torch.int), torch.zeros(2, 130, dtype=torch.int)
    ref_cd_pkg.chamfer_distance.cd.forward(a, b, d1, d2, i1, i2)
    save("chamfer_compiled", dist1=d1.numpy(), dist2=d2.numpy(), idx1=i1.numpy(), idx2=i2.numpy())


def gen_checkpoints():
    """Parameter names and shapes of the reference's pretrained FlowNet3D and DCP checkpoints (the weights
    themselves are too large to keep): the models' state_dict layout must stay loadable."""
    import json
    out = {}
    for ck in ("exp_flownet/models/model.best.t7", "exp_dcp/models/best_model.t7"):
        sd = torch.load(os.path.join(REF, "pretrained", ck), map_location="cpu", weights_only=False)
        out[ck] = {k: list(v.shape) for k, v in sd.items()}
    path = os.path.join(HERE, "reference_checkpoints.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print("wrote", path)


if __name__ == "__main__":
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0")
    os.environ.setdefault("TORCH_EXTENSIONS_DIR", tempfile.mkdtemp(prefix="l3dref_ext_"))
    os.environ["CC"] = "/usr/bin/gcc"; os.environ["CXX"] = "/usr/bin/g++"
    import_reference()
    which = sys.argv[1:] or ["knn", "chamfer", "group", "svd", "dcp", "rpm", "live", "chamfer_compiled", "checkpoints"]
    if "rpm" in which:
        gen_rpm()
    if "knn" in which:
        gen_knn()
    if "chamfer" in which:
        gen_chamfer()
    if "group" in which:
        gen_group()
    if "svd" in which:
        gen_svd()
    if "dcp" in which:
        gen_dcp()
    if "live" in which:
        gen_live()
    if "chamfer_compiled" in which:
        gen_compiled_chamfer()
    if "checkpoints" in which:
        gen_checkpoints()
