"""Callers of the hot path (API-compat): state_dict compatibility with the reference's checkpoints (CPU) and GPU
forward checks."""
import json

import numpy as np
import pytest
import torch


def test_reference_checkpoints_load(golden_dir):
    """The parameter names and shapes of the reference's pretrained FlowNet3D and DCP checkpoints (recorded by
    tests/golden/make_golden.py gen_checkpoints) load strictly into our modules."""
    from learning3d_b200.models import DGCNN, FlowNet3D
    with open(f"{golden_dir}/reference_checkpoints.json") as f:
        shapes = json.load(f)
    ckpt = lambda name: {k: torch.zeros(s) for k, s in shapes[name].items()}
    sd = ckpt("exp_flownet/models/model.best.t7")
    FlowNet3D().load_state_dict(sd, strict=True)                   # identical module tree / names
    dcp = ckpt("exp_dcp/models/best_model.t7")
    emb = {k[len("emb_nn."):]: v for k, v in dcp.items() if k.startswith("emb_nn.")}
    DGCNN(emb_dims=512).load_state_dict(emb, strict=True)
    from learning3d_b200.utils import SVDHead
    SVDHead(512).load_state_dict({"reflect": dcp["head.reflect"]}, strict=True)


@pytest.mark.gpu
def test_dgcnn_forward_matches_torch_graph():
    """DGCNN = get_graph_feature (ours) + a torch conv stack (as in the reference).  The graph feature must
    equal the reference's matmul+topk+gather construction row for row (rows with an exact key tie aside:
    topk's tie order is unspecified); the forward must then agree to conv tolerance."""
    from learning3d_b200.models import DGCNN
    from learning3d_b200.utils import get_graph_feature
    from oracle import ref_torch
    torch.manual_seed(0)
    net = DGCNN(emb_dims=256).cuda().eval()
    x = torch.rand(4, 1024, 3, device="cuda")
    xt = x.permute(0, 2, 1).contiguous()
    with torch.no_grad():
        y = net(x)
        g_ref = ref_torch.get_graph_feature(xt, k=20).contiguous()
        g_our = get_graph_feature(xt, k=20)
        same_rows = (g_ref == g_our).all(1).all(-1)                       # [B, N]
        assert same_rows.float().mean().item() > 0.999
        h, pooled = g_ref, []
        for i in range(1, 5):
            h = torch.relu(getattr(net, f"bn{i}")(getattr(net, f"conv{i}")(h)))
            pooled.append(h.max(dim=-1, keepdim=True)[0])
        want = torch.relu(net.bn5(net.conv5(torch.cat(pooled, 1)))).view(4, -1, 1024)
    assert y.shape == (4, 256, 1024) and torch.isfinite(y).all()
    rel = (y - want).abs().max().item() / max(want.abs().max().item(), 1e-6)
    print("DGCNN forward max rel diff vs reference graph:", rel)
    assert rel < 2e-2      # tie rows can move a neighbour; everything else agrees to conv rounding


@pytest.mark.gpu
def test_flownet3d_forward_runs_on_dropin_ops():
    from learning3d_b200.models import FlowNet3D
    torch.manual_seed(1)
    net = FlowNet3D().cuda().eval()
    pc1 = (torch.rand(2, 3, 2048, device="cuda") * 4 - 2)
    pc2 = pc1 + 0.05 * torch.randn_like(pc1)
    with torch.no_grad():
        flow = net(pc1, pc2, pc1.clone(), pc2.clone())
    assert flow.shape == (2, 3, 2048) and torch.isfinite(flow).all()
    # training-mode backward through gather / group ops
    net.train()
    out = net(pc1, pc2, pc1.clone(), pc2.clone())
    out.square().mean().backward()
    g = net.sa1.mlp_convs[0].weight.grad
    assert g is not None and torch.isfinite(g).all() and g.abs().sum() > 0


@pytest.mark.gpu
def test_dcp_forward_matches_reference_fixture(golden_dir):
    """DCP = DGCNN (fused kNN graph) + Transformer + SVDHead (Kabsch kernel), weights and expected outputs
    from the REAL reference run on CPU (tests/golden/make_golden.py gen_dcp).  End-to-end fp32 through GPU
    convolutions / fused attention vs the reference's CPU kernels: 1e-3 on R, t (H is well conditioned:
    sigma_min/sigma_max = 0.23); the SVD tail itself is checked to 1e-5 in test_gpu_emd_svd.py."""
    from learning3d_b200.models import DCP, DGCNN
    g = np.load(f"{golden_dir}/dcp_small.npz")
    net = DCP(feature_model=DGCNN(emb_dims=32), cycle=True)
    sd = {k[4:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd::")}
    net.load_state_dict(sd, strict=True)
    net = net.cuda().eval()
    with torch.no_grad():
        out = net(torch.from_numpy(g["template"]).cuda(), torch.from_numpy(g["source"]).cuda())
    for k in ("est_R", "est_t", "est_R_", "est_t_", "est_T", "transformed_source"):
        np.testing.assert_allclose(out[k].cpu().numpy(), g["out_" + k], atol=1e-3, err_msg=k)
    R = out["est_R"].cpu().numpy()
    np.testing.assert_allclose(R @ R.transpose(0, 2, 1), np.tile(np.eye(3), (2, 1, 1)), atol=1e-5)
    assert out["r"].shape == (2, 32, 128)


@pytest.mark.gpu
def test_flownet3d_eval_fused_mlps_match_torch_layers():
    """FlowNet3D in eval mode: shared MLPs + max over the neighbours on tcgen05 (BatchNorm folded) and both frames
    batched through the encoder, against the same module with its torch layers (cuDNN fp32, TF32 off)."""
    from learning3d_b200.models import FlowNet3D
    from learning3d_b200.utils import fused_mlp
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(4)
    net = FlowNet3D().cuda()
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
                m.running_mean.normal_(0, 0.1); m.running_var.uniform_(0.5, 1.5)
                m.weight.uniform_(0.7, 1.3); m.bias.normal_(0, 0.1)
    net.eval()
    pc1 = torch.rand(4, 3, 2048, device="cuda") * 4 - 2
    pc2 = pc1 + 0.05 * torch.randn_like(pc1)
    f1 = torch.rand(4, 3, 2048, device="cuda"); f2 = torch.rand(4, 3, 2048, device="cuda")
    with torch.no_grad():
        got = net(pc1, pc2, f1, f2)
        fused_mlp.ENABLED = False
        try:
            want = net(pc1, pc2, f1, f2)
        finally:
            fused_mlp.ENABLED = True
    err = (got - want).abs().max().item()
    print("FlowNet3D eval fused vs torch layers: max |diff| = %.3g (|flow| max %.3g)" % (err, want.abs().max().item()))
    assert err <= 2e-5 * max(1.0, want.abs().max().item())
