"""TEST INFRASTRUCTURE ONLY — deterministic model weights, the seeded inputs of the model-level fixtures
(tests/golden/make_golden_gpu.py) and compact digests of large outputs.

The reference's model classes and ours share parameter names and shapes (tests/test_models.py), so
`seeded_state_dict` gives both the same weights without storing them: every entry is drawn from a numpy
generator keyed by the seed and the entry's name, independent of the order the modules register it.
"""
import zlib

import numpy as np
import torch


def seeded_state_dict(module, seed):
    """A state_dict for `module` with reproducible weights: conv / linear U(+-1/sqrt(fan_in)), normalisation
    scales U(0.7, 1.3), shifts and biases N(0, 0.05), running statistics mean N(0, 0.1) and var U(0.5, 1.5).
    Integer buffers and the SVD head's fixed reflection matrix keep the module's own values."""
    out = {}
    for name, t in module.state_dict().items():
        if not t.is_floating_point() or name.endswith("reflect"):
            out[name] = t.clone()
            continue
        rng = np.random.default_rng([seed, zlib.crc32(name.encode())])
        shape, leaf = tuple(t.shape), name.rsplit(".", 1)[-1]
        if t.dim() >= 2:
            bound = 1.0 / np.sqrt(np.prod(shape[1:]))
            v = rng.uniform(-bound, bound, shape)
        elif leaf == "running_var":
            v = rng.uniform(0.5, 1.5, shape)
        elif leaf == "running_mean":
            v = rng.normal(0.0, 0.1, shape)
        elif leaf in ("weight", "a_2"):
            v = rng.uniform(0.7, 1.3, shape)
        else:
            v = rng.normal(0.0, 0.05, shape)
        out[name] = torch.from_numpy(v.astype(np.float32))
    return out


def row_digest(idx):
    """One uint16 per row of an index array [..., k] that depends only on the SET of indices in the row."""
    h = ((np.asarray(idx, dtype=np.int64) + 1) * 40503) % 65521
    return ((h * h) % 65521).sum(-1).astype(np.int64) % 65521


def random_rigid(B, gen, max_deg=45.0, max_t=1.0):
    """Random rotations (angle <= max_deg about a random axis) and translations U(-max_t, max_t) (SURVEY.md §8d C3)."""
    axis = torch.randn(B, 3, generator=gen)
    axis = axis / axis.norm(dim=1, keepdim=True)
    ang = torch.rand(B, generator=gen) * np.deg2rad(max_deg)
    K = torch.zeros(B, 3, 3)
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 0] = -axis[:, 2], axis[:, 1], axis[:, 2]
    K[:, 1, 2], K[:, 2, 0], K[:, 2, 1] = -axis[:, 0], -axis[:, 1], axis[:, 0]
    s, c = torch.sin(ang)[:, None, None], torch.cos(ang)[:, None, None]
    R = torch.eye(3).expand(B, 3, 3) + s * K + (1 - c) * (K @ K)
    t = (torch.rand(B, 3, generator=gen) * 2 - 1) * max_t
    return R, t


def dcp_inputs(B=32, N=1024):
    """C3 inputs (CPU generator, seed 1234): centred template, source = template under a small random rigid motion
    (<= 5 degrees, |t| <= 0.1).  With untrained weights DCP finds the right correspondences only for small motions;
    then the 3x3 matrix its SVD head decomposes is well conditioned and R is fixed to fp32 precision (the
    reference's own fp32 and fp64 forwards agree to 5e-7), which a 1e-5 comparison needs."""
    gen = torch.Generator().manual_seed(1234)
    template = torch.rand(B, N, 3, generator=gen)
    template = template - template.mean(dim=1, keepdim=True)
    R, t = random_rigid(B, gen, max_deg=5.0, max_t=0.1)
    return template, template @ R.transpose(1, 2) + t[:, None, :]


def flownet_inputs(B=16, N=2048):
    """C4 inputs (CPU generator, seed 1234): pc1, pc2 = pc1 + noise, and two feature clouds, each [B, 3, N]."""
    gen = torch.Generator().manual_seed(1234)
    pc1 = torch.rand(B, 3, N, generator=gen) * 4 - 2
    pc2 = pc1 + 0.05 * torch.randn(B, 3, N, generator=gen)
    f1 = torch.rand(B, 3, N, generator=gen)
    f2 = torch.rand(B, 3, N, generator=gen)
    return pc1, pc2, f1, f2


def rpm_inputs():
    """Inputs of RPMNet's matching tail (CPU generator, seed 5): features [4, 717, 96] with 300 near-matches."""
    gen = torch.Generator().manual_seed(5)
    fs = 0.3 * torch.randn(4, 717, 96, generator=gen)
    fr = 0.3 * torch.randn(4, 717, 96, generator=gen)
    fr[:, :300] = fs[:, :300] + 0.03 * torch.randn(4, 300, 96, generator=gen)
    xyz_ref = torch.rand(4, 717, 3, generator=gen) - 0.5
    xyz_src = torch.rand(4, 717, 3, generator=gen) - 0.5
    return fs, fr, xyz_ref, xyz_src


def rpm_tail(R, fs, fr, xyz_ref, xyz_src):
    """match_features -> sinkhorn -> weighted correspondences -> compute_rigid_transform, with the functions of
    the rpmnet module `R` (the reference's, or ours)."""
    d = R.match_features(fs, fr)
    lp = R.sinkhorn(-2.0 * (d - 0.5), n_iters=5, slack=True)
    perm = torch.exp(lp)
    wt = perm @ xyz_ref / (torch.sum(perm, dim=2, keepdim=True) + 1e-5)
    return d, lp, R.compute_rigid_transform(xyz_src, wt, weights=torch.sum(perm, dim=2))


def sample_index(n, k, key):
    """k sorted distinct positions out of n (all of them when n <= k), the same for every caller passing `key`: the
    fixtures store seeded samples of large outputs, and the tests draw the positions again."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(zlib.crc32(key.encode())).choice(n, k, replace=False))


def array_digest(a):
    """One uint64 per leading index of `a`: the first 8 bytes of the SHA-256 of that slice, with integers taken as
    int32 and floats as float32.  Equal digests mean bit-equal slices, so a fixture can cover every row of a large
    output that must match exactly at the cost of 8 bytes per item."""
    import hashlib
    a = np.asarray(a)
    a = np.ascontiguousarray(a.astype(np.int32 if a.dtype.kind in "iu" else np.float32))
    return np.array([int.from_bytes(hashlib.sha256(x.tobytes()).digest()[:8], "little") for x in a], dtype=np.uint64)
