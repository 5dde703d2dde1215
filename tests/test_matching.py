"""Dense matching (SURVEY.md §8f rank 1): mast3r_slam_backends.iter_proj / refine_matches + VSLAM/utils_matching.py glue.
Oracle: oracle/matching_ref.py (PyTorch restatement) and stored outputs of the reference's OWN kernels compiled from
VSLAM/backend/src/matching_kernels.cu (tests/golden/reference_builds.npz).
Contract: refine_matches is integer/fp16 work -> BIT-EXACT; iter_proj is an fp32 LM iteration -> sub-pixel positions within
1e-3 px and convergence flags equal on >= 99.9 % of points (the reference build itself is compiled with --use_fast_math)."""
import math

import numpy as np
import pytest
import torch

from helpers import golden_sample, reference_builds
from oracle import matching_ref as mr

CFG = {"matching": dict(max_iter=10, lambda_init=1e-8, convergence_thresh=1e-6, dist_thresh=1e-1, radius=4, dilation_max=5)}


def _scene(b=2, h=48, w=64, seed=0, rot_deg=1.5, F=24):
    """A smooth surface seen by two slightly rotated cameras: X11 = view-1 points in frame 1, X21 = view-2 points in frame 1."""
    g = torch.Generator().manual_seed(seed)
    v, u = torch.meshgrid(torch.arange(h, dtype=torch.float32), torch.arange(w, dtype=torch.float32), indexing="ij")
    f = 0.9 * w
    def rays(uu, vv):
        d = torch.stack(((uu - w / 2) / f, (vv - h / 2) / f, torch.ones_like(uu)), -1)
        return d / d.norm(dim=-1, keepdim=True)
    def depth(d):      # smooth surface as a function of direction
        return 3.0 + 0.6 * torch.sin(3.0 * d[..., 0]) * torch.cos(2.0 * d[..., 1]) + 0.3 * d[..., 0]
    X11, X21, D11, D21 = [], [], [], []
    basis = torch.randn(6, F, generator=g)
    def desc(d):
        feats = torch.stack((torch.sin(9 * d[..., 0]), torch.cos(7 * d[..., 1]), torch.sin(5 * d[..., 0] + 4 * d[..., 1]),
                             torch.cos(11 * d[..., 0] - 3 * d[..., 1]), d[..., 0] * 3, d[..., 1] * 3), -1)
        o = feats @ basis
        return o / o.norm(dim=-1, keepdim=True)
    for k in range(b):
        a = math.radians(rot_deg * (k + 1))
        R = torch.tensor([[math.cos(a), 0, math.sin(a)], [0, 1, 0], [-math.sin(a), 0, math.cos(a)]], dtype=torch.float32)
        d1 = rays(u, v)
        d2 = rays(u, v) @ R.T                       # view-2 pixel directions expressed in frame 1
        X11.append(d1 * depth(d1)[..., None] + 1e-4 * torch.randn(h, w, 3, generator=g))
        X21.append(d2 * depth(d2)[..., None] + 1e-4 * torch.randn(h, w, 3, generator=g))
        D11.append(desc(d1)); D21.append(desc(d2))
    return torch.stack(X11), torch.stack(X21), torch.stack(D11), torch.stack(D21)


def test_oracle_recovers_known_correspondence():
    X11, X21, D11, D21 = _scene(b=1, h=32, w=40)
    idx, valid, p, p1 = mr.match_iterative_proj(CFG["matching"], X11, X21, D11, D21)
    assert idx.shape == (1, 32 * 40) and valid.shape == (1, 32 * 40, 1) and valid.float().mean() > 0.5   # coarse 40-px image: truncating to integer pixels costs up to ~0.1 in 3-D
    # a converged match reproduces the 3-D point: X11 sampled at the sub-pixel match == X21
    m = valid[0, :, 0]
    s = mr._bilinear(X11, p[..., 0], p[..., 1])[0][m]
    assert (s - X21.reshape(1, -1, 3)[0][m]).norm(dim=-1).max() < 2e-2
    # matching an image with itself is the identity (interior pixels; the border is clamped to [1, w-2]) when every
    # pixel's descriptor is distinctive (score 1 with itself, ~0 with the others)
    Dr = torch.nn.functional.normalize(torch.randn(1, 32, 40, 24, generator=torch.Generator().manual_seed(7)), dim=-1)
    idx2, valid2, _, _ = mr.match_iterative_proj(CFG["matching"], X11, X11, Dr, Dr)
    grid = torch.arange(32 * 40).view(32, 40)[1:-1, 1:-1].reshape(-1)
    assert (idx2[0][grid] == grid).float().mean() > 0.99


def _pixel_grid(h, w):
    """(u, v) of every pixel in row-major order: the position each point starts from."""
    v, u = torch.meshgrid(torch.arange(h), torch.arange(w), indexing="ij")
    return torch.stack((u.reshape(-1), v.reshape(-1)), -1)


def _gpu_inputs(cuda, **kw):
    return [t.to(cuda).contiguous() for t in _scene(**kw)]


@pytest.mark.gpu
def test_prep_and_iter_proj_match_oracle(cuda):
    from artdeco_b200 import matching as M
    X11, X21, D11, D21 = _gpu_inputs(cuda, b=2, h=96, w=128, seed=1)
    rays, pts, p_init = M.prep_for_iter_proj(X11, X21, None)
    r_ref, pts_ref, p_ref = mr.prep_for_iter_proj(X11, X21, None)
    assert (rays - r_ref).abs().max() < 2e-6 and (pts - pts_ref).abs().max() < 2e-7 and torch.equal(p_init, p_ref)
    init = torch.randint(0, 96 * 128, (2, 96 * 128), device=cuda)
    assert torch.equal(M.prep_for_iter_proj(X11, X21, init)[2], mr.prep_for_iter_proj(X11, X21, init)[2])
    c = CFG["matching"]
    p, conv = M.iter_proj(rays, pts, p_init, c["max_iter"], c["lambda_init"], c["convergence_thresh"])
    p_o, conv_o = mr.iter_proj(r_ref, pts_ref, p_ref, c["max_iter"], c["lambda_init"], c["convergence_thresh"])
    assert conv.dtype == torch.bool and conv.float().mean() > 0.6
    both = conv & conv_o
    assert (conv == conv_o).float().mean() >= 0.999
    assert ((p - p_o).abs().amax(-1)[both] < 1e-3).float().mean() >= 0.999


@pytest.mark.gpu
@pytest.mark.parametrize("F", [24, 16])
def test_refine_matches_bit_exact_vs_oracle(cuda, F):
    from artdeco_b200 import matching as M
    X11, X21, D11, D21 = _gpu_inputs(cuda, b=2, h=40, w=56, seed=2, F=F)
    g = torch.Generator().manual_seed(3)
    p1 = torch.stack((torch.randint(-2, 58, (2, 40 * 56), generator=g), torch.randint(-2, 42, (2, 40 * 56), generator=g)), -1).to(cuda)
    p1[:, :100] = p1[:, :100].clamp(0, 39)          # some far outside, some inside
    a = D11.half().contiguous()
    q = (D21 + 0.05 * torch.randn(D21.shape, generator=g).to(cuda)).reshape(2, -1, F).half().contiguous()
    out, lin = M.refine_matches(a, q, p1, 3, 4, return_linear=True)
    ref = mr.refine_matches(a, q, p1, 3, 4)
    assert torch.equal(out, ref), "refine_matches must reproduce the reference's fp16 arithmetic exactly"
    assert torch.equal(lin, out[..., 0] + 56 * out[..., 1])
    # radius 0 / dilation 0 keep the input
    assert torch.equal(M.refine_matches(a, q, p1, 0, 3)[0], mr.refine_matches(a, q, p1, 0, 3))


@pytest.mark.gpu
def test_matches_the_reference_cuda_build(cuda):
    """The reference's own matching_kernels.cu (built for sm_100 with its --use_fast_math flags) on the same inputs: its
    convergence flags, a seeded sample of its positions, and its refine_matches input and output are stored in
    tests/golden/reference_builds.npz."""
    from artdeco_b200 import matching as M
    gold = reference_builds()
    X11, X21, D11, D21 = _gpu_inputs(cuda, b=2, h=192, w=256, seed=4)
    c = CFG["matching"]
    rays, pts, p_init = M.prep_for_iter_proj(X11, X21, None)
    p, conv = M.iter_proj(rays, pts, p_init, c["max_iter"], c["lambda_init"], c["convergence_thresh"])
    conv_r = torch.from_numpy(np.unpackbits(gold["match_iter_proj_converged"], count=conv.numel()).astype(bool))
    conv = conv.reshape(-1).cpu()
    assert (conv == conv_r).float().mean() >= 0.999
    i = golden_sample(conv.numel(), len(gold["match_iter_proj_p"]))
    p_r = torch.from_numpy(gold["match_iter_proj_p"])
    both = conv[i] & conv_r[i]
    assert ((p.reshape(-1, 2).cpu()[i] - p_r).abs().amax(-1)[both] < 1e-3).float().mean() >= 0.999
    p1 = _pixel_grid(192, 256) + torch.from_numpy(gold["match_refine_p1_offset"]).long()
    a, q = D11.half().contiguous(), D21.reshape(2, -1, 24).half().contiguous()
    (mine,) = M.refine_matches(a, q, p1.to(cuda), c["radius"], c["dilation_max"])
    theirs = p1 + torch.from_numpy(gold["match_refine_out_offset"]).long()
    assert torch.equal(mine.cpu(), theirs), "refine_matches vs the reference build: bit-exact"


@pytest.mark.gpu
def test_match_end_to_end_at_512(cuda):
    """utils_matching.match at the BASELINE image size: agreement with the oracle flow, and the identity property."""
    from artdeco_b200 import matching as M
    X11, X21, D11, D21 = _gpu_inputs(cuda, b=2, h=512, w=512, seed=5, rot_deg=0.8)
    idx, valid = M.match(CFG, X11, X21, D11, D21)
    assert idx.shape == (2, 512 * 512) and idx.dtype == torch.int64 and valid.shape == (2, 512 * 512, 1)
    idx_o, valid_o, _, _ = mr.match_iterative_proj(CFG["matching"], X11, X21, D11, D21)
    assert (valid == valid_o).float().mean() >= 0.999
    assert (idx == idx_o).float().mean() >= 0.995      # a sub-pixel position next to an integer boundary may truncate differently
    # the fused flow's chunk-planar fp16 descriptors must give exactly what the row-major kernel gives on the same p1
    p1, v1 = M._project_and_filter(CFG["matching"], X11, X21, None)
    _, lin = M.refine_matches(D11.half().contiguous(), D21.reshape(2, -1, 24).half().contiguous(), p1, 4, 5, return_linear=True)
    assert torch.equal(lin, idx) and torch.equal(v1.unsqueeze(-1), valid)
    Dr = torch.nn.functional.normalize(torch.randn(2, 512, 512, 24, generator=torch.Generator().manual_seed(7)), dim=-1).to(cuda)
    ident, v2 = M.match(CFG, X11, X11, Dr, Dr)
    grid = torch.arange(512 * 512, device=cuda).view(512, 512)[1:-1, 1:-1].reshape(-1)
    assert (ident[0][grid] == grid).float().mean() > 0.99 and v2.float().mean() > 0.95
    idx_p, valid_p = M.match_pi3(CFG, X11, X21)
    assert idx_p.shape == (2, 512 * 512) and torch.equal(valid_p.unsqueeze(-1), valid)


@pytest.mark.gpu
def test_matching_rejects_bad_inputs(cuda):
    from artdeco_b200 import _lib, matching as M
    with pytest.raises(_lib.ArtdecoB200Error):
        M.iter_proj(torch.zeros(1, 8, 8, 9), torch.zeros(1, 64, 3), torch.zeros(1, 64, 2), 1, 1e-8, 1e-6)
    with pytest.raises(TypeError):
        M.refine_matches(torch.zeros(1, 8, 8, 24, device=cuda), torch.zeros(1, 64, 24, device=cuda),
                         torch.zeros(1, 64, 2, dtype=torch.int64, device=cuda), 1, 1)
    with pytest.raises(ValueError):
        M.iter_proj(torch.zeros(1, 8, 8, 9, device=cuda).transpose(1, 2), torch.zeros(1, 64, 3, device=cuda),
                    torch.zeros(1, 64, 2, device=cuda), 1, 1e-8, 1e-6)
