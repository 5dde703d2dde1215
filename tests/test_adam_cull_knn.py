"""Sparse Adam, LoD cull and grid-hash KNN: CPU checks of the oracles, GPU parity through the C ABI."""
import numpy as np
import pytest
import torch

import oracle
from artdeco_b200 import synthetic
from helpers import assert_close, golden_sample, reference_builds


# ----------------------------------------------------------------------------- oracle (CPU) ----
def test_knn_oracle_matches_cdist():
    g = torch.Generator().manual_seed(0)
    pts = torch.randn(500, 3, generator=g)
    d2 = torch.cdist(pts.double(), pts.double()) ** 2
    d2.fill_diagonal_(float("inf"))
    ref, ref_i = d2.topk(3, largest=False)
    m = oracle.knn_mean3(pts.numpy())
    assert np.allclose(m, ref.mean(1).numpy(), rtol=1e-5)
    d, ids = oracle.knn_index(pts.numpy(), 3)
    assert (ids == ref_i.numpy()).mean() > 0.999
    assert np.allclose(d, ref.numpy(), rtol=1e-4, atol=1e-7)


def test_knn_oracle_small_and_duplicates():
    pts = np.array([[0, 0, 0], [1, 0, 0], [1, 0, 0]], np.float32)
    d, ids = oracle.knn_index(pts, 4)
    assert ids[0].tolist() == [1, 2, -1, -1] and ids[1].tolist()[:2] == [2, 0]   # duplicate at distance 0 counts
    assert d[0, 2] > 1e30 and d[1, 0] == 0.0


# ----------------------------------------------------------------------------- Adam (GPU) ----
@pytest.mark.gpu
@pytest.mark.parametrize("N,M", [(1000, 3), (1000, 48), (777, 1), (513, 4)])
@pytest.mark.parametrize("lr_kind", ["scalar0d", "per_row", "per_elem", "float"])
def test_adam_update_matches_oracle(cuda, N, M, lr_kind):
    from artdeco_b200.adam import adamUpdate, adamUpdateBasic
    g = torch.Generator().manual_seed(N + M)
    p, gr, m1 = (torch.randn(N, M, generator=g) for _ in range(3))
    m2 = torch.rand(N, M, generator=g)
    vis = torch.rand(N, generator=g) > 0.4
    if lr_kind == "scalar0d":
        lr = torch.tensor(3e-3)
    elif lr_kind == "per_row":
        lr = torch.rand(N, generator=g) * 1e-2
    elif lr_kind == "per_elem":
        lr = torch.rand(N, M, generator=g) * 1e-2
    else:
        lr = 2e-3
    lr_np = lr.numpy() if isinstance(lr, torch.Tensor) else np.float32(lr)
    P, A, V = oracle.adam(p.numpy(), gr.numpy(), m1.numpy(), m2.numpy(), vis.numpy(), lr_np.reshape(-1), 0.5, 0.99, 1e-15)
    pd, gd, ad, vd = (t.clone().to(cuda) for t in (p, gr, m1, m2))
    lr_d = lr.to(cuda) if isinstance(lr, torch.Tensor) else lr
    adamUpdate(pd, gd, ad, vd, vis.to(cuda), lr_d, 0.5, 0.99, 1e-15, N, M)
    # fp32 elementwise op: tolerance 1e-6 of scale (FMA contraction on the GPU, none in the oracle)
    assert_close(pd, P, rtol=2e-6, what="param")
    assert_close(ad, A, rtol=2e-6, what="exp_avg")
    assert_close(vd, V, rtol=2e-6, what="exp_avg_sq")
    inv = ~vis
    assert torch.equal(pd.cpu()[inv], p[inv]) and torch.equal(ad.cpu()[inv], m1[inv]), "invisible rows must be untouched"
    if lr_kind in ("float", "scalar0d"):
        pb, ab, vb = p.clone().to(cuda), m1.clone().to(cuda), m2.clone().to(cuda)
        adamUpdateBasic(pb, gd, ab, vb, lr_d, 0.8, 0.99, 1e-15)
        Pb, Ab, Vb = oracle.adam(p.numpy().reshape(-1, 1), gr.numpy().reshape(-1, 1), m1.numpy().reshape(-1, 1),
                                 m2.numpy().reshape(-1, 1), None, lr_np.reshape(-1), 0.8, 0.99, 1e-15)
        assert_close(pb.reshape(-1, 1), Pb, rtol=2e-6, what="basic param")


@pytest.mark.gpu
def test_adam_rejects_bad_lr_shape(cuda):
    from artdeco_b200 import _lib
    from artdeco_b200.adam import adamUpdate
    t = torch.zeros(10, 3, device=cuda)
    with pytest.raises(_lib.ArtdecoB200Error):
        adamUpdate(t, t.clone(), t.clone(), t.clone(), torch.ones(10, dtype=torch.bool, device=cuda),
                   torch.ones(7, device=cuda), 0.9, 0.99, 1e-8, 10, 3)


# ----------------------------------------------------------------------------- LoD cull (GPU) ----
@pytest.mark.gpu
@pytest.mark.parametrize("N", [0, 1, 100_000])
def test_lod_select_matches_reference_formula(cuda, N):
    """Formula of h3dgsv3.py:626-645 evaluated with torch on the CPU (it IS the reference code path)."""
    from artdeco_b200.cull import lod_cull, lod_select
    sc = synthetic.raster_scene(max(N, 1), seed=4)
    xyz, d_max = sc["means"][:N], sc["d_max"][:N] * 0.3
    cam = torch.tensor([0.3, -0.2, 1.0])
    dist = (xyz - cam).norm(dim=1, keepdim=True)
    sel = (dist < 2 * d_max).squeeze(-1)
    amask = torch.logical_and(dist > d_max, dist < 2 * d_max).squeeze(-1)
    ratio = (2 * d_max - dist) / d_max
    ratio[~amask] = 1.0
    mask, ids, r = lod_select(xyz.to(cuda), d_max.to(cuda), cam.to(cuda))
    # the strict '<' tests sit on fp32 distances: allow the handful of points whose distance differs in the last ulp
    mism = (mask.cpu() != sel)
    assert mism.sum() <= max(2, N // 100000)
    if N:
        ok = ~mism
        assert_close(r.cpu()[ok], ratio.squeeze(-1)[ok], rtol=1e-5, what="alpha_ratio")
        assert torch.equal(ids.cpu().long(), torch.nonzero(mask.cpu()).squeeze(-1)), "ids == ascending mask positions"
    # differentiable wrapper: gradients reach opacity, gathered params and xyz (through the fade ratio)
    if N == 100_000:
        xg = xyz.to(cuda).requires_grad_(True)
        og = sc["opacities"][:N, None].to(cuda).requires_grad_(True)
        m2, xs, ops, sh_s = lod_cull(xg, d_max.to(cuda), og, cam.to(cuda), sc["sh"][:N].to(cuda))
        (ops.sum() + xs.sum()).backward()
        xr = xyz.clone().requires_grad_(True)
        orf = sc["opacities"][:N, None].clone().requires_grad_(True)
        dist_r = (xr - cam).norm(dim=1, keepdim=True)
        ratio_r = (2 * d_max - dist_r) / d_max
        ratio_r = torch.where(amask[:, None], ratio_r, torch.ones_like(ratio_r))
        ((orf * ratio_r)[sel].sum() + xr[sel].sum()).backward()
        if not mism.any():
            assert_close(og.grad, orf.grad, rtol=1e-5, what="v_opacity")
            assert_close(xg.grad, xr.grad, rtol=1e-5, what="v_xyz")


@pytest.mark.gpu
@pytest.mark.parametrize("N,K", [(1, 1), (50_000, 7), (200_000, 40)])
def test_weed_out_mask_matches_the_reference_loop(cuda, N, K):
    """weed_out_gaussians (h3dgsv3.py:942-953) restated line for line with torch on the CPU (the per-key-frame loop IS the
    reference code path) against the one-pass kernel; the same fp32 strict-'<' caveat as the LoD select applies."""
    from artdeco_b200.cull import weed_out_mask
    sc = synthetic.raster_scene(N, seed=5)
    xyz, d_max = sc["means"], sc["d_max"] * 0.2
    g = torch.Generator().manual_seed(3)
    cams = torch.stack([torch.rand(K, generator=g) * 16 - 8, torch.rand(K, generator=g) * 9 - 4.5, torch.rand(K, generator=g) * 20], -1)
    thr = 0.3
    visible_count = torch.zeros(N, dtype=torch.int)
    for k in range(K):
        ob_dist = (xyz - cams[k]).norm(dim=1, keepdim=True)
        visible_count += (ob_dist < 2 * d_max).squeeze(-1).int()
    weed = (visible_count / K) > thr
    keep, cnt = weed_out_mask(xyz.to(cuda), d_max.to(cuda), cams.to(cuda), thr, return_count=True)
    dc = (cnt.cpu() != visible_count)
    assert dc.sum() <= max(2, N * K // 100000), "visible counts (last-ulp distance ties only)"
    assert ((keep.cpu() != weed) & ~dc).sum() == 0, "keep rule count/K > threshold"


# ----------------------------------------------------------------------------- KNN (GPU) ----
@pytest.mark.gpu
@pytest.mark.parametrize("P,kind", [(5, "cloud"), (3000, "cloud"), (20000, "scene"), (4000, "plane"), (2000, "dups")])
def test_distcuda2_bit_exact_vs_oracle(cuda, P, kind):
    from artdeco_b200.knn import distCUDA2
    g = torch.Generator().manual_seed(P)
    if kind == "scene":
        pts = synthetic.raster_scene(P, seed=0)["means"]
    elif kind == "plane":
        pts = torch.rand(P, 3, generator=g) * torch.tensor([5.0, 3.0, 0.0]) + torch.tensor([0, 0, 2.0])
    elif kind == "dups":
        pts = torch.randn(P // 2, 3, generator=g).repeat(2, 1)
    else:
        pts = torch.randn(P, 3, generator=g) * torch.tensor([3.0, 1.0, 0.2])
    ref = oracle.knn_mean3(pts.numpy())
    out = distCUDA2(pts.to(cuda)).cpu().numpy()
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32)), \
        f"distCUDA2 must be bit-identical to the oracle; max diff {np.abs(out - ref).max()}"


@pytest.mark.gpu
@pytest.mark.parametrize("P,K", [(2, 4), (3000, 3), (5000, 8), (2000, 16)])
def test_distindex2_exact_knn_sets(cuda, P, K):
    from artdeco_b200.knn import distIndex2
    g = torch.Generator().manual_seed(P + K)
    pts = torch.randn(P, 3, generator=g)
    d_ref, i_ref = oracle.knn_index(pts.numpy(), K)
    d, ids = distIndex2(pts.to(cuda), K)
    d, ids = d.view(P, K).cpu().numpy(), ids.view(P, K).cpu().numpy()
    assert np.array_equal(d.view(np.uint32), d_ref.view(np.uint32)), "sorted squared distances are bit-exact"
    # ids: exact wherever the K-th and (K+1)-th distances are not tied (ties are traversal-dependent in the reference too)
    distinct = np.ones(P, bool)
    distinct[1:] &= True
    same = (ids == i_ref).all(1)
    tied = np.array([len(np.unique(row)) < len(row) for row in d_ref])
    assert (same | tied).all()
    assert same.mean() > 0.99


@pytest.mark.gpu
def test_distindexq_query_subset_and_candidates(cuda):
    from artdeco_b200.knn import distIndexQ
    g = torch.Generator().manual_seed(9)
    P, K = 4000, 5
    pts = torch.randn(P, 3, generator=g)
    q = torch.randperm(P, generator=g)[:700].to(torch.int32)
    n = torch.randperm(P, generator=g)[:1500].to(torch.int32)
    cand = np.zeros(P, np.uint8)
    cand[n.numpy()] = 1
    d_ref, i_ref = oracle.knn_index(pts.numpy(), K, q.numpy(), cand)
    d, ids = distIndexQ(pts.to(cuda), q.to(cuda), n.to(cuda), K)
    d, ids = d.view(-1, K).cpu().numpy(), ids.view(-1, K).cpu().numpy()
    assert np.array_equal(d.view(np.uint32), d_ref.view(np.uint32))
    assert (ids == i_ref).mean() > 0.999
    assert cand[ids[ids >= 0]].all(), "neighbours come from the candidate set only"


@pytest.mark.gpu
def test_knn_1m_properties(cuda):
    """Full size (1M points of the bench scene): symmetric-consistency properties instead of the O(P^2) oracle."""
    from artdeco_b200.knn import distCUDA2, distIndex2
    pts = synthetic.raster_scene(1_000_000, seed=0)["means"].to(cuda)
    m = distCUDA2(pts)
    d, ids = distIndex2(pts, 3)
    d, ids = d.view(-1, 3), ids.view(-1, 3)
    assert bool((d[:, 1:] >= d[:, :-1]).all()) and bool((ids >= 0).all())
    # (torch divides by a scalar through a reciprocal multiply, hence 1 ulp of slack instead of torch.equal)
    assert torch.allclose(m, (d[:, 0] + d[:, 1] + d[:, 2]) / 3.0, rtol=3e-7, atol=0), \
        "distCUDA2 == mean of distIndex2's three distances"
    # recompute the reported distances from the reported ids
    nb = pts[ids.long()]
    dd = nb - pts[:, None, :]
    rec = torch.fma(dd[..., 2], dd[..., 2], torch.fma(dd[..., 1], dd[..., 1], dd[..., 0] * dd[..., 0])) \
        if hasattr(torch, "fma") else (dd ** 2).sum(-1)
    assert torch.allclose(rec, d, rtol=1e-5, atol=0)
    # a sample of points checked against brute force
    idx = torch.randperm(1_000_000, device=cuda)[:256]
    bf = ((pts[idx][:, None, :] - pts[None, :, :]) ** 2).sum(-1)
    bf[torch.arange(256, device=cuda), idx] = float("inf")
    ref = bf.topk(3, largest=False).values
    assert torch.allclose(ref, d[idx], rtol=1e-5, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [5000, 200_000])
def test_distcuda2_bit_identical_to_the_reference_build(cuda, P):
    """Against the reference's OWN simple_knn.cu compiled for sm_100 (oracle/build_ref.py): seeded samples of its outputs
    on these points are stored in tests/golden/reference_builds.npz."""
    from artdeco_b200.knn import distCUDA2, distIndex2
    gold = reference_builds()
    want_mean, want_sorted = gold[f"knn_{P}_distcuda2"], gold[f"knn_{P}_distindex2_sorted"]
    pts = synthetic.raster_scene(P, seed=2)["means"].to(cuda)
    got = distCUDA2(pts).cpu().numpy()[golden_sample(P, len(want_mean))]
    assert np.array_equal(got.view(np.uint32), want_mean.view(np.uint32)), "distCUDA2 must equal the reference bit for bit"
    K = 6
    do, _ = distIndex2(pts, K)
    got = do.view(P, K).cpu().numpy()[golden_sample(P, len(want_sorted), seed=1)]
    assert np.array_equal(got.view(np.uint32), want_sorted.view(np.uint32)), \
        "same K nearest distances (reference order is unspecified)"


# ----------------------------------------------------------------------------- covariance MLP (GPU) ----
@pytest.mark.gpu
@pytest.mark.parametrize("Fg,Fl,N", [(16, 16, 5000), (32, 32, 3000), (16, 16, 1)])
def test_cov_mlp_matches_reference_torch_block(cuda, Fg, Fl, N):
    """The reference block itself (h3dgsv3.py:656-662 with mlp_cov of :173-177) evaluated by torch in fp64 is the oracle."""
    import torch.nn as nn
    import torch.nn.functional as F
    from artdeco_b200.covmlp import cov_mlp_modulate
    g = torch.Generator().manual_seed(Fg + N)
    G = 37
    D = Fg + Fl
    mlp = nn.Sequential(nn.Linear(D, D), nn.ReLU(True), nn.Linear(D, 7))
    with torch.no_grad():
        for p in mlp.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * 0.3)
    scaling, rotation = torch.rand(N, 3, generator=g) * 0.1, torch.randn(N, 4, generator=g)
    lf, gf = torch.randn(N, Fl, generator=g), torch.randn(G, Fg, generator=g)
    cls = torch.randint(0, G, (N, 1), generator=g)
    vs, vr = torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g)
    # reference in fp64 on the CPU
    mlp64 = nn.Sequential(nn.Linear(D, D), nn.ReLU(True), nn.Linear(D, 7)).double()
    mlp64.load_state_dict({k: v.double() for k, v in mlp.state_dict().items()})
    ins = [t.double().requires_grad_(True) for t in (scaling, rotation, lf, gf)]
    sr = mlp64(torch.cat([ins[3][cls.squeeze(-1)], ins[2]], 1))
    s_ref = ins[0] * torch.sigmoid(sr[:, :3])
    r_ref = F.normalize(ins[1] * sr[:, 3:])
    ((s_ref * vs.double()).sum() + (r_ref * vr.double()).sum()).backward()
    # ours
    mlp_c = mlp.to(cuda)
    outs = [t.to(cuda).requires_grad_(True) for t in (scaling, rotation, lf, gf)]
    s_o, r_o = cov_mlp_modulate(outs[0], outs[1], outs[2], outs[3], cls.to(cuda), mlp_c)
    ((s_o * vs.to(cuda)).sum() + (r_o * vr.to(cuda)).sum()).backward()
    assert_close(s_o, s_ref, rtol=1e-5, what="scaling_out")
    assert_close(r_o, r_ref, rtol=1e-5, what="rotation_out")
    for name, a, b in zip(("v_scaling", "v_rotation", "v_local_feat", "v_global_feat"), outs, ins):
        assert_close(a.grad, b.grad, rtol=2e-5, what=name)
    for (n1, p1), (_, p2) in zip(mlp_c.named_parameters(), mlp64.named_parameters()):
        assert_close(p1.grad, p2.grad, rtol=2e-5, what="v_" + n1)
