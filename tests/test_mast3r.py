"""MASt3R: oracle restatement vs committed goldens (CPU), CUDA model vs goldens and vs the oracle (GPU).

Goldens (tests/golden/mast3r_small.pt, mast3r_full.pt) were produced by running the REAL reference module in the build
container on deterministic weights (tests/golden/make_mast3r_golden.py); weights are regenerated here from the same
recipe (synthetic.det_weights), so nothing but a few hundred KB of outputs is committed.
Tolerance: 1e-4 of each tensor's scale (BASELINE.json: "within 1e-4 relative fp32 for ... pointmaps")."""
import pathlib

import pytest
import torch

from artdeco_b200 import synthetic
from helpers import rel_err
from oracle import mast3r_torch as mt

GOLD = pathlib.Path(__file__).parent / "golden"
KEYS = ("pts3d", "conf", "desc", "desc_conf")


def _gold(tag):
    p = GOLD / f"mast3r_{tag}.pt"
    if not p.exists():
        pytest.skip(f"{p.name} not generated")
    return torch.load(p, weights_only=False)


def _gold_err(got, g, key):
    """max |got - golden| over the stored sample, relative to the golden tensor's scale (stored with it: max |x| over a
    denser grid than the sample, so that a sparser sample does not tighten the tolerance)."""
    got = got.detach().cpu().double()
    want = g[key].double()
    assert got.shape == want.shape, (key, got.shape, want.shape)
    return float((got - want).abs().max()) / g[key + ".scale"]


def test_oracle_matches_reference_golden_small():
    g = _gold("small")
    cfg, H, W = g["cfg"], g["H"], g["W"]
    sd = synthetic.det_weights(mt.param_shapes(cfg))
    img1, img2 = synthetic.mast3r_pair(1, H, W, seed=0)
    with torch.inference_mode():
        f1, p1 = mt.encode_image(sd, cfg, img1)
        f2, p2 = mt.encode_image(sd, cfg, img2)
        d1, d2 = mt.decoder(sd, cfg, f1, p1, f2, p2)
        o1 = mt.downstream_head(sd, cfg, 1, d1, H, W)
        o2 = mt.downstream_head(sd, cfg, 2, d2, H, W)
    assert rel_err(f1, g["enc1"]) < 1e-5 and rel_err(d1[-1], g["dec1_last"]) < 1e-5 and rel_err(d2[6], g["dec2_mid"]) < 1e-5
    for k in KEYS:
        assert rel_err(o1[k], g["h1." + k]) < 3e-5, k
        assert rel_err(o2[k], g["h2." + k]) < 3e-5, k


def test_det_weights_are_order_independent():
    s = mt.param_shapes(mt.SMALL_CFG)
    a = synthetic.det_weights(s)
    b = synthetic.det_weights(dict(reversed(list(s.items()))))
    assert all(torch.equal(a[k], b[k]) for k in s) and len(s) > 400


def _run_cuda(cfg, H, W, dev, precision="bf16x3"):
    from artdeco_b200.mast3r import AsymmetricMASt3R
    sd = synthetic.det_weights(mt.param_shapes(cfg))
    m = AsymmetricMASt3R(precision=precision, **cfg)
    m.load_state_dict(sd)
    m.to(dev)
    img1, img2 = synthetic.mast3r_pair(1, H, W, seed=0)
    shape = torch.tensor([[H, W]])
    f1, p1, _ = m._encode_image(img1.to(dev), shape)
    f2, p2, _ = m._encode_image(img2.to(dev), shape)
    d1, d2 = m._decoder(f1, p1, f2, p2)
    r1 = m._downstream_head(1, [t.float() for t in d1], shape)
    r2 = m._downstream_head(2, [t.float() for t in d2], shape.to(dev))      # on-device shape as at utils_mast3r.py:177
    return m, sd, (f1, p1, d1, d2, r1, r2)


@pytest.mark.gpu
def test_cuda_model_matches_reference_golden_small(cuda):
    g = _gold("small")
    m, sd, (f1, p1, d1, d2, r1, r2) = _run_cuda(g["cfg"], g["H"], g["W"], cuda)
    assert len(d1) == 13 and d1[0].shape[-1] == g["cfg"]["enc_embed_dim"] and p1.dtype == torch.int64
    assert rel_err(f1, g["enc1"]) < 1e-4, "encoder tokens"
    assert rel_err(d1[-1], g["dec1_last"]) < 1e-4 and rel_err(d2[6], g["dec2_mid"]) < 1e-4, "decoder tokens"
    for k in KEYS:
        assert rel_err(r1[k], g["h1." + k]) < 1e-4, f"head1 {k}"
        assert rel_err(r2[k], g["h2." + k]) < 1e-4, f"head2 {k}"
    # forward(): the named surface (dust3r/model.py:199-211)
    img1, img2 = synthetic.mast3r_pair(1, g["H"], g["W"], seed=0)
    o1, o2 = m.forward({"img": img1.to(cuda)}, {"img": img2.to(cuda)})
    assert "pts3d_in_other_view" in o2 and "pts3d" not in o2
    assert rel_err(o1["pts3d"], g["h1.pts3d"]) < 1e-4 and rel_err(o2["pts3d_in_other_view"], g["h2.pts3d"]) < 1e-4


@pytest.mark.gpu
def test_cuda_model_matches_reference_golden_full(cuda):
    """ViT-L/ViT-B at 512x512 (the BASELINE configuration) against strided samples of the real reference's outputs."""
    g = _gold("full")
    s, ts = g["stride"], g["tok_stride"]
    m, sd, (f1, p1, d1, d2, r1, r2) = _run_cuda(g["cfg"], g["H"], g["W"], cuda)
    assert f1.shape == (1, 1024, 1024)
    assert _gold_err(f1[:, ::ts], g, "enc1") < 1e-4
    assert _gold_err(d1[-1][:, ::ts], g, "dec1_last") < 1e-4 and _gold_err(d2[6][:, ::ts], g, "dec2_mid") < 1e-4
    for k in KEYS:
        assert _gold_err(r1[k][:, ::s, ::s], g, "h1." + k) < 1e-4, f"head1 {k}"
        assert _gold_err(r2[k][:, ::s, ::s], g, "h2." + k) < 1e-4, f"head2 {k}"


@pytest.mark.gpu
def test_graphed_bench_batch_replay_matches_golden_and_eager(cuda):
    """The configuration bench.py times: GraphedForwardPair(model, BENCH_PAIRS_PER_GPU, 512, 512) on two streams, REPLAYED (the race fixed
    in round 1 only showed under replay).  Batch item 0 is the golden pair, so all four outputs of both views are checked
    against the real reference's outputs (mast3r_full.pt); every output of the graph must be bit-identical to the eager
    forward_pair on the same batch, on the first and on the second replay (utils_mast3r.py:30-36 is the eager call)."""
    from artdeco_b200.mast3r import BENCH_PAIRS_PER_GPU as B, AsymmetricMASt3R, GraphedForwardPair, forward_pair
    g = _gold("full")
    s, H, W = g["stride"], g["H"], g["W"]
    sd = synthetic.det_weights(mt.param_shapes(g["cfg"]))
    m = AsymmetricMASt3R(precision="bf16x3", **g["cfg"]).load_state_dict(sd).to(cuda)
    a1, a2 = synthetic.mast3r_pair(1, H, W, seed=0)
    r1, r2 = synthetic.mast3r_pair(B - 1, H, W, seed=21)
    i1, i2 = torch.cat((a1, r1)).to(cuda), torch.cat((a2, r2)).to(cuda)
    e1, e2 = forward_pair(m, i1, i2)
    e1 = {k: v.clone() for k, v in e1.items()}
    e2 = {k: v.clone() for k, v in e2.items()}
    graphed = GraphedForwardPair(m, B, H, W)
    for replay in range(2):
        if replay == 1:      # a different batch in between, so that replay 2 cannot pass on stale buffers
            graphed(i2, i1)
        o1, o2 = graphed(i1, i2)
        torch.cuda.synchronize()
        for k in KEYS:
            assert _gold_err(o1[k][:1, ::s, ::s], g, "h1." + k) < 1e-4, f"replay {replay} head1 {k} vs reference golden"
            assert _gold_err(o2[k][:1, ::s, ::s], g, "h2." + k) < 1e-4, f"replay {replay} head2 {k} vs reference golden"
            assert torch.equal(o1[k], e1[k]) and torch.equal(o2[k], e2[k]), f"replay {replay}: graph != eager ({k})"


@pytest.mark.gpu
def test_cuda_model_vs_oracle_odd_shape_and_batch(cuda):
    """512x384-style aspect (PINGPONG's real shape, scaled down) and batch 2, against the oracle run on the GPU in fp32."""
    cfg, H, W = mt.SMALL_CFG, 96, 128
    from artdeco_b200.mast3r import AsymmetricMASt3R
    sd = synthetic.det_weights(mt.param_shapes(cfg))
    m = AsymmetricMASt3R(**cfg).load_state_dict(sd).to(cuda)
    img1, img2 = synthetic.mast3r_pair(2, H, W, seed=3)
    sdg = {k: v.to(cuda) for k, v in sd.items()}
    prev = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.inference_mode():
            a1, a2 = mt.forward_pair(sdg, cfg, img1.to(cuda), img2.to(cuda))
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
    from artdeco_b200.mast3r import forward_pair
    b1, b2 = forward_pair(m, img1.to(cuda), img2.to(cuda))
    for k in KEYS:
        assert rel_err(b1[k], a1[k]) < 1e-4 and rel_err(b2[k], a2[k]) < 1e-4, k


@pytest.mark.gpu
def test_single_pass_bf16_is_outside_tolerance(cuda):
    """Documents why bf16x3 is the default: one bf16 pass misses the 1e-4 contract by two orders of magnitude."""
    g = _gold("small")
    _, _, (f1, *_rest) = _run_cuda(g["cfg"], g["H"], g["W"], cuda, precision="bf16")
    e = rel_err(f1, g["enc1"])
    assert 1e-4 < e < 0.2


@pytest.mark.gpu
def test_symmetric_batch_wrapper_matches_per_pair_loop(cuda):
    """utils_mast3r.py:42-71: the reference loops over pairs and runs decoder(i,j), decoder(j,i) per pair; the batched
    wrapper must return the same X/C/D/Q stacking (ii, ji, jj, ij) as that loop run with our own per-pair decoder."""
    from types import SimpleNamespace
    from artdeco_b200.mast3r import AsymmetricMASt3R, wrappers
    cfg, H, W = mt.SMALL_CFG, 64, 96
    m = AsymmetricMASt3R(**cfg).load_state_dict(synthetic.det_weights(mt.param_shapes(cfg))).to(cuda)
    img_i, img_j = synthetic.mast3r_pair(3, H, W, seed=5)
    fi, pi, _ = m._encode_image(img_i.to(cuda), None)
    fj, pj, _ = m._encode_image(img_j.to(cuda), None)
    shapes = torch.tensor([[H, W]] * 3)
    X, C, D, Q = wrappers.mast3r_decode_symmetric_batch(m, fi, pi, fj, pj, shapes, shapes)
    assert X.shape == (4, 3, H, W, 3) and C.shape == (4, 3, H, W) and D.shape == (4, 3, H, W, 24) and Q.shape == (4, 3, H, W)
    for b in range(3):
        r11, r21 = wrappers.decoder(m, fi[b:b + 1], fj[b:b + 1], pi[b:b + 1], pj[b:b + 1], shapes[b], shapes[b])
        r22, r12 = wrappers.decoder(m, fj[b:b + 1], fi[b:b + 1], pj[b:b + 1], pi[b:b + 1], shapes[b], shapes[b])
        for n, r in enumerate((r11, r21, r22, r12)):
            # same kernels, different batch size: tiling of the reductions is batch-independent -> tight agreement
            assert rel_err(X[n, b], r["pts3d"][0]) < 2e-6 and rel_err(D[n, b], r["desc"][0]) < 2e-6
            assert rel_err(C[n, b], r["conf"][0]) < 2e-6 and rel_err(Q[n, b], r["desc_conf"][0]) < 2e-6
    # asymmetric / mono wrappers: shapes and agreement with the oracle on the same weights
    fr_i, fr_j = SimpleNamespace(img=img_i[0].to(cuda)), SimpleNamespace(img=img_j[0].to(cuda))
    Xa, Ca, Da, Qa, f1, p1 = wrappers.mast3r_asymmetric_inference(m, fr_i, fr_j)
    assert Xa.shape == (2, H, W, 3) and Da.shape == (2, H, W, 24) and f1.shape[0] == 1
    assert rel_err(Xa[0], X[0, 0]) < 2e-6 and rel_err(Xa[1], X[1, 0]) < 2e-6
    # matching wrappers (utils_mast3r.py:74-112,144-171) chain the decode into artdeco_b200.matching
    cfgm = {"matching": dict(max_iter=10, lambda_init=1e-8, convergence_thresh=1e-6, dist_thresh=1e-1, radius=2, dilation_max=2)}
    out = wrappers.mast3r_match_symmetric(cfgm, m, fi, pi, fj, pj, shapes, shapes)
    assert len(out) == 8 and out[0].shape == (3, H * W) and out[2].shape == (3, H * W, 1) and out[4].shape == (3, H * W, 1)
    from artdeco_b200 import matching
    i2j, vj = matching.match(cfgm, torch.cat((X[0], X[2]), 0), torch.cat((X[1], X[3]), 0), torch.cat((D[0], D[2]), 0),
                             torch.cat((D[1], D[3]), 0))
    assert torch.equal(out[0], i2j[:3]) and torch.equal(out[1], i2j[3:]) and torch.equal(out[3], vj[3:])
    oa = wrappers.mast3r_match_asymmetric(cfgm, m, fr_i, fr_j)
    assert len(oa) == 10 and oa[0].shape == (1, H * W) and oa[2].shape == (H * W, 3) and oa[4].shape == (H * W, 1)
    Xii, Cii, feat, pos = wrappers.mast3r_inference_mono(m, fr_i)
    assert Xii.shape == (H * W, 3) and Cii.shape == (H * W, 1)
    sdg = {k: v.to(cuda) for k, v in synthetic.det_weights(mt.param_shapes(cfg)).items()}
    prev = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.inference_mode():
            a1, _ = mt.forward_pair(sdg, cfg, img_i[:1].to(cuda), img_i[:1].to(cuda))
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
    assert rel_err(Xii, a1["pts3d"][0].reshape(-1, 3)) < 1e-4


@pytest.mark.gpu
def test_curope_inplace_matches_pytorch_rope(cuda):
    """curope.rope_2d / cuRoPE2D (curope.cpp:49-68, curope2d.py:12-40) against the reference's PyTorch formulation
    (croco/models/pos_embed.py:112-159, restated in oracle/mast3r_torch.py:rope2d), incl. the inverse rotation."""
    from artdeco_b200.mast3r.curope import cuRoPE2D, rope_2d
    g = torch.Generator().manual_seed(0)
    for (B, Hh, N, D) in [(2, 12, 77, 64), (1, 3, 5, 32), (3, 16, 1024, 64)]:
        # [B,H,N,D] VIEW of a [B,N,H,D] buffer, as croco's attention produces it (blocks.py:98-103)
        tok = torch.randn(B, N, Hh, D, generator=g).transpose(1, 2)
        pos = torch.stack([torch.randint(0, 32, (B, N), generator=g), torch.randint(0, 48, (B, N), generator=g)], -1)
        ref = mt.rope2d(tok.double(), pos, base=100.0)
        t = tok.transpose(1, 2).contiguous().to(cuda).transpose(1, 2)
        out = cuRoPE2D(100.0)(t, pos.to(cuda))
        assert out.data_ptr() == t.data_ptr(), "in place"
        assert rel_err(out, ref) < 2e-6
        # F0 = -1 undoes it (the reference's backward, curope2d.py:25-29)
        bnhd = t.transpose(1, 2)
        rope_2d(bnhd, pos.to(cuda), 100.0, -1.0)
        assert rel_err(t, tok) < 2e-6
    with pytest.raises(ValueError):
        rope_2d(torch.zeros(1, 4, 2, 6, device=cuda), torch.zeros(1, 4, 2, dtype=torch.int64, device=cuda), 100.0, 1.0)
    with pytest.raises(ValueError):
        rope_2d(torch.zeros(1, 2, 4, 8, device=cuda).transpose(1, 2), torch.zeros(1, 4, 2, dtype=torch.int64, device=cuda), 100.0, 1.0)
