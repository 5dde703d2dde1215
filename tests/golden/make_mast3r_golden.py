"""Runs the REAL reference MASt3R (imported from /root/reference, CPU fp32) on deterministic weights and writes
tests/golden/mast3r_small.pt; also checks oracle/mast3r_torch.py against it.  Run from the repo root in the build
container (the GPU box has no /root/reference): ``python tests/golden/make_mast3r_golden.py [--full]``."""
import pathlib
import sys
import time

import torch

ROOT = pathlib.Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, "/root/reference/VSLAM/thirdparty/mast3r")
import mast3r.utils.path_to_dust3r  # noqa: E402,F401
from mast3r.model import AsymmetricMASt3R  # noqa: E402

from artdeco_b200 import synthetic  # noqa: E402
from oracle import mast3r_torch as mt  # noqa: E402

inf = float("inf")


def build_ref(cfg, img):
    return AsymmetricMASt3R(pos_embed="RoPE100", patch_embed_cls="PatchEmbedDust3R", img_size=img, head_type="catmlp+dpt",
                            output_mode="pts3d+desc24", depth_mode=("exp", -inf, inf), conf_mode=("exp", 1, inf),
                            two_confs=True, desc_conf_mode=("exp", 0, inf), landscape_only=False, **cfg).eval()


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-20))


@torch.inference_mode()
def run(cfg, H, W, tag, stride, tok_stride, scale_stride):
    model = build_ref(cfg, (H, W))
    sd = synthetic.det_weights(mt.param_shapes(cfg))
    missing = model.load_state_dict(sd, strict=False)
    unexpected = [k for k in missing.unexpected_keys]
    assert not unexpected, unexpected
    # parameters of the reference that inference never reads (mask_token, refinenet4.resConfUnit1, aliases)
    not_set = [k for k in missing.missing_keys if "layer_rn" not in k and "mask_token" not in k and "refinenet4.resConfUnit1" not in k]
    assert not not_set, not_set
    img1, img2 = synthetic.mast3r_pair(1, H, W, seed=0)
    shape = torch.tensor([[H, W]])
    t0 = time.time()
    f1, p1, _ = model._encode_image(img1, shape)
    f2, p2, _ = model._encode_image(img2, shape)
    d1, d2 = model._decoder(f1, p1, f2, p2)
    d1, d2 = list(d1), list(d2)
    r1 = model._downstream_head(1, [t.float() for t in d1], shape)
    r2 = model._downstream_head(2, [t.float() for t in d2], shape)
    print(f"[{tag}] reference forward {time.time() - t0:.1f}s")
    # the oracle restatement must agree with the real thing
    of1, op1 = mt.encode_image(sd, cfg, img1)
    of2, op2 = mt.encode_image(sd, cfg, img2)
    od1, od2 = mt.decoder(sd, cfg, of1, op1, of2, op2)
    o1 = mt.downstream_head(sd, cfg, 1, od1, H, W)
    o2 = mt.downstream_head(sd, cfg, 2, od2, H, W)
    errs = {"enc": rel(of1, f1), "pos": float((op1 != p1).sum()), "dec_last": rel(od1[-1], d1[-1]), "dec2_mid": rel(od2[6], d2[6])}
    for k in ("pts3d", "conf", "desc", "desc_conf"):
        errs["h1." + k] = rel(o1[k], r1[k]); errs["h2." + k] = rel(o2[k], r2[k])
    print(f"[{tag}] oracle vs reference:", {k: f"{v:.2e}" for k, v in errs.items()})
    assert max(errs.values()) < 2e-5, errs
    s, ts, c = stride, tok_stride, scale_stride
    gold = dict(cfg=cfg, H=H, W=W, stride=s, tok_stride=ts, enc1=f1[:, ::ts].clone(), dec1_last=d1[-1][:, ::ts].clone(),
                dec2_mid=d2[6][:, ::ts].clone(),
                enc_absmax=float(f1.abs().max()), dec_absmax=float(d1[-1].abs().max()))
    # each tensor's scale (max |x|) over a grid denser than the stored one: the tests' tolerance is relative to it
    gold.update({"enc1.scale": float(f1[:, ::c].abs().max()), "dec1_last.scale": float(d1[-1][:, ::c].abs().max()),
                 "dec2_mid.scale": float(d2[6][:, ::c].abs().max())})
    for k in ("pts3d", "conf", "desc", "desc_conf"):
        gold["h1." + k] = r1[k][:, ::s, ::s].clone(); gold["h2." + k] = r2[k][:, ::s, ::s].clone()
        gold["h1." + k + ".absmax"] = float(r1[k].abs().max())
        gold["h1." + k + ".scale"] = float(r1[k][:, ::c, ::c].abs().max())
        gold["h2." + k + ".scale"] = float(r2[k][:, ::c, ::c].abs().max())
    torch.save(gold, pathlib.Path(__file__).parent / f"mast3r_{tag}.pt")
    print(f"[{tag}] wrote golden; |pts3d|max={gold['h1.pts3d.absmax']:.3f} conf max={float(r1['conf'].max()):.3f}")


if __name__ == "__main__":
    run(mt.SMALL_CFG, 64, 48, "small", 1, 1, 1)
    if "--full" in sys.argv:
        # every 64th token and every 16th pixel keep the file under 1 MB; scales over every 8th
        run(mt.FULL_CFG, 512, 512, "full", 16, 64, 8)
