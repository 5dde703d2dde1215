"""Runs the reference's own CUDA extensions (built into oracle/_ref by oracle/build_ref.py) on the inputs of the tests that
compare against them, and writes seeded samples of their outputs to tests/golden/reference_builds.npz.  Needs a GPU and
oracle/_ref: ``python tests/golden/make_reference_builds_golden.py [OUT.npz]`` from the repo root.  The tests regenerate
the same inputs from the same seeds, so only outputs are stored."""
import pathlib
import sys

import numpy as np
import torch

ROOT = pathlib.Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from artdeco_b200 import synthetic  # noqa: E402
from artdeco_b200.matching import prep_for_iter_proj  # noqa: E402
from helpers import golden_sample as sample_idx  # noqa: E402
from oracle import build_ref  # noqa: E402
from test_matching import CFG, _pixel_grid, _scene  # noqa: E402

C1, C2 = 0.01 ** 2, 0.03 ** 2
N_SAMPLE = 4096          # elements kept per dense output
N_ROWS = 1024            # rows kept per [P, K] distance table
N_POINTS = 8192          # match positions kept


def _np(t):
    return t.detach().float().cpu().numpy().reshape(-1)


def ssim(out, dev):
    ref = build_ref.load("fused_ssim_ref")
    # test_ssim.py::test_matches_the_reference_cuda_build
    g = torch.Generator().manual_seed(3)
    a, b = torch.rand(2, 3, 270, 480, generator=g).to(dev), torch.rand(2, 3, 270, 480, generator=g).to(dev)
    m, d1, d2, d3 = ref.fusedssim(C1, C2, a, b, True)
    up = torch.rand(2, 3, 270, 480, generator=g).to(dev)
    grad = ref.fusedssim_backward(C1, C2, a, b, up, d1, d2, d3)
    i = sample_idx(m.numel(), N_SAMPLE, 0)
    out.update(ssim_map=_np(m)[i], ssim_dm_dmu1=_np(d1)[i], ssim_grad=_np(grad)[i])
    # test_ssim.py::test_ssim_full_size_matches_oracle_and_reference_build
    for tag, shape in (("baseline_1x3x1080p", (1, 3, 1080, 1920)), ("reference_test_5x5x1080p", (5, 5, 1080, 1920))):
        g = torch.Generator().manual_seed(5)
        a = torch.rand(*shape, generator=g).to(dev)
        b = torch.rand(*shape, generator=g).to(dev)
        m, d1, d2, d3 = ref.fusedssim(C1, C2, a, b, True)
        up = torch.rand(*shape, generator=g).to(dev)
        grad = ref.fusedssim_backward(C1, C2, a, b, up, d1, d2, d3)
        i = sample_idx(m.numel(), N_SAMPLE, 0)
        out[f"ssim_full_{tag}_map"] = _np(m)[i]
        out[f"ssim_full_{tag}_grad"] = _np(grad)[i]


def knn(out, dev):
    # test_adam_cull_knn.py::test_distcuda2_bit_identical_to_the_reference_build
    ref = build_ref.load("simple_knn_ref")
    for P in (5000, 200_000):
        pts = synthetic.raster_scene(P, seed=2)["means"].to(dev)
        i = sample_idx(P, N_SAMPLE, 0)
        out[f"knn_{P}_distcuda2"] = _np(ref.distCUDA2(pts))[i]
        dr, _ = ref.distIndex2(pts, 6)
        rows = sample_idx(P, N_ROWS, 1)
        out[f"knn_{P}_distindex2_sorted"] = dr.view(P, 6).sort(dim=1).values.cpu().numpy()[rows]


def matching(out, dev):
    # test_matching.py::test_matches_the_reference_cuda_build
    ref = build_ref.load("mast3r_matching_ref")
    X11, X21, D11, D21 = [t.to(dev).contiguous() for t in _scene(b=2, h=192, w=256, seed=4)]
    c = CFG["matching"]
    rays, pts, p_init = prep_for_iter_proj(X11, X21, None)
    p_r, conv_r = ref.iter_proj(rays, pts, p_init, c["max_iter"], c["lambda_init"], c["convergence_thresh"])
    i = sample_idx(conv_r.numel(), N_POINTS, 0)
    out["match_iter_proj_p"] = p_r.reshape(-1, 2).cpu().numpy()[i]
    out["match_iter_proj_converged"] = np.packbits(conv_r.reshape(-1).cpu().numpy())
    p1 = p_r.long()
    a, q = D11.half().contiguous(), D21.reshape(2, -1, 24).half().contiguous()
    (theirs,) = ref.refine_matches(a, q, p1, c["radius"], c["dilation_max"])
    # refine_matches is compared bit for bit on the reference's own integer positions, so those are stored whole, as small
    # offsets: p1 from each point's own pixel, the refined position from p1
    d_p1 = (p1.cpu() - _pixel_grid(192, 256)).numpy()
    d_out = (theirs - p1).cpu().numpy()
    assert max(np.abs(d_p1).max(), np.abs(d_out).max()) < 128
    out["match_refine_p1_offset"] = d_p1.astype(np.int8)
    out["match_refine_out_offset"] = d_out.astype(np.int8)


if __name__ == "__main__":
    dest = pathlib.Path(sys.argv[1]) if len(sys.argv) > 1 else pathlib.Path(__file__).parent / "reference_builds.npz"
    dev = torch.device("cuda:0")
    out = {}
    ssim(out, dev)
    knn(out, dev)
    matching(out, dev)
    torch.cuda.synchronize()
    dest.parent.mkdir(parents=True, exist_ok=True)
    np.savez_compressed(dest, **out)
    print(f"wrote {dest} ({dest.stat().st_size} bytes):", {k: (v.shape, str(v.dtype)) for k, v in out.items()})
