"""fused-SSIM: CPU checks of the oracle, GPU parity of the CUDA kernels (through the C ABI) against it.
Tolerance: the reference's own test (fused-ssim/tests/test.py:82-91) uses torch.isclose defaults (rtol 1e-5) on the
scalar and on the gradient; we assert rtol 1e-5 on the scalar and 1e-4-of-scale on maps and gradients."""
import pytest
import torch

from oracle import ssim_ref
from helpers import assert_close, golden_sample, reference_builds


def test_oracle_window_matches_reference_constants():
    # cGauss in the reference kernel (ssim.cu:12-24) is this window
    w = ssim_ref.gaussian(11, 1.5)
    ref = torch.tensor([0.001028380123898387, 0.0075987582094967365, 0.036000773310661316, 0.10936068743467331,
                        0.21300552785396576, 0.26601171493530273, 0.21300552785396576, 0.10936068743467331,
                        0.036000773310661316, 0.0075987582094967365, 0.001028380123898387])
    assert torch.allclose(w, ref, rtol=1e-6, atol=0)


def test_oracle_identity_is_one():
    x = torch.rand(1, 3, 40, 50)
    assert abs(float(ssim_ref.ssim(x, x)) - 1.0) < 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 3, 64, 64), (2, 3, 97, 131), (1, 1, 7, 5), (5, 5, 135, 240), (1, 3, 486, 648)])
@pytest.mark.parametrize("padding", ["same", "valid"])
def test_fused_ssim_matches_oracle(cuda, shape, padding):
    from artdeco_b200.ssim import fused_ssim
    if padding == "valid" and min(shape[2:]) <= 10:
        pytest.skip("valid padding needs > 10 px")
    g = torch.Generator().manual_seed(0)
    a = torch.rand(*shape, generator=g)
    b = torch.rand(*shape, generator=g)
    a_ref = a.clone().double().requires_grad_(True)
    ref = ssim_ref.ssim(a_ref, b.double(), padding)
    ref.backward()
    a_gpu = a.to(cuda).requires_grad_(True)
    out = fused_ssim(a_gpu, b.to(cuda), padding=padding)
    out.backward()
    # rtol 1e-5 as in the reference test, plus an fp32 floor: the map has O(1) entries of both signs, so for random
    # images the mean is ~1e-4 and an fp32 sum cannot resolve it to 1e-5 relative (observed |err| ~2e-8).
    assert abs(float(out.detach()) - float(ref.detach())) <= 1e-5 * abs(float(ref.detach())) + 2e-7
    assert_close(a_gpu.grad, a_ref.grad, what="dL/dimg1")


@pytest.mark.gpu
def test_fusedssim_map_and_derivative_surface(cuda):
    """ext-level surface (ext.cpp:4-7): map + 3 derivative maps, train=False returns empty derivative tensors."""
    from artdeco_b200.ssim import fusedssim, fusedssim_backward
    g = torch.Generator().manual_seed(1)
    a, b = torch.rand(2, 3, 50, 70, generator=g), torch.rand(2, 3, 50, 70, generator=g)
    m, d1, d2, d3 = fusedssim(0.01 ** 2, 0.03 ** 2, a.to(cuda), b.to(cuda), True)
    assert_close(m, ssim_ref.ssim_map(a.double(), b.double()), what="ssim map")
    m2, e1, e2, e3 = fusedssim(0.01 ** 2, 0.03 ** 2, a.to(cuda), b.to(cuda), False)
    assert e1.numel() == e2.numel() == e3.numel() == 0 and torch.equal(m, m2)
    up = torch.rand(2, 3, 50, 70, generator=g)
    grad = fusedssim_backward(0.01 ** 2, 0.03 ** 2, a.to(cuda), b.to(cuda), up.to(cuda), d1, d2, d3)
    a_ref = a.double().requires_grad_(True)
    (ssim_ref.ssim_map(a_ref, b.double()) * up.double()).sum().backward()
    assert_close(grad, a_ref.grad, what="fusedssim_backward")


@pytest.mark.gpu
def test_ssim_1080p_properties(cuda):
    """Full BASELINE size [1,3,1080,1920]: identical images -> 1, symmetric in its arguments, and the fused-mean
    path equals the map path."""
    from artdeco_b200.ssim import fused_ssim, fusedssim
    g = torch.Generator().manual_seed(2)
    a = torch.rand(1, 3, 1080, 1920, generator=g).to(cuda)
    b = torch.rand(1, 3, 1080, 1920, generator=g).to(cuda)
    assert abs(float(fused_ssim(a, a, train=False)) - 1.0) < 1e-5
    ab, ba = float(fused_ssim(a, b, train=False)), float(fused_ssim(b, a, train=False))
    assert abs(ab - ba) <= 1e-6 * abs(ab)
    m, _, _, _ = fusedssim(0.01 ** 2, 0.03 ** 2, a, b, False)
    assert abs(float(m.double().mean()) - ab) <= 1e-5 * abs(ab)


@pytest.mark.gpu
def test_ssim_rejects_cpu_tensors(cuda):
    from artdeco_b200 import _lib
    from artdeco_b200.ssim import fused_ssim
    with pytest.raises(_lib.ArtdecoB200Error):
        fused_ssim(torch.rand(1, 3, 16, 16), torch.rand(1, 3, 16, 16))


def _sampled(t, n):
    return t.detach().reshape(-1)[torch.from_numpy(golden_sample(t.numel(), n)).to(t.device)].cpu()


@pytest.mark.gpu
def test_matches_the_reference_cuda_build(cuda):
    """Against the reference's OWN ssim.cu compiled for sm_100 (--use_fast_math, as its setup.py does): a seeded sample of
    its outputs on these inputs is stored in tests/golden/reference_builds.npz."""
    from artdeco_b200.ssim import fusedssim, fusedssim_backward
    gold = reference_builds()
    n = len(gold["ssim_map"])
    g = torch.Generator().manual_seed(3)
    a, b = torch.rand(2, 3, 270, 480, generator=g).to(cuda), torch.rand(2, 3, 270, 480, generator=g).to(cuda)
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    mo, o1, o2, o3 = fusedssim(C1, C2, a, b, True)
    assert_close(_sampled(mo, n), gold["ssim_map"], rtol=1e-5, what="ssim map vs reference build")
    assert_close(_sampled(o1, n), gold["ssim_dm_dmu1"], rtol=1e-5, what="dm_dmu1")
    up = torch.rand(2, 3, 270, 480, generator=g).to(cuda)
    assert_close(_sampled(fusedssim_backward(C1, C2, a, b, up, o1, o2, o3), n), gold["ssim_grad"],
                 rtol=1e-5, what="dL/dimg1 vs reference build")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 3, 1080, 1920), (5, 5, 1080, 1920)], ids=["baseline_1x3x1080p", "reference_test_5x5x1080p"])
def test_ssim_full_size_matches_oracle_and_reference_build(cuda, shape):
    """Full-size check as in the reference's own test (fused-ssim/tests/test.py:57-91: B=5, CH=5, 1080x1920) and at the
    BASELINE shape [1,3,1080,1920]: scalar and gradient against the conv2d formulation (the oracle; fp64 on the GPU so
    it takes milliseconds), and map / gradient against stored samples of the reference's own ssim.cu on these inputs."""
    from artdeco_b200.ssim import fused_ssim, fusedssim, fusedssim_backward
    gold = reference_builds()
    tag = {(1, 3, 1080, 1920): "baseline_1x3x1080p", (5, 5, 1080, 1920): "reference_test_5x5x1080p"}[shape]
    gmap, ggrad = gold[f"ssim_full_{tag}_map"], gold[f"ssim_full_{tag}_grad"]
    g = torch.Generator().manual_seed(5)
    a = torch.rand(*shape, generator=g).to(cuda)
    b = torch.rand(*shape, generator=g).to(cuda)
    a_ref = a.double().requires_grad_(True)
    ref = ssim_ref.ssim(a_ref, b.double())
    ref.backward()
    a_gpu = a.clone().requires_grad_(True)
    out = fused_ssim(a_gpu, b)
    out.backward()
    assert abs(float(out.detach()) - float(ref.detach())) <= 1e-5 * abs(float(ref.detach())) + 2e-7
    assert_close(a_gpu.grad, a_ref.grad, what="dL/dimg1 (full size)")
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    mo, o1, o2, o3 = fusedssim(C1, C2, a, b, True)
    assert_close(_sampled(mo, len(gmap)), gmap, rtol=1e-5, what="ssim map vs reference build (full size)")
    up = torch.rand(*shape, generator=g).to(cuda)
    assert_close(_sampled(fusedssim_backward(C1, C2, a, b, up, o1, o2, o3), len(ggrad)), ggrad,
                 rtol=1e-5, what="dL/dimg1 vs reference build (full size)")
