"""The TMA-fed 3xTF32 tcgen05 GEMMs (csrc/gemm_tma.cu) against fp64 matmul: fp32-equivalent accuracy
(1e-5 normwise would already fail a single-pass tf32 product, whose error is ~5e-4)."""
import pytest
import torch

from parity_util import relerr

pytestmark = pytest.mark.gpu


def _st():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("M,N,K,pad", [(128, 128, 32, 0), (300, 256, 128, 0), (1000, 64, 256, 8), (640, 512, 64, 4), (129, 16, 96, 0),
                                       (4096, 128, 136, 0), (50000, 128, 128, 0), (20011, 64, 64, 0), (30000, 256, 256, 0),
                                       (77, 512, 64, 4), (1, 128, 128, 0)])
def test_gemm_nt_tma(M, N, K, pad):
    """resident weights (N, K <= 128), streamed weights, ragged M / N / K tails, many tiles per CTA (stage-ring wrap),
    fewer rows than one 128-row tile (TMA zero-fills the rest; nothing is stored past M)."""
    from regt_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(M + N + K)
    A = (torch.rand(M, K + pad, generator=g) - 0.5).cuda()
    Bt = (torch.rand(N, K + pad, generator=g) - 0.5).cuda()
    C = torch.full((M, N + pad), float("nan"), device="cuda")
    scratch = torch.empty(2 * ((N + 127) // 128 * 128) * ((K + 31) // 32 * 32), device="cuda")
    rc = lib.regt_debug_gemm_nt_tma(A.data_ptr(), K + pad, Bt.data_ptr(), K + pad, C.data_ptr(), N + pad, M, N, K,
                                    scratch.data_ptr(), _st())
    _lib.check(rc, "regt_debug_gemm_nt_tma")
    ref = A[:, :K].double() @ Bt[:, :K].double().t()
    assert relerr(C[:, :N], ref) <= 1e-5
    if pad:
        assert torch.isnan(C[:, N:]).all()


@pytest.mark.parametrize("M,K,N,splits", [(256, 128, 128, 1), (1000, 256, 64, 4), (5000, 512, 128, 7), (70, 64, 32, 3),
                                          (4097, 128, 288, 5), (777, 64, 0, 2), (40000, 128, 128, 37), (1000, 256, 128, 4),
                                          (3000, 128, 256, 3), (20, 64, 32, 1)])
def test_gemm_tn_tma(M, K, N, splits):
    """the row contraction against B and, in the same pass over A, the 32-column plane B2 (the F-wide weight gradients);
    M < 32 is one zero-filled 32-row box."""
    from regt_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(M + N + K)
    A = (torch.rand(M, K + 4, generator=g) - 0.5).cuda()
    B = (torch.rand(M, max(N, 4) + 8, generator=g) - 0.5).cuda()
    B2 = (torch.rand(M, 32, generator=g) - 0.5).cuda()
    Cp = torch.full((splits, K, max(N, 1)), float("nan"), device="cuda")
    Cp2 = torch.full((splits, K, 32), float("nan"), device="cuda")
    rc = lib.regt_debug_gemm_tn_tma(A.data_ptr(), K + 4, B.data_ptr() if N else None, max(N, 4) + 8, Cp.data_ptr() if N else None, M, K, N,
                                    splits, B2.data_ptr(), 32, Cp2.data_ptr(), _st())
    _lib.check(rc, "regt_debug_gemm_tn_tma")
    if N:
        assert relerr(Cp.double().sum(0), A[:, :K].double().t() @ B[:, :N].double()) <= 1e-5
    assert relerr(Cp2.double().sum(0), A[:, :K].double().t() @ B2.double()) <= 1e-5


@pytest.mark.parametrize("M,H,splits", [(3000, 128, 5), (20000, 256, 10), (40000, 128, 37), (20, 128, 1)])
def test_gemm_tn_multi_segment(M, H, splits):
    """the cell backward's single launch: D [M, 4H] against h (z | r blocks), h*R (h~ block) and the feature plane (all blocks)."""
    from regt_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(M + H)
    D = (torch.rand(M, 4 * H, generator=g) - 0.5).cuda()
    h = (torch.rand(M, H, generator=g) - 0.5).cuda()
    hR = (torch.rand(M, H, generator=g) - 0.5).cuda()
    F = (torch.rand(M, 32, generator=g) - 0.5).cuda()
    C0 = torch.full((splits, 2 * H, H), float("nan"), device="cuda")
    C1 = torch.full((splits, H, H), float("nan"), device="cuda")
    C2 = torch.full((splits, 4 * H, 32), float("nan"), device="cuda")
    rc = lib.regt_debug_gemm_tn_multi(D.data_ptr(), 4 * H, M, H, h.data_ptr(), hR.data_ptr(), C0.data_ptr(), C1.data_ptr(), splits,
                                      F.data_ptr(), C2.data_ptr(), _st())
    _lib.check(rc, "regt_debug_gemm_tn_multi")
    Dd = D.double()
    assert relerr(C0.double().sum(0), Dd[:, :2 * H].t() @ h.double()) <= 1e-5
    assert relerr(C1.double().sum(0), Dd[:, 2 * H:3 * H].t() @ hR.double()) <= 1e-5
    assert relerr(C2.double().sum(0), Dd.t() @ F.double()) <= 1e-5


@pytest.mark.parametrize("M,K,N,splits", [(5000, 512, 128, 1), (5000, 512, 128, 3), (20000, 1024, 256, 10)])
def test_gemm_tn_tma_stage_reuse_stress(M, K, N, splits):
    """regression: the raw TMA stage must not be released before the converters' shared-memory loads have returned
    (an mbarrier arrive does not wait for earlier loads: the tail loads of a warp once read the next chunk's bytes,
    a few times per hundred launches).  Many chunks per CTA, repeated launches, exact per-split check."""
    from regt_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(1)
    A = (torch.rand(M, K, generator=g) - 0.5).cuda()
    B = (torch.rand(M, N, generator=g) - 0.5).cuda()
    B2 = (torch.rand(M, 32, generator=g) - 0.5).cuda()
    ref = A.double().t() @ B.double()
    ref2 = A.double().t() @ B2.double()
    for _ in range(8):
        Cp = torch.full((splits, K, N), float("nan"), device="cuda")
        Cp2 = torch.full((splits, K, 32), float("nan"), device="cuda")
        rc = lib.regt_debug_gemm_tn_tma(A.data_ptr(), K, B.data_ptr(), N, Cp.data_ptr(), M, K, N, splits, B2.data_ptr(), 32, Cp2.data_ptr(), _st())
        _lib.check(rc, "regt_debug_gemm_tn_tma")
        assert float((Cp.double().sum(0) - ref).abs().max()) <= 1e-5 * float(ref.abs().max())
        assert float((Cp2.double().sum(0) - ref2).abs().max()) <= 1e-5 * float(ref2.abs().max())


@pytest.mark.parametrize("H,ntile,splits", [(128, 5, 1), (128, 37, 4), (64, 9, 2), (128, 300, 37)])
def test_gemm_kt_transposed_tiles(H, ntile, splits):
    """the row contraction of the fused cell backward over transposed tiles (csrc/gemm_tma.cu k_gemm_kt): D^T [tile][4 row
    quarters][4H][32], h^T / (h*R)^T [tile][4][H][32], F^T [tile][4][32][32] -> dB_z|dB_r = [Dz|Dr]^T h, dB_h = Dc^T hR, D^T F."""
    from regt_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(H + ntile)
    AT = (torch.rand(ntile * 4, 4 * H, 32, generator=g) - 0.5).cuda()
    B0T = (torch.rand(ntile * 4, H, 32, generator=g) - 0.5).cuda()
    B1T = (torch.rand(ntile * 4, H, 32, generator=g) - 0.5).cuda()
    FT = (torch.rand(ntile * 4, 32, 32, generator=g) - 0.5).cuda()
    C0 = torch.full((splits, 2 * H, H), float("nan"), device="cuda")
    C1 = torch.full((splits, H, H), float("nan"), device="cuda")
    C2 = torch.full((splits, 4 * H, 32), float("nan"), device="cuda")
    rc = lib.regt_debug_gemm_kt(AT.data_ptr(), ntile, H, B0T.data_ptr(), B1T.data_ptr(), FT.data_ptr(), C0.data_ptr(), C1.data_ptr(),
                                C2.data_ptr(), splits, _st())
    _lib.check(rc, "regt_debug_gemm_kt")
    torch.cuda.synchronize()
    A, B0, B1, Fm = AT.double(), B0T.double(), B1T.double(), FT.double()
    ref0 = torch.einsum("tkr,tnr->kn", A[:, :2 * H], B0)
    ref1 = torch.einsum("tkr,tnr->kn", A[:, 2 * H:3 * H], B1)
    ref2 = torch.einsum("tkr,tnr->kn", A, Fm)
    assert relerr(C0.double().sum(0), ref0) <= 1e-5
    assert relerr(C1.double().sum(0), ref1) <= 1e-5
    assert relerr(C2.double().sum(0), ref2) <= 1e-5
