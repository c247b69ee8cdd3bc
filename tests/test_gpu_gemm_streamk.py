"""GPU: the DMMA GEMM (csrc/gpk_gemm.cu) against a plain FP64 torch product of the same operands, on shapes from one partial
wave of 64 x 64 tiles to several (the shapes a stream-K tail would have split; that path was measured slower and removed,
DESIGN.md 7a); every call is one launch of the one-tile-per-CTA kernel."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _handle():
    import torch
    from gp_algos_b200 import _lib
    ts = torch.cuda.Stream(priority=-1)
    torch.cuda.set_stream(ts)
    return _lib.Handle(0, ts.cuda_stream), ts


@pytest.mark.parametrize("n,k", [(4096, 1024), (4096, 272), (3200, 640), (1920, 4096)])
def test_syrk_lower_matches_torch(n, k):
    import torch
    h, ts = _handle()
    g = torch.Generator(device="cuda").manual_seed(n + k)
    P = torch.randn(k, n, dtype=torch.float64, device="cuda", generator=g)       # n x k column-major
    C0 = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g)
    C = C0.clone()
    l0 = h.launch_count()
    h.check(h.lib.gpk_syrk_lower_dev(h.h, P.data_ptr(), n, C.data_ptr(), n, n, k))
    h.synchronize()
    assert h.launch_count() - l0 == 1
    ref = C0 - P.T @ P                                                             # C is stored transposed; the product is symmetric
    got, want = C.cpu().numpy(), ref.cpu().numpy()
    c0 = C0.cpu().numpy()
    scale = np.abs(want).max()
    for bt in range(n // 64):                                                     # only lower 64-tiles (column-major) are written
        rows = slice(bt * 64, n)
        blk_got = got[bt * 64:(bt + 1) * 64, rows]                                 # got[c, r]: column block bt, rows >= its start
        assert np.allclose(blk_got, want[bt * 64:(bt + 1) * 64, rows], rtol=0, atol=1e-12 * scale)
        assert np.array_equal(got[bt * 64:(bt + 1) * 64, :bt * 64], c0[bt * 64:(bt + 1) * 64, :bt * 64])   # strictly upper tiles untouched
    torch.cuda.set_stream(torch.cuda.default_stream())


@pytest.mark.parametrize("m,p,k,beta", [(2048, 1024, 512, 1.0), (4096, 512, 256, 0.0), (8192, 256, 1024, -0.5)])
def test_gemm_nt_stream_k_matches_torch(m, p, k, beta):
    import torch
    h, ts = _handle()
    g = torch.Generator(device="cuda").manual_seed(m + p + k)
    Pm = torch.randn(k, m, dtype=torch.float64, device="cuda", generator=g)        # m x k column-major
    Qm = torch.randn(k, p, dtype=torch.float64, device="cuda", generator=g)        # p x k column-major
    C0 = torch.randn(p, m, dtype=torch.float64, device="cuda", generator=g)        # m x p column-major
    C = C0.clone()
    l0 = h.launch_count()
    h.check(h.lib.gpk_gemm_nt_dev(h.h, m, p, k, 1.5, Pm.data_ptr(), m, Qm.data_ptr(), p, beta, C.data_ptr(), m, 0))
    h.synchronize()
    assert h.launch_count() - l0 == 1
    ref = 1.5 * (Qm.T @ Pm) + beta * C0                                            # [c, i] layout of the column-major C
    assert torch.allclose(C, ref, rtol=0, atol=1e-12 * float(ref.abs().max()))
    torch.cuda.set_stream(torch.cuda.default_stream())
