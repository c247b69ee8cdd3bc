"""GPU: the DMMA GEMM (csrc/gpk_gemm.cu) kernel by kernel.

`gpk_debug_gemm` issues one GEMM with a descriptor given field by field, so every operand layout, k-range flag, output
selection and Cin mode is reached directly rather than through the factorisations that use it:

- exact-result matrix: integer operands in [-8, 8] and alpha, beta in {1, -1, 0.5, 0, 2} make every partial sum exact in
  FP64, so D must equal the NumPy product exactly, whatever the summation order.  Operand regions that the k-range flags
  exclude beyond the diagonal 64-tile hold NaN (proving they are never read), the triangle inside the diagonal tile holds
  real zeros, padding and batch gaps of the operands hold NaN, and every element of D outside the written tiles must keep
  its sentinel;
- rounding-level check on N(0,1) operands of large shapes against the FP64 host product;
- argument validation (GPK_EINVAL without a launch);
- the public wrappers gpk_syrk_lower_dev and gpk_gemm_nt_dev at their documented contract.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
TRI_OUT, KB_R, KB_S, KE_R, KE_S, HEAVY_LAST = 1, 2, 4, 8, 16, 32
SENT = -777.25                      # sentinel for D elements the kernel must not write
NAN = float("nan")


@pytest.fixture(scope="module")
def h():
    from gp_algos_b200 import _lib
    hd = _lib.Handle(0)
    yield hd
    hd.close()


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _run(h, fn):
    """Enqueue `fn` on the handle's stream after every pending torch upload; return (status, launches issued)."""
    import torch
    torch.cuda.synchronize()
    l0 = h.launch_count()
    rc = fn()
    h.synchronize()
    return rc, h.launch_count() - l0


# ------------------------------------------------------------------------------------------------------------------------
# operands and the reference
# ------------------------------------------------------------------------------------------------------------------------
def _operand(rng, rows, K, kcontig, ld_extra, batch, gap, lo, hi, normal=False):
    """Batched operand X(x, k), x < rows, k < K, stored k-contiguous (X[k + x*ld]) or x-contiguous (X[x + k*ld]).
    lo (kb_* flag): X(x, k) is never read for k below the diagonal 64-tile of x, and is zero inside that tile for k < x.
    hi (ke_* flag): never read for k beyond the diagonal tile, zero inside it for k > x.
    Returns (flat buffer with NaN wherever the kernel must not read, ld, batch stride, logical values with the unread
    region as 0)."""
    ld = max((K if kcontig else rows) + ld_extra, 2)
    nstore = rows if kcontig else K
    stride = nstore * ld + gap
    buf = np.full(batch * stride + gap + 2, NAN)
    x = np.arange(rows)[:, None]
    k = np.arange(K)[None, :]
    t0 = (x // 64) * 64
    readable = np.ones((rows, K), dtype=bool)
    zero = np.zeros((rows, K), dtype=bool)
    if lo:
        readable &= k >= t0
        zero |= k < x
    if hi:
        readable &= k < t0 + 64
        zero |= k > x
    vals = np.empty((batch, rows, K))
    for b in range(batch):
        v = rng.standard_normal((rows, K)) if normal else rng.integers(-8, 9, size=(rows, K)).astype(np.float64)
        v[zero] = 0.0
        vals[b] = np.where(readable, v, 0.0)
        stored = np.where(readable, v, NAN)
        mat = buf[b * stride:b * stride + nstore * ld].reshape(nstore, ld)
        if kcontig:
            mat[:, :K] = stored
        else:
            mat[:, :rows] = stored.T
    return buf, ld, stride, vals


def _tile_mask(R, S, tri_out):
    r = (np.arange(R)[:, None] // 64) * 64
    s = (np.arange(S)[None, :] // 64) * 64
    return (s >= r) if tri_out else np.ones((R, S), dtype=bool)


def _regions(buf, batch, stride, rows, ld, cols):
    return [buf[b * stride:b * stride + rows * ld].reshape(rows, ld)[:, :cols] for b in range(batch)]


def _gemm_case(h, rng, R, S, K, batch, alpha, beta, pk, qk, flags, cin, ld_extra, normal=False):
    """Runs one gpk_debug_gemm; returns (status, launches, D buffer after, expected D buffer, |alpha||P||Q|^t + |beta||C| per
    batch entry for rounding bounds (None for integer operands))."""
    gap = 34 if batch > 1 else 0
    P, ldp, sP, Pv = _operand(rng, R, K, pk, ld_extra, batch, gap, flags & KB_R, flags & KE_R, normal)
    Q, ldq, sQ, Qv = _operand(rng, S, K, qk, ld_extra, batch, gap, flags & KB_S, flags & KE_S, normal)
    ldd = S + ld_extra
    sD = R * ldd + gap
    Dbuf = np.full(batch * sD + gap, SENT)
    tiles = _tile_mask(R, S, flags & TRI_OUT)
    C = [rng.standard_normal((R, S)) if normal else rng.integers(-8, 9, size=(R, S)).astype(np.float64) for _ in range(batch)]
    Cbuf, ldc, sC = None, 0, 0
    if cin == "alias":
        for b, reg in enumerate(_regions(Dbuf, batch, sD, R, ldd, S)):
            reg[...] = C[b]
        ldc, sC = ldd, sD
    elif cin == "distinct":
        ldc = S + ld_extra + 4
        sC = R * ldc + gap + 2
        Cbuf = np.full(batch * sC + gap, NAN)       # padding, gaps and tiles that are not computed: never read
        for b, reg in enumerate(_regions(Cbuf, batch, sC, R, ldc, S)):
            reg[tiles] = C[b][tiles]
    expected = Dbuf.copy()
    bound = []
    for b, reg in enumerate(_regions(expected, batch, sD, R, ldd, S)):
        val = alpha * (Pv[b] @ Qv[b].T)
        mag = abs(alpha) * (np.abs(Pv[b]) @ np.abs(Qv[b]).T)
        if cin != "none":
            val = val + beta * C[b]
            mag = mag + abs(beta) * np.abs(C[b])
        reg[tiles] = val[tiles]
        bound.append(mag)
    dP, dQ, dD = _dev(P), _dev(Q), _dev(Dbuf)
    dC = _dev(Cbuf) if Cbuf is not None else None
    cptr = dD.data_ptr() if cin == "alias" else (dC.data_ptr() if dC is not None else None)
    rc, launches = _run(h, lambda: h.lib.gpk_debug_gemm(
        h.h, dP.data_ptr(), ldp, sP, dQ.data_ptr(), ldq, sQ, dD.data_ptr(), ldd, sD, cptr, ldc, sC,
        R, S, K, batch, alpha, beta, int(bool(pk)), int(bool(qk)), flags))
    return rc, launches, dD.cpu().numpy(), expected, (bound if normal else None), (sD, ldd, tiles)


# ------------------------------------------------------------------------------------------------------------------------
# exact-result matrix
# ------------------------------------------------------------------------------------------------------------------------
LAYOUTS = [(0, 0), (0, 1), (1, 0), (1, 1)]
FLAGSETS = [("plain", 0), ("kb_r", KB_R), ("kb_s", KB_S), ("ke_r", KE_R), ("ke_s", KE_S), ("kb_r+kb_s", KB_R | KB_S),
            ("tri_out", TRI_OUT), ("tri_out+kb_r+kb_s", TRI_OUT | KB_R | KB_S)]
# (name, R, S, K, extra ld): one tile; S/64 in {1, 7, 9, 50} around the 8-wide raster band; K in {0, 16, 48, 64, 80, 1024},
# above and below R and S; ragged leading dimensions (rows + 2)
SHAPES = [("one_tile", 64, 64, 64, 0), ("s7", 128, 448, 48, 2), ("s9", 192, 576, 80, 2), ("s50", 64, 3200, 16, 0),
          ("k1024", 320, 128, 1024, 2), ("k0", 128, 192, 0, 2)]
# (Cin, heavy_last, batch): each (layout, flags) pair meets all six across the shapes
VARIANTS = [("none", 0, 1), ("alias", 1, 3), ("distinct", 0, 3), ("none", 1, 3), ("alias", 0, 1), ("distinct", 1, 1)]
SCALARS = [1.0, -1.0, 0.5, 0.0, 2.0]

EXACT_CASES = []
for li, lay in enumerate(LAYOUTS):
    for fi, (fname, fl) in enumerate(FLAGSETS):
        for si, shp in enumerate(SHAPES):
            cin, heavy, batch = VARIANTS[(li + fi + si) % 6]
            alpha = SCALARS[(li + 2 * fi + si) % 5]
            beta = SCALARS[(2 * li + fi + 3 * si) % 5]
            flags = fl | (HEAVY_LAST if heavy else 0)
            EXACT_CASES.append(pytest.param(len(EXACT_CASES), lay, flags, shp, cin, batch, alpha, beta,
                                            id=f"pk{lay[0]}qk{lay[1]}-{fname}{'-heavy' if heavy else ''}-{shp[0]}-cin_{cin}"
                                               f"-b{batch}-a{alpha:g}-be{beta:g}"))


@pytest.mark.parametrize("seed,layout,flags,shape,cin,batch,alpha,beta", EXACT_CASES)
def test_gemm_exact(h, seed, layout, flags, shape, cin, batch, alpha, beta):
    _, R, S, K, ld_extra = shape
    rng = np.random.default_rng(seed)
    rc, launches, got, want, _, (sD, ldd, tiles) = _gemm_case(h, rng, R, S, K, batch, alpha, beta, layout[0], layout[1],
                                                               flags, cin, ld_extra)
    assert rc == 0
    assert launches == 1
    assert np.isfinite(got).all(), "NaN/inf in D: an operand region outside the k-range (or unread Cin) was read"
    bad = np.flatnonzero(got != want)
    if bad.size:
        i = bad[0]
        b, rem = divmod(i, sD)
        r, s = divmod(rem, ldd) if rem < R * ldd else (None, None)
        where = "batch gap / tail" if r is None else ("ld padding" if s >= S else
                                                       f"tile ({r // 64}, {s // 64}) {'written' if tiles[r, s] else 'not selected'}")
        pytest.fail(f"{bad.size} elements differ; first: batch {b}, r={r}, s={s} ({where}): got {got[i]!r}, want {want[i]!r}")


# ------------------------------------------------------------------------------------------------------------------------
# rounding level on large N(0,1) shapes
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("R,S,K,layout,flags,cin", [
    (2048, 2048, 4096, (1, 1), TRI_OUT, "alias"),
    (1024, 1024, 4096, (0, 0), TRI_OUT | KB_R | KB_S, "none"),
    (1024, 1536, 1024, (0, 1), HEAVY_LAST, "distinct"),
    (1536, 1024, 1024, (1, 0), KE_S | HEAVY_LAST, "distinct"),
])
def test_gemm_rounding_bound(h, R, S, K, layout, flags, cin):
    rng = np.random.default_rng(R + S + K + flags)
    alpha, beta = -1.0, 0.75
    rc, launches, got, want, bound, (sD, ldd, tiles) = _gemm_case(h, rng, R, S, K, 1, alpha, beta, layout[0], layout[1],
                                                                   flags, cin, 2, normal=True)
    assert rc == 0 and launches == 1
    g = got[:R * ldd].reshape(R, ldd)
    w = want[:R * ldd].reshape(R, ldd)
    assert np.array_equal(g[:, :S][~tiles], w[:, :S][~tiles]) and np.all(g[:, S:] == SENT), "unselected tiles or padding written"
    err = np.abs(g[:, :S] - w[:, :S])[tiles]
    lim = 2 * (K + 2) * U * bound[0][tiles]
    ratio = float(np.max(err / lim))
    assert ratio <= 1.0, f"max |D - D_ref| / (2(K+2)u(|a||P||Q|^t + |b||C|)) = {ratio:.3g}"


# ------------------------------------------------------------------------------------------------------------------------
# argument validation
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("what", ["R", "S", "K", "ldp", "ldq", "ldd", "ldc", "P", "Q", "D", "Cin"])
def test_gemm_rejects_bad_descriptor(h, what):
    import torch
    from gp_algos_b200 import _lib
    buf = torch.zeros(4 * 256 * 256 + 64, dtype=torch.float64, device="cuda")
    base = buf.data_ptr()
    arg = dict(P=base, Q=base + 8 * 70000, D=base + 8 * 140000, Cin=base + 8 * 210000, ldp=256, ldq=256, ldd=256, ldc=256,
               R=128, S=128, K=64)
    if what in ("R", "S"):
        arg[what] = 96
    elif what == "K":
        arg["K"] = 24
    elif what.startswith("ld"):
        arg[what] = 255
    else:
        arg[what] += 8                                                          # 8-byte aligned, not 16
    rc, launches = _run(h, lambda: h.lib.gpk_debug_gemm(
        h.h, arg["P"], arg["ldp"], 0, arg["Q"], arg["ldq"], 0, arg["D"], arg["ldd"], 0, arg["Cin"], arg["ldc"], 0,
        arg["R"], arg["S"], arg["K"], 1, 1.0, 1.0, 0, 0, 0))
    assert rc == _lib.GPK_EINVAL
    assert launches == 0


def test_gemm_rejects_unknown_flag(h):
    import torch
    from gp_algos_b200 import _lib
    buf = torch.zeros(3 * 64 * 64, dtype=torch.float64, device="cuda")
    p = buf.data_ptr()
    rc, launches = _run(h, lambda: h.lib.gpk_debug_gemm(h.h, p, 64, 0, p + 8 * 4096, 64, 0, p + 16 * 4096, 64, 0, None, 0, 0,
                                                        64, 64, 64, 1, 1.0, 0.0, 0, 0, 64))
    assert rc == _lib.GPK_EINVAL and launches == 0


# ------------------------------------------------------------------------------------------------------------------------
# public wrappers
# ------------------------------------------------------------------------------------------------------------------------
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
def test_gemm_nt_matches_torch(m, p, k, beta):
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


def _gemm_nt(h, m, p, k, alpha, Pl, Ql, beta, C0, q_lower_tri=0, ldextra=2):
    """gpk_gemm_nt_dev on host arrays (logical m x k, p x k, m x p); column-major buffers with ld = rows + ldextra whose
    padding is NaN.  Returns (C after, launches)."""
    ldp, ldq, ldc = m + ldextra, p + ldextra, m + ldextra

    def colmajor(a, rows, ld, cols):
        buf = np.full((max(cols, 1), ld), NAN)
        buf[:cols, :rows] = a.T
        return buf

    dP, dQ, dC = _dev(colmajor(Pl, m, ldp, k)), _dev(colmajor(Ql, p, ldq, k)), _dev(colmajor(C0, m, ldc, p))
    rc, launches = _run(h, lambda: h.lib.gpk_gemm_nt_dev(h.h, m, p, k, alpha, dP.data_ptr(), ldp, dQ.data_ptr(), ldq, beta,
                                                         dC.data_ptr(), ldc, q_lower_tri))
    h.check(rc)
    out = dC.cpu().numpy()
    assert np.isnan(out[:p, m:]).all(), "padding of C written"
    return out[:p, :m].T, launches


def _ints(rng, *shape):
    return rng.integers(-8, 9, size=shape).astype(np.float64)


def test_gemm_nt_beta0_does_not_read_c(h):
    rng = np.random.default_rng(11)
    m, p, k = 384, 256, 80
    Pl, Ql = _ints(rng, m, k), _ints(rng, p, k)
    C, launches = _gemm_nt(h, m, p, k, -0.5, Pl, Ql, 0.0, np.full((m, p), NAN))
    assert launches == 1
    assert np.array_equal(C, -0.5 * (Pl @ Ql.T))


@pytest.mark.parametrize("beta", [0.0, 1.0, -0.5])
def test_gemm_nt_k0_scales_c(h, beta):
    rng = np.random.default_rng(12)
    m, p = 256, 192
    C0 = _ints(rng, m, p) if beta != 0.0 else np.full((m, p), NAN)
    C, _ = _gemm_nt(h, m, p, 0, 2.0, np.zeros((m, 0)), np.zeros((p, 0)), beta, C0)
    assert np.array_equal(C, np.zeros((m, p)) if beta == 0.0 else beta * C0)


def test_gemm_nt_alpha0(h):
    rng = np.random.default_rng(13)
    m, p, k = 192, 320, 64
    C0 = _ints(rng, m, p)
    C, _ = _gemm_nt(h, m, p, k, 0.0, _ints(rng, m, k), _ints(rng, p, k), -1.0, C0)
    assert np.array_equal(C, -C0)


@pytest.mark.parametrize("m,p,k", [(384, 640, 640), (256, 512, 384), (128, 1152, 1152)])
def test_gemm_nt_q_lower_tri_reads_only_lower(h, m, p, k):
    """q_lower_tri: Q(c, kk) = 0 for kk > c.  Strict upper triangle of Q: real zeros inside the diagonal 128-blocks, NaN
    beyond them (the layout gpk_potrf_inv_block_dev leaves in L^-1)."""
    rng = np.random.default_rng(m + p + k)
    Pl = _ints(rng, m, k)
    Ql = np.tril(_ints(rng, p, k))
    Qn = Ql.copy()
    c = np.arange(p)[:, None]
    kk = np.arange(k)[None, :]
    Qn[kk >= (c // 128 + 1) * 128] = NAN
    C0 = _ints(rng, m, p)
    C, launches = _gemm_nt(h, m, p, k, 1.0, Pl, Qn, 2.0, C0, q_lower_tri=1)
    assert launches == 1
    assert np.array_equal(C, Pl @ Ql.T + 2.0 * C0)
