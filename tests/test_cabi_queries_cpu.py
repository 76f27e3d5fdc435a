"""Every default-params, scratch-size and block-size query of the C ABI, for f64 / f32 / c64 / c32 (and u32 / u64 index types where
they exist), against faer's formulas with the element size of T. The queries need no GPU; they are the same formula for every dtype,
so one wrong element size in one dtype's copy shows here.

Formulas: temp_mat_scratch::<T>(dim, 1) for the LLT / LDLT factorizations (llt/factor.rs:58-66, ldlt/factor.rs:715-724), EMPTY for
the LLT / LDLT solves and llt_reconstruct, StackReq::new::<I>(min(nrows, ncols)) for the LU factorization (lu/partial_pivoting/
factor.rs:224-233), permute_rows_in_place_scratch temp_mat(dim, rhs_ncols) for the LU solves, the block-Householder sequence scratch
temp_mat(block_size, ncols) for QR and everything on its factors (qr/no_pivoting/solve.rs:3-37, householder.rs), temp_mat(dim, dim)
or temp_mat(nrows, ncols) for the reconstructs / inverses, a copy of A for svd / self_adjoint_evd. Default params: ldlt/factor.rs:
705-714, lu/partial_pivoting/factor.rs:212-222, qr/no_pivoting/factor.rs:91-116 and the reference's svd / evd / hessenberg
defaults."""
import ctypes as C

import pytest

DTYPES = (("f64", 8), ("f32", 4), ("c64", 16), ("c32", 8))
ITYPES = (("u32", 4), ("u64", 8))
Z = C.c_size_t


class HessenbergParams(C.Structure):
    _fields_ = [("par_threshold", C.c_size_t), ("blocking_threshold", C.c_size_t)]


def ref_qr_block_size(nrows, ncols):
    prod, size = nrows * ncols, min(nrows, ncols)
    for lim, bs in ((8192 * 8192, 256), (2048 * 2048, 128), (1024 * 1024, 64), (512 * 512, 48), (128 * 128, 32), (32 * 32, 8),
                    (16 * 16, 4)):
        if prod > lim:
            break
    else:
        bs = 1
    return max(1, min(bs, size))


@pytest.fixture(scope="module")
def q(fb):
    """A private handle on the product library, so that the argument types set here touch no other test's."""
    capi = fb.capi
    lib = C.CDLL(capi.LIB_PATH)
    P = capi.Par

    def fn(name, argtypes, restype=capi.Layout):
        f = getattr(lib, "libfaer_v0_23_" + name)
        f.argtypes, f.restype = argtypes, restype
        return f

    fn.lib, fn.capi, fn.par = lib, capi, capi.par_default()
    fn.P = P
    return fn


@pytest.mark.parametrize("suf,es", DTYPES)
def test_default_params(q, suf, es):
    capi = q.capi
    p = q(f"LltParams_{suf}", [], capi.LltParams)()
    assert (p.recursion_threshold, p.block_size) == (64, 128)
    p = q(f"LdltParams_{suf}", [], capi.LdltParams)()
    assert (p.recursion_threshold, p.block_size) == (64, 128)
    p = q(f"PartialPivLuParams_{suf}", [], capi.PartialPivLuParams)()
    assert (p.recursion_threshold, p.block_size, p.par_threshold) == (16, 64, 128 * 128)
    p = q(f"QrParams_{suf}", [], capi.QrParams)()
    assert (p.blocking_threshold, p.par_threshold) == (48 * 48, 192 * 256)
    assert q(f"BidiagParams_{suf}", [], capi.BidiagParams)().par_threshold == 192 * 256
    p = q(f"SvdParams_{suf}", [], capi.SvdParams)()
    assert p.bidiag.par_threshold == 192 * 256 and (p.qr.blocking_threshold, p.qr.par_threshold) == (48 * 48, 192 * 256)
    assert p.recursion_threshold == 128 and p.qr_ratio_threshold == 11.0 / 6.0
    assert q(f"TridiagParams_{suf}", [], capi.TridiagParams)().par_threshold == 192 * 256
    p = q(f"SelfAdjointEvdParams_{suf}", [], capi.SelfAdjointEvdParams)()
    assert p.tridiag.par_threshold == 192 * 256 and p.recursion_threshold == 128
    p = q(f"HessenbergParams_{suf}", [], HessenbergParams)()
    assert (p.par_threshold, p.blocking_threshold) == (192 * 256, 256 * 256)


@pytest.mark.parametrize("suf,es", DTYPES)
def test_cholesky_scratch(q, suf, es):
    capi, P, par = q.capi, q.P, q.par
    for dim, k in ((0, 0), (1, 3), (1000, 7), (257, 64)):
        lay = q(f"llt_factor_in_place_scratch_{suf}", [Z, P, capi.LltParams])(dim, par, capi.LltParams(64, 128))
        assert (lay.len_bytes, lay.align_bytes) == (dim * es, 64)
        lay = q(f"ldlt_factor_in_place_scratch_{suf}", [Z, P, capi.LdltParams])(dim, par, capi.LdltParams(64, 128))
        assert (lay.len_bytes, lay.align_bytes) == (dim * es, 64)
        for name in ("llt_solve_in_place_scratch", "ldlt_solve_in_place_scratch"):
            lay = q(f"{name}_{suf}", [Z, Z, P])(dim, k, par)
            assert (lay.len_bytes, lay.align_bytes) == (0, 1)
        lay = q(f"llt_reconstruct_scratch_{suf}", [Z, P])(dim, par)
        assert (lay.len_bytes, lay.align_bytes) == (0, 1)
        for name in ("llt_inverse_scratch", "ldlt_reconstruct_scratch", "ldlt_inverse_scratch"):
            lay = q(f"{name}_{suf}", [Z, P])(dim, par)
            assert (lay.len_bytes, lay.align_bytes) == (dim * dim * es, 64)


@pytest.mark.parametrize("suf,es", DTYPES)
@pytest.mark.parametrize("it,ib", ITYPES)
def test_lu_scratch(q, suf, es, it, ib):
    capi, P, par = q.capi, q.P, q.par
    for m, n, k in ((0, 0, 0), (300, 200, 7), (200, 300, 1), (64, 64, 64)):
        lay = q(f"partial_piv_lu_factor_in_place_scratch_{it}_{suf}", [Z, Z, P, capi.PartialPivLuParams])(
            m, n, par, capi.PartialPivLuParams(16, 64, 128 * 128))
        assert (lay.len_bytes, lay.align_bytes) == (min(m, n) * ib, ib)
        for name in ("partial_piv_lu_solve_in_place_scratch", "partial_piv_lu_solve_transpose_in_place_scratch"):
            lay = q(f"{name}_{it}_{suf}", [Z, Z, P])(m, k, par)
            assert (lay.len_bytes, lay.align_bytes) == (m * k * es, 64)
        lay = q(f"partial_piv_lu_reconstruct_scratch_{it}_{suf}", [Z, Z, P])(m, n, par)
        assert (lay.len_bytes, lay.align_bytes) == (m * n * es, 64)
        lay = q(f"partial_piv_lu_inverse_scratch_{it}_{suf}", [Z, P])(n, par)
        assert (lay.len_bytes, lay.align_bytes) == (n * n * es, 64)


@pytest.mark.parametrize("suf,es", DTYPES)
def test_qr_scratch(q, suf, es):
    capi, P, par = q.capi, q.P, q.par
    bs_fn = q(f"qr_recommended_block_size_{suf}", [Z, Z], Z)
    for m, n in ((0, 0), (1, 1), (16, 17), (100, 100), (513, 512), (4000, 300), (10000, 9000), (3, 100000)):
        assert bs_fn(m, n) == ref_qr_block_size(m, n), (m, n)
    for m, n, bs, k in ((1000, 300, 32, 7), (300, 300, 16, 5), (0, 0, 1, 0), (64, 48, 48, 1)):
        lay = q(f"qr_factor_in_place_scratch_{suf}", [Z, Z, Z, P, capi.QrParams])(m, n, bs, par, capi.QrParams(48 * 48, 192 * 256))
        assert (lay.len_bytes, lay.align_bytes) == (bs * n * es, 64)
        for side in ("left", "right"):
            for name in (f"apply_householder_on_the_{side}_scratch", f"apply_householder_transpose_on_the_{side}_scratch"):
                lay = q(f"{name}_{suf}", [Z, Z, Z])(m, bs, k)
                assert (lay.len_bytes, lay.align_bytes) == (bs * k * es, 64)
        lay = q(f"qr_solve_lstsq_in_place_scratch_{suf}", [Z, Z, Z, Z, P])(m, n, bs, k, par)
        assert (lay.len_bytes, lay.align_bytes) == (bs * k * es, 64)
        for name in ("qr_solve_in_place_scratch", "qr_solve_transpose_in_place_scratch"):
            lay = q(f"{name}_{suf}", [Z, Z, Z, P])(n, bs, k, par)
            assert (lay.len_bytes, lay.align_bytes) == (bs * k * es, 64)
        lay = q(f"qr_reconstruct_scratch_{suf}", [Z, Z, Z, P])(m, n, bs, par)
        assert (lay.len_bytes, lay.align_bytes) == (bs * n * es, 64)
        lay = q(f"qr_inverse_scratch_{suf}", [Z, Z, P])(n, bs, par)
        assert (lay.len_bytes, lay.align_bytes) == (bs * n * es, 64)


@pytest.mark.parametrize("suf,es", DTYPES)
def test_svd_evd_scratch(q, suf, es):
    capi, P, par = q.capi, q.P, q.par
    svd_p = q(f"SvdParams_{suf}", [], capi.SvdParams)()
    evd_p = q(f"SelfAdjointEvdParams_{suf}", [], capi.SelfAdjointEvdParams)()
    svd = q(f"svd_scratch_{suf}", [Z, Z, C.c_int, C.c_int, P, capi.SvdParams])
    evd = q(f"self_adjoint_evd_scratch_{suf}", [Z, C.c_int, P, capi.SelfAdjointEvdParams])
    for m, n in ((0, 0), (7, 3), (100, 250), (512, 512)):
        for cu in (0, 1, 2):
            lay = svd(m, n, cu, 2 - cu, par, svd_p)
            assert (lay.len_bytes, lay.align_bytes) == (m * n * es, 64)
        for cu in (0, 1):
            lay = evd(n, cu, par, evd_p)
            assert (lay.len_bytes, lay.align_bytes) == (n * n * es, 64)
