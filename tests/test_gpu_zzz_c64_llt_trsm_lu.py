"""c64 (complex128) triangular solves and Cholesky LLT through the C ABI (csrc/cplx.cu) against the oracle's c64 restatement
of the same recursions (triangular_solve.rs:220-604 with the conjugation flag, cholesky/llt/factor.rs:68-97 for complex T):
solves within the backward bound for all four variants x conj, LLT: L L^H = A within 64 n u |A|, close to the oracle's factor,
strict upper triangle untouched, NonPositivePivot index and regularisation count exact, the solve on the factor."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
U = 2.0 ** -53


def crandn(rng, shape):
    return np.asfortranarray(rng.standard_normal(shape) + 1j * rng.standard_normal(shape))


def test_c64_triangular_solves_vs_oracle(fb, oracle):
    la = fb.linalg
    rng = np.random.default_rng(141)
    for n, k in [(1, 1), (5, 3), (32, 7), (33, 40), (100, 64), (257, 130)]:
        T = crandn(rng, (n, n)) + 4 * np.sqrt(n) * np.eye(n)
        B = crandn(rng, (n, k))
        for lower in (True, False):
            for unit in (False, True):
                for conj in (0, 1):
                    Tt = np.asfortranarray(np.tril(T) if lower else np.triu(T))
                    if unit:
                        Tt = np.asfortranarray(Tt / (2.0 * np.sqrt(n)))  # keep the unit-diagonal system well conditioned
                    want = B.copy(order="F"); oracle.solve_triangular(Tt, want, lower, unit, bool(conj))
                    got = B.copy(order="F")
                    f = {(True, False): la.solve_lower_triangular_in_place, (False, False): la.solve_upper_triangular_in_place,
                         (True, True): la.solve_unit_lower_triangular_in_place, (False, True): la.solve_unit_upper_triangular_in_place}[(lower, unit)]
                    f(Tt, got, conj)
                    Te = (np.tril(Tt, -1) if lower else np.triu(Tt, 1)) + (np.eye(n) if unit else np.diag(np.diag(Tt)))
                    Te = Te.conj() if conj else Te
                    res = np.abs(Te @ got - B)
                    bound = 16 * n * U * (np.abs(Te) @ np.abs(got) + np.abs(B)) + 1e-300
                    assert np.all(res <= bound), (n, k, lower, unit, conj, float((res / bound).max()))
                    assert np.allclose(got, want, rtol=1e-9, atol=1e-9 * np.abs(want).max()), (n, k, lower, unit, conj)


def test_c64_llt_vs_oracle(fb, oracle):
    la = fb.linalg
    rng = np.random.default_rng(142)
    for n in [1, 2, 31, 32, 33, 64, 100, 257, 600]:
        G = crandn(rng, (n, n))
        A = np.asfortranarray(G @ G.conj().T + n * np.eye(n))
        want = A.copy(order="F"); fail, cnt = oracle.llt(want)
        assert fail == -1
        got = A.copy(order="F")
        got[np.triu_indices(n, 1)] = 123.0 + 7j  # the strict upper triangle is neither read nor written
        info = la.cholesky_in_place(got)
        assert info.dynamic_regularization_count == 0
        assert np.all(got[np.triu_indices(n, 1)] == 123.0 + 7j), n
        L = np.tril(got)
        assert np.max(np.abs(L @ L.conj().T - A)) <= 64 * n * U * np.max(np.abs(A)), n
        assert np.allclose(L, np.tril(want), rtol=1e-10, atol=1e-10 * np.abs(want).max()), n
        # solve on the factor, both conjugation settings
        B = crandn(rng, (n, 3))
        for conj in (0, 1):
            X = B.copy(order="F"); la.llt_solve_in_place(got, X, conj)
            Ae = A.conj() if conj else A
            assert np.max(np.abs(Ae @ X - B)) <= 256 * n * U * np.linalg.cond(A) * np.max(np.abs(B)), (n, conj)


def test_c64_llt_error_index_and_regularization(fb, oracle):
    la = fb.linalg
    rng = np.random.default_rng(143)
    n = 90
    G = crandn(rng, (n, n))
    A = np.asfortranarray(G @ G.conj().T + n * np.eye(n))
    bad = A.copy(order="F"); bad[57, 57] = -1.0
    want = bad.copy(order="F"); fail, _ = oracle.llt(want)
    assert fail >= 0
    with pytest.raises(la.LltError) as e:
        la.cholesky_in_place(bad.copy(order="F"))
    assert f"index: {fail}" in str(e.value)
    # dynamic regularisation: pivots <= eps are replaced by delta, the count comes back exactly
    R = A.copy(order="F"); R[10, 10] = 1e-30; R[11:, 10] = 0; R[10, :10] = 0
    want = R.copy(order="F"); fail, cnt = oracle.llt(want, delta=1e-3, eps=1e-8)
    got = R.copy(order="F"); info = la.cholesky_in_place(got, regularization=(1e-3, 1e-8))
    assert fail == -1 and info.dynamic_regularization_count == cnt and cnt >= 1


def test_c64_lu_vs_oracle(fb, oracle):
    """c64 partial-pivoting LU (lu/partial_pivoting/factor.rs:19-295 for complex T; pivot = first row attaining the largest
    |re| + |im|): permutations and transposition count bit-exact vs the oracle, factors to rounding, and the solve on the factors
    with both conjugation settings (lu/partial_pivoting/solve.rs:21-54)."""
    la = fb.linalg
    rng = np.random.default_rng(144)
    for (m, n) in [(1, 1), (7, 7), (16, 16), (17, 17), (40, 40), (130, 70), (70, 130), (300, 300), (800, 800)]:
        for idx in (np.uint32, np.uint64):
            A = crandn(rng, (m, n))
            want = A.copy(order="F"); po, pio, nt = oracle.lu(want)
            got = A.copy(order="F")
            p = np.zeros(m, dtype=idx); pi = np.zeros(m, dtype=idx)
            info = la.lu_in_place(got, p, pi)
            assert np.array_equal(p.astype(np.int64), po) and np.array_equal(pi.astype(np.int64), pio), (m, n)
            assert info.transposition_count == nt, (m, n)
            assert np.allclose(got, want, rtol=1e-9, atol=1e-9 * np.abs(want).max()), (m, n)
            if m == n:
                B = crandn(rng, (n, 3))
                for conj in (0, 1):
                    X = B.copy(order="F"); la.lu_solve_in_place(got, p, pi, X, conj)
                    Ae = A.conj() if conj else A
                    assert np.max(np.abs(Ae @ X - B)) <= 256 * n * U * np.linalg.cond(A) * np.max(np.abs(B)), (n, conj)
                    X = B.copy(order="F"); la.lu_solve_transpose_in_place(got, p, pi, X, conj)  # solve.rs:55-86
                    assert np.max(np.abs(Ae.T @ X - B)) <= 256 * n * U * np.linalg.cond(A) * np.max(np.abs(B)), (n, conj, "T")


@pytest.mark.parametrize("cdt,rdt", [(np.complex128, np.float64), (np.complex64, np.float32)])
def test_lu_solves_on_a_device_rhs_aligned_to_the_real_type(fb, cdt, rdt):
    """faer's c64 / c32 are aligned like f64 / f32 only, so a device rhs may start at 8 mod 16 bytes (c64) or 4 mod 8 (c32). The
    complex LU solves, row permutation included, use such a rhs in place and solve within the same backward bound as on the host."""
    import torch
    la, capi = fb.linalg, fb.capi
    lib = capi.load()
    rng = np.random.default_rng(7)
    n, k = 300, 3
    A = crandn(rng, (n, n)).astype(cdt)
    LU = A.copy(order="F")
    p = np.zeros(n, np.uint64); pi = np.zeros(n, np.uint64)
    la.lu_in_place(LU, p, pi)
    B = crandn(rng, (n, k)).astype(cdt)
    suf = "c64" if cdt == np.complex128 else "c32"
    u = U if cdt == np.complex128 else 2.0 ** -24
    bound = 256 * n * u * np.linalg.cond(A.astype(np.complex128)) * np.max(np.abs(B))
    for name, op in (("partial_piv_lu_solve_in_place", A), ("partial_piv_lu_solve_transpose_in_place", A.T)):
        # one real element in front of the complex entries: the base is aligned to the real type and no more
        buf = torch.zeros(1 + 2 * n * k, dtype=torch.float64 if rdt == np.float64 else torch.float32, device="cuda")
        buf[1:] = torch.from_numpy(np.ascontiguousarray(B.T).view(rdt).reshape(-1)).cuda()
        ptr = buf.data_ptr() + buf.element_size()
        assert ptr % (2 * buf.element_size()) != 0
        getattr(lib, f"libfaer_v0_23_{name}_u64_{suf}")(capi.mat_ref(LU), capi.mat_ref(LU), 0, capi.slice_mut(p), capi.slice_mut(pi),
                                                       capi.MatMut(ptr, n, k, 1, n), capi.par_default(), capi.MemAlloc(None, 0))
        torch.cuda.synchronize()
        got = buf[1:].cpu().numpy().view(cdt).reshape(k, n).T
        assert np.max(np.abs(op.astype(np.complex128) @ got.astype(np.complex128) - B)) <= bound, name
