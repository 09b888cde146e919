"""Row-bundle storage order of H.v (csrc/bundle.cu): every bundle size gives the same H.v as the oracle, and the
encode/decode pair is an exact in-place permutation (export_upper / get_row are bit-identical to the plain layout)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


from conftest import C2_FCIDUMP


def _heg_big(oracle):
    import sqmc_b200 as sq
    # 81 plane waves (two-word strings), one HCI iteration: the Hartree-Fock row holds 3045 entries, the rest ~100
    S = oracle.System.heg(3, 0.5, 14, 7, 2.5)
    hs = sq.HegSystem(3, 0.5, 14, 7, 2.5)
    r = S.hci(2e-3, n_states=1, max_iters=1)
    return S, hs, r["up"], r["dn"]


@pytest.mark.parametrize("space,cap", [("c2", None), ("heg_big", None), ("c2", 256), ("heg_big", 1024)])
def test_bundles_match_oracle_and_round_trip_exactly(oracle, c2_space, space, cap, monkeypatch):
    """cap: lowers the encoder's shared-memory staging capacity so that long bundles take its tag-only path
    (entries keep their row-contiguous order and only receive the row tag)."""
    import sqmc_b200 as sq
    if cap:
        monkeypatch.setenv("SQMC_BUNDLE_CAP", str(cap))
    from sqmc_b200 import spaces
    if space == "c2":
        S, r = c2_space
        up, dn = r["up"], r["dn"]
        H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    else:
        S, hs, up, dn = _heg_big(oracle)
        H = sq.SparseHamiltonian(hs)
    n = len(up)
    cnt, idx, val = S.build_upper(up, dn)
    H.generate_sparse_ham_upper_triangular(up, dn)
    x = spaces.splitmix_vector(n, seed=7)
    y_ref = oracle.matvec_upper(cnt, idx, val, x)
    H.set_row_bundle(0)
    plain = H.export_upper()
    rows = [1, 2, n // 3, n // 2, n - 1, n]
    plain_rows = [H.get_row(r) for r in rows]
    for R in (2, 4, 0, 2, 4):
        H.set_row_bundle(R)
        y = H.matvec(x)
        assert np.max(np.abs(y - y_ref)) <= 1e-10 * max(1.0, np.max(np.abs(y_ref))), R
        e = H.export_upper()
        for a, b in zip(plain, e):
            assert np.array_equal(a, b), R          # bit-exact: counts, 1-based columns, values
        for r, (pc, pv) in zip(rows, plain_rows):
            c, v = H.get_row(r)
            assert np.array_equal(pc, c) and np.array_equal(pv, v), (R, r)
    assert np.array_equal(plain[0], cnt) and np.array_equal(plain[1], idx) and np.array_equal(plain[2], val)


def test_bundled_davidson_and_projector(oracle, c2_space):
    import sqmc_b200 as sq
    S, r = c2_space
    up, dn = r["up"], r["dn"]
    cnt, idx, val = S.build_upper(up, dn)
    ref = oracle.davidson(cnt, idx, val, n_states=1)
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    H.generate_sparse_ham_upper_triangular(up, dn)
    energies = []
    for R in (0, 2, 4):
        H.set_row_bundle(R)
        d = H.davidson_sparse(n_states=1)
        energies.append(float(d["evals"][0]))
        assert abs(energies[-1] - ref["evals"][0]) < 1e-8
    tau = 0.01
    w = np.abs(ref["evecs"][:, 0]) + 0.01
    _, dw_ref = oracle.projector_step(cnt, idx, -tau * val, tau, ref["evals"][0], w)
    H.scale_values(-tau)
    for R in (4, 0, 2):
        H.set_row_bundle(R)
        dw = H.projector_step(tau, ref["evals"][0], w)
        assert np.max(np.abs(dw - dw_ref)) <= 1e-12 * np.max(np.abs(dw_ref)) + 1e-15


def test_two_state_davidson_uses_the_pair_kernel(oracle, c2_space_ts):
    """n_states = 2 (the shipped C2 input): the H.v of each block of two new vectors go through the two-vector kernel on
    bundled matrices and through two single products on plain rows; both reproduce the oracle's Ritz values."""
    import sqmc_b200 as sq
    s, r = c2_space_ts
    cnt, idx, val = s.build_upper(r["up"], r["dn"])
    ref = oracle.davidson(cnt, idx, val, n_states=2)
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=True, z=1))
    H.generate_sparse_ham_upper_triangular(r["up"], r["dn"])
    got = {}
    for R in (4, 0, 2):
        H.set_row_bundle(R)
        d = H.davidson_sparse(n_states=2)
        assert np.max(np.abs(d["evals"] - ref["evals"])) < 1e-8
        assert d["n_matvec"] == ref["n_matvec"]
        got[R] = d
    # same arithmetic per vector whichever kernel applied H: eigenvectors agree to rounding
    for R in (0, 2):
        for q in range(2):
            a, b = got[4]["evecs"][:, q], got[R]["evecs"][:, q]
            assert min(np.max(np.abs(a - b)), np.max(np.abs(a + b))) < 1e-9


@pytest.mark.parametrize("n", [1, 2, 3, 5, 9, 33])
def test_tiny_spaces_in_every_layout(oracle, heg_space, n):
    """fewer rows than a bundle, ragged last bundle, single-determinant space: build, H.v, row access, Davidson, Lanczos"""
    import sqmc_b200 as sq
    s, r = heg_space
    up, dn = r["up"][:n], r["dn"][:n]
    cnt, idx, val = s.build_upper(up, dn)
    H = sq.SparseHamiltonian(sq.HegSystem(3, 0.5, 14, 7, 1.49))
    assert H.generate_sparse_ham_upper_triangular(up, dn) == len(idx)
    x = np.linspace(-1.0, 1.0, n) + 0.25
    yref = oracle.matvec_upper(cnt, idx, val, x)
    ref = oracle.davidson(cnt, idx, val, n_states=1)
    for R in (4, 2, 0):
        H.set_row_bundle(R)
        assert np.max(np.abs(H.matvec(x) - yref)) <= 1e-12 * max(np.max(np.abs(yref)), 1e-300)
        e = H.export_upper()
        assert np.array_equal(e[0], cnt) and np.array_equal(e[1], idx) and np.array_equal(e[2], val)
        c, v = H.get_row(n)
        assert c[-1] == n and v[-1] == val[-1]        # full row, ascending columns: its last entry is the diagonal of row n
        assert abs(H.davidson_sparse(n_states=1)["evals"][0] - ref["evals"][0]) < 1e-8
        assert abs(H.matrix_lanczos_sparse()["lowest_eigenvalue"] - oracle.lanczos(cnt, idx, val)["lowest"]) < 1e-8


@pytest.mark.parametrize("R", [2, 4])
def test_unaligned_vector_takes_lsu_gathers_with_identical_result(c2_space, R):
    """A vector whose base is not 512-byte aligned cannot back a linear texture: the bundle kernel gathers it with LSU loads
    instead.  The same x read from a 512-byte aligned and from an 8-byte offset device address gives the same y, bit for bit,
    and that y agrees with the plain-row product.  sqmc_b200_matvec_dev works in the library's internal row order."""
    import ctypes as C
    import sqmc_b200 as sq
    from sqmc_b200 import _lib, spaces
    S, r = c2_space
    H = sq.SparseHamiltonian(sq.ChemSystem(C2_FCIDUMP, time_sym=False, z=1))
    H.generate_sparse_ham_upper_triangular(r["up"], r["dn"])
    n = len(r["up"])
    L = _lib.load()
    x = spaces.splitmix_vector(n, seed=11)
    base, ybuf = C.c_void_p(), C.c_void_p()
    _lib.check(L.sqmc_b200_device_malloc(C.byref(base), (n + 128) * 8))
    _lib.check(L.sqmc_b200_device_malloc(C.byref(ybuf), n * 8))
    try:
        aligned = (base.value + 511) // 512 * 512
        assert aligned + 8 + n * 8 <= base.value + (n + 128) * 8

        def product(x_addr):
            _lib.check(L.sqmc_b200_memcpy_h2d(x_addr, x.ctypes.data, n * 8))
            _lib.check(L.sqmc_b200_matvec_dev(H._h, x_addr, ybuf, None))
            y = np.empty(n)
            _lib.check(L.sqmc_b200_memcpy_d2h(y.ctypes.data, ybuf, n * 8))
            return y

        H.set_row_bundle(0)
        y_plain = product(aligned)
        H.set_row_bundle(R)
        y_tex = product(aligned)
        y_lsu = product(aligned + 8)
        assert np.array_equal(y_tex, y_lsu)
        assert np.max(np.abs(y_tex - y_plain)) <= 1e-12 * np.max(np.abs(y_plain))
    finally:
        L.sqmc_b200_device_free(base)
        L.sqmc_b200_device_free(ybuf)
