"""-m "not gpu": the host side of CSR-resident training: prepare_adatas keeps sparse inputs sparse, CsrCounts canonicalises a
scipy matrix before the upload (duplicates summed, zeros dropped, columns sorted, dtype rule, int64 offsets, gene limit), and
synth.make_counts_csr draws the same counts as synth.make_counts."""
import numpy as np
import pandas as pd
import pytest
import scipy.sparse as sp
import torch


def _groups(rng, sparse, n=(13, 9), genes=(6, 4)):
    from spvipes_b200.model import GroupedData
    out = {}
    for k, (N, G) in zip(("a", "b"), zip(n, genes)):
        X = rng.poisson(0.7, (N, G)).astype(np.float32)
        X[2] = 0  # an empty row
        out[k] = GroupedData(X=sp.csr_matrix(X) if sparse else X, obs=pd.DataFrame({"cell_types": rng.integers(0, 3, N)}),
                             var_names=[f"g{i}" for i in range(G)])
    return out


def test_prepare_adatas_sparse_inputs_stay_sparse():
    from spvipes_b200.model import prepare_adatas
    rng = np.random.default_rng(0)
    dense_in = _groups(rng, False)
    sparse_in = {k: type(v)(X=sp.csr_matrix(v.X), obs=v.obs, var_names=v.var_names) for k, v in dense_in.items()}
    d, s = prepare_adatas(dense_in), prepare_adatas(sparse_in)
    assert isinstance(d.X, np.ndarray) and d.X.dtype == np.float32
    assert sp.issparse(s.X) and s.X.format == "csr" and s.X.dtype == np.float32
    assert np.array_equal(np.asarray(s.X.todense()), d.X)
    assert s.uns["groups_var_indices"][1].tolist() == d.uns["groups_var_indices"][1].tolist()
    # one sparse input is enough for a sparse join
    mixed = prepare_adatas({"a": sparse_in["a"], "b": dense_in["b"]})
    assert sp.issparse(mixed.X) and np.array_equal(mixed.X.toarray(), d.X)


def test_prepare_adatas_dense_inputs_unchanged():
    """all-dense inputs: the zero-filled outer join, byte for byte"""
    from spvipes_b200.model import prepare_adatas
    rng = np.random.default_rng(1)
    ins = _groups(rng, False)
    out = prepare_adatas(ins)
    ref = np.zeros((13 + 9, 10), dtype=np.float32)
    ref[:13, :6] = ins["a"].X
    ref[13:, 6:] = ins["b"].X
    assert out.X.dtype == ref.dtype and out.X.tobytes() == ref.tobytes()


def _canon(m):
    from spvipes_b200.engine import CsrCounts
    return CsrCounts.canonical_arrays(m)


def test_canonical_sums_duplicates_and_drops_zeros():
    # row 0: duplicates (col 3 twice, col 1 three times), unsorted; row 1 empty; row 2: an explicit zero; row 3 dense
    data = np.array([2, 5, 1, 1, 1, 0, 4, 7, 1, 1, 1, 1], dtype=np.float32)
    ind = np.array([3, 3, 1, 1, 1, 2, 0, 4, 0, 1, 2, 3])
    ptr = np.array([0, 5, 5, 8, 12])
    m = sp.csr_matrix((data, ind, ptr), shape=(4, 5))
    assert not m.has_canonical_format
    indptr, indices, values, shape = _canon(m)
    assert shape == (4, 5)
    assert indptr.dtype == np.int64 and indices.dtype == np.uint16 and values.dtype == np.uint16
    assert indptr.tolist() == [0, 2, 2, 4, 8]
    assert indices.tolist() == [1, 3, 0, 4, 0, 1, 2, 3]
    assert values.tolist() == [3, 7, 4, 7, 1, 1, 1, 1]
    rebuilt = sp.csr_matrix((values, indices.astype(np.int64), indptr), shape=shape).toarray()
    assert np.array_equal(rebuilt, m.toarray())


@pytest.mark.parametrize("vals,expect", [
    ([1.0, 65535.0], np.uint16),
    ([3, 9], np.uint16),                # integer dtype
    ([0.5, 2.0], np.float32),           # non-integer
    ([-1.0, 2.0], np.float32),          # negative
    ([65536.0, 2.0], np.float32),       # beyond uint16
    ([70000, 1], np.float32),           # integer dtype beyond uint16
])
def test_canonical_dtype_rule(vals, expect):
    vals = np.asarray(vals)
    m = sp.csr_matrix((vals, np.array([0, 2]), np.array([0, 1, 2])), shape=(2, 3))
    _, _, values, _ = _canon(m)
    assert values.dtype == expect
    assert np.array_equal(values.astype(np.float64), vals.astype(np.float32).astype(np.float64))


def test_canonical_empty_matrix():
    indptr, indices, values, shape = _canon(sp.csr_matrix((3, 7), dtype=np.float32))
    assert indptr.tolist() == [0, 0, 0, 0] and indptr.dtype == np.int64 and len(indices) == 0 and values.dtype == np.uint16


def test_canonical_rejects_too_many_genes():
    from spvipes_b200 import _lib as L
    lib = L.load()
    for src, vals in ((L.SRC_U16_LOG1P, [1.0]), (L.SRC_F32_LOG1P, [0.5])):
        limit = int(lib.spv_csr_max_genes(src))
        ok = sp.csr_matrix((np.asarray(vals), np.array([limit - 1]), np.array([0, 1])), shape=(1, limit))
        _canon(ok)
        bad = sp.csr_matrix((np.asarray(vals), np.array([0]), np.array([0, 1])), shape=(1, limit + 1))
        with pytest.raises(ValueError, match=str(limit)):
            _canon(bad)
    assert lib.spv_csr_max_genes(L.SRC_U16_LOG1P) == 65536
    # float32: the 227 KB of shared memory a CTA may use, less the 32 bytes of the library-size reduction
    assert lib.spv_csr_max_genes(L.SRC_F32_LOG1P) == (227 * 1024 - 32) // 16 * 4


@pytest.mark.parametrize("src,ld_xs,dst,ld_dst,n_cov,cov,G", [
    (1, 96, None, 0, 0, None, 100),      # ld_xs < G
    (1, 100, None, 0, 0, None, 100),     # uint16 pitch not a multiple of 8
    (2, 102, None, 0, 0, None, 100),     # float pitch not a multiple of 4
    (1, 104, 4096, 100, 0, None, 100),   # ld_dst not a multiple of 8
    (1, 104, 4096, 104, 2, None, 100),   # covariate columns without codes
    (1, 104, 4096, 104, 5, 4096, 100),   # ld_dst < G + n_cov
    (1, 65544, None, 0, 0, None, 65537), # beyond the uint16 limit
    (0, 104, None, 0, 0, None, 100),     # not a count source
])
def test_gather_rejects_bad_arguments(src, ld_xs, dst, ld_dst, n_cov, cov, G):
    """argument errors are reported before anything is launched (the pointers here are never dereferenced)"""
    from spvipes_b200 import _lib as L
    fake = 4096
    rc = L.load().spv_csr_gather(src, fake, fake, fake, None, 4, G, fake, ld_xs, dst, None, ld_dst, None, cov, n_cov, None)
    assert rc == -1


def test_from_scipy_cpu_roundtrip():
    from spvipes_b200.engine import CsrCounts
    rng = np.random.default_rng(2)
    X = rng.poisson(0.3, (20, 11)).astype(np.float32)
    c = CsrCounts.from_scipy(sp.csr_matrix(X), device="cpu")
    assert c.shape == (20, 11) and c.indptr.dtype == torch.int64 and c.values.dtype == torch.uint16
    m = sp.csr_matrix((c.values.numpy(), c.indices.numpy().astype(np.int64), c.indptr.numpy()), shape=c.shape)
    assert np.array_equal(m.toarray(), X)
    assert c.resident_bytes() == 8 * 21 + 4 * int(c.indptr[-1])


@pytest.mark.parametrize("chunk", [64, 1000])
def test_make_counts_csr_equals_make_counts(chunk):
    from spvipes_b200 import synth
    a = synth.make_counts((300, 130), (77, 40), n_labels=4, device="cpu", chunk=chunk)
    b = synth.make_counts_csr((300, 130), (77, 40), n_labels=4, device="cpu", chunk=chunk)
    for g in (0, 1):
        c = b.X[g]
        assert c.indptr.dtype == torch.int64 and c.indices.dtype == torch.uint16 and c.values.dtype == torch.uint16
        m = sp.csr_matrix((c.values.numpy(), c.indices.numpy().astype(np.int64), c.indptr.numpy()), shape=c.shape)
        assert m.has_canonical_format and (m.data != 0).all()
        assert np.array_equal(m.toarray(), a.X[g].numpy().astype(np.int64))
        assert torch.equal(a.labels[g], b.labels[g])
