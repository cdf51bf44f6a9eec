"""Expression-matrix ingestion (scope row f4): the product's C++ readers (plaid_b200/csrc/matio.cu, host
code, no GPU needed) against independent decoders — the oracle's RDX reader, scipy.io.mmread — on generated
files, among them one holding the contents of the reference's bundled fixture (tests/golden)."""
import gzip
import os

import numpy as np
import pytest
import scipy.io
import scipy.sparse as sp

import plaid_b200 as pb
from plaid_b200 import _lib as L
from oracle import rdata


def _rand_csc(P, N, density, seed, integer=False):
    rng = np.random.default_rng(seed)
    m = sp.random(P, N, density=density, format="csc", random_state=rng, data_rvs=lambda k: rng.normal(size=k))
    if integer:
        m.data = np.floor(np.abs(m.data) * 5) + 1
    m.sort_indices()
    return m


def _same(a: pb.NamedMatrix, m, rn, cn):
    b = a.mat
    assert b.shape == m.shape
    assert np.array_equal(b.indptr, m.indptr) and np.array_equal(b.indices, m.indices)
    assert np.array_equal(b.data, m.data)  # bit-exact: XDR doubles / decimal text that round-trips
    assert a.rownames == (list(rn) if rn is not None else None)
    assert a.colnames == (list(cn) if cn is not None else None)


def test_pbmc3k_fixture_contents_round_trip(tmp_path, fixture_mats, golden):
    """The contents of the reference's inst/extdata/pbmc3k-50cells.rda (dgCMatrix X, 7728 x 50, with its gene and
    barcode names, plus the character vector celltype), as decoded into tests/golden/pbmc3k50_hallmarks.npz, written
    by oracle.rdata.write_rda.  The R-written file itself is not part of the repository: this pins the reader on the
    reference's values and names, not on the exact bytes R's save() emits."""
    m, rn, cn = fixture_mats[:3]
    celltype = [str(s) for s in golden["celltype"]]
    path = str(tmp_path / "pbmc3k-50cells.rda")
    rdata.write_rda(path, {"X": (m, rn, cn), "celltype": celltype})
    assert rdata.read_rda(path)["celltype"] == celltype  # the writer's character vector, by the independent reader
    _same(pb.read_rda(path), m, rn, cn)
    _same(pb.read_rda(path, "X"), m, rn, cn)
    with pytest.raises(L.PlaidGpuError, match="celltype"):
        pb.read_rda(path, "celltype")  # a character vector, not a dgCMatrix


@pytest.mark.parametrize("version,compress,rds", [(3, True, False), (2, False, False), (3, True, True)])
def test_generated_rda_round_trip(tmp_path, version, compress, rds):
    m = _rand_csc(211, 37, 0.08, seed=version)
    m.data[m.indptr[5]:m.indptr[6]] = 0.0  # an empty column
    m.eliminate_zeros()
    rn = [f"g{k}" for k in range(211)]
    cn = [f"cell-{k}" for k in range(37)]
    other = _rand_csc(5, 4, 0.5, seed=9)
    path = str(tmp_path / "x.rda")
    rdata.write_rda(path, {"X": (m, rn, cn), "other": (other, None, None)}, version=version, compress=compress, rds=rds)
    if not rds:  # the writer is itself checked by the oracle's independent reader
        back = rdata.read_rda(path)
        assert np.array_equal(np.asarray(back["X"]["x"]), m.data)
    _same(pb.read_rda(path), m, rn, cn)
    if not rds:
        _same(pb.read_rda(path, "other"), other, None, None)
        with pytest.raises(L.PlaidGpuError, match="no object named"):
            pb.read_rda(path, "nope")


def test_rda_errors(tmp_path):
    p = tmp_path / "bad.rda"
    p.write_bytes(b"not an R file")
    with pytest.raises(L.PlaidGpuError, match="not an R save"):
        pb.read_rda(str(p))
    with pytest.raises(L.PlaidGpuError, match="cannot open"):
        pb.read_rda(str(tmp_path / "missing.rda"))
    good = tmp_path / "ok.rda"
    rdata.write_rda(str(good), {"X": (_rand_csc(30, 6, 0.3, seed=1), None, None)}, compress=False)
    raw = good.read_bytes()
    (tmp_path / "cut.rda").write_bytes(raw[:len(raw) // 2])
    with pytest.raises(L.PlaidGpuError, match="unexpected end"):
        pb.read_rda(str(tmp_path / "cut.rda"))
    gz = gzip.compress(raw)
    (tmp_path / "cut.gz.rda").write_bytes(gz[:len(gz) // 2])
    with pytest.raises(L.PlaidGpuError, match="corrupt gzip"):
        pb.read_rda(str(tmp_path / "cut.gz.rda"))


def _write_mtx(path, m, field="real", shuffle_seed=None, comments=True):
    coo = m.tocoo()
    order = np.arange(coo.nnz)
    if shuffle_seed is not None:
        order = np.random.default_rng(shuffle_seed).permutation(coo.nnz)
    lines = [f"%%MatrixMarket matrix coordinate {field} general"]
    if comments:
        lines += ["%metadata_json: {\"software_version\": \"test\"}", "%"]
    lines.append(f"{m.shape[0]} {m.shape[1]} {coo.nnz}")
    for k in order:
        if field == "pattern":
            lines.append(f"{coo.row[k] + 1} {coo.col[k] + 1}")
        elif field == "integer":
            lines.append(f"{coo.row[k] + 1} {coo.col[k] + 1} {int(coo.data[k])}")
        else:
            lines.append(f"{coo.row[k] + 1} {coo.col[k] + 1} {float(coo.data[k])!r}")
    text = "\n".join(lines) + "\n"
    if str(path).endswith(".gz"):
        with gzip.open(path, "wt") as fh:
            fh.write(text)
    else:
        with open(path, "w") as fh:
            fh.write(text)


def test_mtx_matches_scipy(tmp_path):
    m = _rand_csc(301, 58, 0.05, seed=4)
    for name, kw in [("a.mtx", {}), ("b.mtx.gz", dict(shuffle_seed=3)), ("c.mtx", dict(comments=False))]:
        path = str(tmp_path / name)
        _write_mtx(path, m, **kw)
        ref = sp.csc_matrix(scipy.io.mmread(path, spmatrix=True))
        ref.sort_indices()
        _same(pb.read_mtx(path), ref, None, None)
        _same(pb.read_mtx(path), m, None, None)  # repr() round-trips doubles exactly
    mi = _rand_csc(120, 40, 0.1, seed=5, integer=True)
    _write_mtx(str(tmp_path / "i.mtx"), mi, field="integer", shuffle_seed=1)
    _same(pb.read_mtx(str(tmp_path / "i.mtx")), mi, None, None)
    mp = mi.copy()
    mp.data[:] = 1.0
    _write_mtx(str(tmp_path / "p.mtx"), mi, field="pattern")
    _same(pb.read_mtx(str(tmp_path / "p.mtx")), mp, None, None)


def test_mtx_duplicates_crlf_and_errors(tmp_path):
    p = tmp_path / "d.mtx"
    p.write_text("%%MatrixMarket matrix coordinate real general\r\n3 2 4\r\n3 1 1.5\r\n1 1 2\r\n3 1 0.25\r\n2 2 -1e-3\r\n")
    X = pb.read_mtx(str(p)).mat
    assert np.array_equal(X.toarray(), np.array([[2.0, 0.0], [0.0, -1e-3], [1.75, 0.0]]))
    assert np.array_equal(X.indices, [0, 2, 1])
    s = tmp_path / "s.mtx"
    s.write_text("%%MatrixMarket matrix coordinate integer symmetric\n3 3 3\n1 1 4\n3 1 2\n3 2 7\n")
    assert np.array_equal(pb.read_mtx(str(s)).mat.toarray(), np.array([[4, 0, 2], [0, 0, 7], [2, 7, 0]], dtype=float))
    for text, msg in [("hello\n", "banner"), ("%%MatrixMarket matrix array real general\n2 2\n1\n2\n3\n4\n", "coordinate"),
                      ("%%MatrixMarket matrix coordinate real general\n2 2 2\n1 1 1.0\n", "truncated"),
                      ("%%MatrixMarket matrix coordinate real general\n2 2 1\n3 1 1.0\n", "out of range"),
                      # a non-square "symmetric" file: the mirrored entry (col = row - 1 >= N) used to corrupt the heap
                      ("%%MatrixMarket matrix coordinate real symmetric\n5 2 2\n5 1 1.0\n4 2 2.0\n", "square")]:
        b = tmp_path / "bad.mtx"
        b.write_text(text)
        with pytest.raises(L.PlaidGpuError, match=msg):
            pb.read_mtx(str(b))


def test_10x_directory(tmp_path):
    m = _rand_csc(50, 12, 0.2, seed=8, integer=True)
    d = tmp_path / "filtered_feature_bc_matrix"
    d.mkdir()
    _write_mtx(str(d / "matrix.mtx.gz"), m, field="integer")
    genes = [f"SYM{k}" for k in range(50)]
    genes[7] = genes[3]  # duplicated symbol: kept as is
    with gzip.open(d / "features.tsv.gz", "wt") as fh:
        fh.write("".join(f"ENSG{k:011d}\t{g}\tGene Expression\n" for k, g in enumerate(genes)))
    with gzip.open(d / "barcodes.tsv.gz", "wt") as fh:
        fh.write("".join(f"AAAC{k:04d}-1\n" for k in range(12)))
    X = pb.read_10x(str(d))
    _same(X, m, genes, [f"AAAC{k:04d}-1" for k in range(12)])
    d2 = tmp_path / "v2"  # CellRanger 2 layout: genes.tsv, uncompressed
    d2.mkdir()
    _write_mtx(str(d2 / "matrix.mtx"), m, field="integer")
    (d2 / "genes.tsv").write_text("".join(f"ENSG{k:011d}\t{g}\n" for k, g in enumerate(genes)))
    (d2 / "barcodes.tsv").write_text("".join(f"B{k}\n" for k in range(12)))
    _same(pb.read_10x(str(d2)), m, genes, [f"B{k}" for k in range(12)])
    (d2 / "barcodes.tsv").write_text("B0\n")
    with pytest.raises(L.PlaidGpuError, match="barcodes"):
        pb.read_10x(str(d2))
    with pytest.raises(L.PlaidGpuError, match="no matrix.mtx"):
        pb.read_10x(str(tmp_path))


def test_mtx_large_file_is_parsed_in_slices(tmp_path):
    """> 8 MB of entry lines: the parser cuts the text into per-thread slices at line ends; entry order (and
    with it the summation order of duplicates) must be that of the file"""
    rng = np.random.default_rng(11)
    P, N, nz = 5000, 900, 700_000
    r = rng.integers(1, P + 1, size=nz)
    c = rng.integers(1, N + 1, size=nz)
    v = np.round(rng.normal(size=nz), 3)
    path = str(tmp_path / "big.mtx")
    with open(path, "w") as fh:
        fh.write(f"%%MatrixMarket matrix coordinate real general\n{P} {N} {nz}\n")
        np.savetxt(fh, np.column_stack([r, c, v]), fmt="%d %d %.3f")
    assert os.path.getsize(path) > (8 << 20)
    got = pb.read_mtx(path).mat
    # reference: stable bucket by column, then stable sort by row, duplicates summed left to right
    order = np.lexsort((np.arange(nz), r, c))
    rr, cc, vv = r[order] - 1, c[order] - 1, v[order]
    first = np.ones(nz, dtype=bool)
    first[1:] = (rr[1:] != rr[:-1]) | (cc[1:] != cc[:-1])
    starts = np.flatnonzero(first)
    sums = np.array([np.add.reduce(vv[a:b]) if b - a < 3 else float(np.cumsum(vv[a:b])[-1])
                     for a, b in zip(starts, np.append(starts[1:], nz))])
    assert np.array_equal(got.indices, rr[first]) and np.array_equal(np.diff(got.indptr), np.bincount(cc[first], minlength=N))
    assert np.array_equal(got.data, sums)
