"""
CPU checks of the matrix builders and NumPy references that tests/test_gpu_kernels.py holds the kernels to: the edge
reference against the oracle's compress + edge step and the golden edge lists the reference itself produced, and the
builders against the row shapes they promise.
"""
import numpy as np
import pytest
import scipy.sparse as sp

import test_gpu_kernels as K


def _golden_map(g):
    n = len(g['lengths'])
    m = sp.coo_matrix((g['map_data'], (g['map_row'], g['map_col'])), shape=(n, n), dtype=np.uint32).tocsr()
    m.sort_indices()
    return n, m


def _oracle_edges(bal_coo, mask):
    from oracle import oracle
    return oracle.graph_edges(oracle.compress(bal_coo, mask))


def test_staged_edge_reference_matches_the_oracle(golden):
    g = golden
    n = len(g['lengths'])
    bal = sp.csr_matrix((g['bal_data'], g['bal_indices'], g['bal_indptr']), shape=(n, n))
    want = K.ref_compress(bal.indptr, bal.indices, bal.data, g['mask'])
    scl = K.ref_scale(want['vmax'])
    u, v, w, oscl = _oracle_edges(bal.tocoo(), g['mask'])
    assert scl == oscl == float(g['scl'])
    assert np.array_equal(want['u'], u) and np.array_equal(want['v'], v)
    assert np.array_equal(want['u'], g['edge_u']) and np.array_equal(want['v'], g['edge_v'])
    assert np.max(np.abs(want['w_unscaled'] * scl - w) / w) <= 1e-15
    assert want['n_accepted'] == int(g['sub_n']) and want['n_kept'] == int(g['sub_nnz'])


def test_fused_edge_reference_matches_the_oracle(golden):
    """Counts, sites and the golden x: the fused value x_i ((c (1/(s_i s_j))) x_j) is the oracle's site normalisation
    followed by its x_i (a_ij x_j), so u and v are the oracle's and w agrees to 1e-15."""
    from oracle import oracle
    g = golden
    n, m = _golden_map(g)
    sites = g['sites'].copy()
    sites[::7] = 0
    x = g['kr_x']
    vals = K.ref_fused_values(m.indptr, m.indices, m.data, sites, x)
    want = K.ref_compress(m.indptr, m.indices, vals, g['mask'])
    c = m.tocoo()
    a = oracle.norm_by_sites(c.row, c.col, c.data.astype(np.float64), oracle.get_sites(sites))
    bal = sp.coo_matrix((x[c.row] * (a * x[c.col]), (c.row, c.col)), shape=(n, n))
    u, v, w, scl = _oracle_edges(bal, g['mask'])
    assert np.array_equal(want['u'], u) and np.array_equal(want['v'], v)
    assert np.max(np.abs(want['w_unscaled'] * K.ref_scale(want['vmax']) - w) / w) <= 1e-15


def test_block_references_tile_the_whole_matrix():
    """The per-block references, concatenated over every tiling, give the whole-matrix results."""
    m = K.adversarial_counts()
    ip, idx = m['indptr'], m['indices']
    mask = K.adv_mask(m, 'alternating')
    vals = K.ref_fused_values(ip, idx, m['counts'], m['sites'], m['x'])
    whole = K.ref_compress(ip, idx, vals, mask)
    full_sig = K.ref_max_offdiag(ip, idx, m['counts'])
    from oracle import oracle
    assert np.array_equal(full_sig, oracle.max_offdiag(sp.csr_matrix((m['counts'], idx, ip), shape=(m['n'],) * 2)))
    for tile in K.TILINGS:
        parts, sig = [], []
        for lo, hi in K.tiling(tile):
            bip, bidx, s = K._block(m, lo, hi)
            parts.append(K.ref_compress(bip, bidx, vals[s], mask, lo))
            sig.append(K.ref_max_offdiag(bip, bidx, m['counts'][s], lo))
            assert np.array_equal(K.ref_fused_values(bip, bidx, m['counts'][s], m['sites'], m['x'], lo), vals[s])
        assert np.array_equal(np.concatenate(sig), full_sig)
        assert np.array_equal(np.concatenate([p['u'] for p in parts]), whole['u'])
        assert np.array_equal(np.concatenate([p['v'] for p in parts]), whole['v'])
        assert np.array_equal(np.concatenate([p['w_unscaled'] for p in parts]), whole['w_unscaled'])
        assert max(p['vmax'] for p in parts) == whole['vmax']


def test_adversarial_builder_shapes():
    m = K.adversarial_counts()
    n, ip, idx, cnt = m['n'], m['indptr'], m['indices'], m['counts']
    a = sp.csr_matrix((cnt, idx, ip), shape=(n, n))
    assert (a != a.T).nnz == 0 and cnt.dtype == np.uint32 and cnt.max() == K.U32_MAX
    assert np.all(np.diff(idx.astype(np.int64) + K.row_of_entry(ip) * n) > 0)          # sorted, unique
    assert K.seg_len(ip) == K.EDGE_SEG
    rows = m['rows']
    for lab, L, below, diag in K.ADV_ROWS:
        r = rows[lab]
        cols = idx[ip[r]:ip[r + 1]]
        assert len(cols) == L, lab
        assert np.count_nonzero(cols < r) == below, lab
        assert (r in cols) == (diag != 'none'), lab
        if diag == 'zero':
            assert cnt[ip[r] + below] == 0
    assert (m['sites'] == 0).any() and m['x'].min() < 2e-3 and m['x'].max() > 500


def test_dense_block_shapes():
    d = K.dense_block()
    ip, idx = d['indptr'], d['indices']
    T = K.seg_len(ip)
    assert T == d['T'] == 5415 and T % 2 == 1 and T % 32 != 0
    lens = np.diff(ip)
    assert set(lens.tolist()) == set(K.DENSE_LENGTHS)
    assert np.all(np.diff(idx.astype(np.int64) + K.row_of_entry(ip) * d['n']) > 0)
    for r in np.flatnonzero(lens == 9003)[:5]:
        assert idx[ip[r] + T] == K.DENSE_LO + r                    # the diagonal opens piece 2
    for r in np.flatnonzero(lens == 9002)[:5]:
        assert idx[ip[r] + T - 1] == K.DENSE_LO + r                # the diagonal closes piece 1


@pytest.mark.parametrize('case', ['symmetric', 'tol', 'half_tol', 'missing_mirror', 'explicit_zero',
                                  'long_row_entry'])
def test_asymmetry_reference(case):
    m = K.adversarial_counts()
    m['normed'] = K.ref_site_norm(m['indptr'], m['indices'], m['counts'], m['sites'])
    n, ip, idx, a, want = K._asym_case(m, case)
    assert K.ref_asymmetry_count(n, ip, idx, a, K.ASYM_TOL) == want
    assert K.dense_is_hermitian(n, ip, idx, a, K.ASYM_TOL) == (want == 0)
