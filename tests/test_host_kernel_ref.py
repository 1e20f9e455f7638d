"""CPU checks of oracle/kernel_ref.py, the float64 restatements the kernel-contract GPU tests compare against: wherever
the model oracle (oracle/cf_oracle.py, itself pinned to the reference's golden vectors) covers the same case, the
restatement must agree with it, so a GPU failure points at the kernel and not at the restatement."""
import numpy as np
import torch

from oracle import cf_oracle as O
from oracle import inputs
from oracle import kernel_ref as K
from oracle import philox as P


def _adj(seed=3):
    rows, cols = inputs.bipartite_edges(120, 90, 1500, seed)
    return O.normalized_adjacency(rows, cols, 120, 90)


def _csr(adj, owned=None):
    """kernel_ref CSR dict of the rows ``owned`` (global ids, ascending; default all), with rev over the full CSR."""
    n = adj.n
    full_ptr = np.zeros(n + 1, dtype=np.int64)
    full_ptr[1:] = np.cumsum(np.bincount(adj.rows, minlength=n))
    key = adj.rows * n + adj.cols
    rev = np.searchsorted(key, adj.cols * n + adj.rows)
    assert np.array_equal(key[rev], adj.cols * n + adj.rows)
    if owned is None:
        return dict(rowptr=full_ptr, colidx=adj.cols.astype(np.int32), vals=adj.vals, rows=np.arange(n), rev=rev, n=n)
    sel = np.concatenate([np.arange(full_ptr[r], full_ptr[r + 1]) for r in owned])
    ptr = np.concatenate([[0], np.cumsum(np.diff(full_ptr)[owned])])
    return dict(rowptr=ptr, colidx=adj.cols[sel].astype(np.int32), vals=adj.vals[sel], rows=np.asarray(owned), rev=None, n=n)


def _args(dim, V=1, **kw):
    a = dict(dim=dim, n_views=V, in_views=1, transpose=0, reduce_views=0, sum_src_views=[], reg_coef=0.0, reg_coef_dev=None,
             edge_mode=[0] * V, edge_keep=[1.0] * V, edge_scale=[1.0] * V, edge_mask=[None] * V, noise_mode=[0] * V, noise_eps=0.0,
             seed=[0] * V, edge_stream_id=0, noise_stream_id=0)
    a.update(kw)
    return a


def test_layer_sum_through_sum_src_is_lightgcn():
    """x_out of one layer feeds the next; sum_out = x + the running sum (sum_src, 1 view) -- the LightGCN layer sum."""
    adj = _adj()
    csr = _csr(adj)
    e0 = np.random.RandomState(0).randn(adj.n, 16).astype(np.float32)
    x, tot = e0[:, None, :], e0[:, None, :]
    for _ in range(3):
        r = K.propagate_layer(csr, _args(16, sum_src_views=[1]), x, sum_src=[tot])
        x, tot = r['x'], r['sum']
    want = O.lightgcn_embeds(adj.torch_coo(torch.float64), torch.from_numpy(e0).double(), 3).numpy()
    np.testing.assert_allclose(tot[:, 0], want, rtol=1e-12, atol=1e-12)
    # NodeDrop is applied to the layer-0 input: the restatement on the dropped rows is LightGCN of node_dropped(E0)
    keep = torch.from_numpy(np.random.RandomState(1).rand(adj.n) < 0.6)
    x0 = O.node_dropped(torch.from_numpy(e0).double(), keep).numpy()
    r = K.propagate_layer(csr, _args(16, sum_src_views=[1]), x0[:, None, :], sum_src=[x0[:, None, :]])
    np.testing.assert_allclose(r['sum'][:, 0], O.lightgcn_embeds(adj.torch_coo(torch.float64), torch.from_numpy(x0), 1).numpy(), rtol=1e-12, atol=1e-12)


def test_noise_term_is_simgcl_perturbation():
    adj = _adj(4)
    csr = _csr(adj)
    rs = np.random.RandomState(2)
    e0 = rs.randn(adj.n, 12).astype(np.float32)
    us = [rs.rand(adj.n, 12).astype(np.float32) for _ in range(2)]
    x, tot = e0[:, None, :], e0[:, None, :]
    for k in range(2):
        r = K.propagate_layer(csr, _args(12, sum_src_views=[1], noise_mode=[2], noise_eps=0.3), x, sum_src=[tot], noise_u=[us[k]])
        x, tot = r['x'], r['sum']
    want = O.simgcl_embeds(adj.torch_coo(torch.float64), torch.from_numpy(e0).double(), 2, float(np.float32(0.3)),
                           [torch.from_numpy(u).double() for u in us]).numpy()
    np.testing.assert_allclose(tot[:, 0], want, rtol=1e-12, atol=1e-12)
    # noise_mode 1 draws the same uniforms as the numpy Philox restatement
    seed = 0xDEADBEEF12345
    a1 = _args(12, noise_mode=[1], noise_eps=0.3, seed=[seed], noise_stream_id=5)
    a2 = _args(12, noise_mode=[2], noise_eps=0.3)
    np.testing.assert_array_equal(K.propagate_layer(csr, a1, e0[:, None, :])['x'],
                                  K.propagate_layer(csr, a2, e0[:, None, :], noise_u=[P.noise_uniform(seed, 5, adj.n, 12)])['x'])


def test_edge_masks_are_edge_drop_forward_and_transposed():
    adj = _adj(5)
    csr = _csr(adj)
    rs = np.random.RandomState(3)
    x = rs.randn(adj.n, 8).astype(np.float32)
    keep = 0.7
    a_d = lambda m: O.edge_dropped(adj, m, keep, True, torch.float64)
    mask = rs.rand(adj.nnz) < keep
    inj = _args(8, edge_mode=[2], edge_keep=[keep], edge_scale=[1 / keep], edge_mask=[mask.astype(np.uint8)])
    got = K.propagate_layer(csr, inj, x[:, None, :])
    np.testing.assert_allclose(got['x'][:, 0], torch.spmm(a_d(mask), torch.from_numpy(x).double()).numpy(), rtol=1e-6, atol=1e-12)
    assert np.array_equal(got['keep'][0], mask)
    got_t = K.propagate_layer(csr, dict(inj, transpose=1), x[:, None, :])
    np.testing.assert_allclose(got_t['x'][:, 0], (a_d(mask).to_dense().T @ torch.from_numpy(x).double()).numpy(), rtol=1e-6, atol=1e-12)
    # edge_mode 1: the keep test of the Philox restatement, keyed (row, col) forward and (col, row) transposed
    seed = 77
    rng = _args(8, edge_mode=[1], edge_keep=[keep], edge_scale=[1 / keep], seed=[seed], edge_stream_id=2)
    m1 = P.edge_keep(seed, 2, adj.rows, adj.cols, keep)
    np.testing.assert_allclose(K.propagate_layer(csr, rng, x[:, None, :])['x'][:, 0],
                               torch.spmm(a_d(m1), torch.from_numpy(x).double()).numpy(), rtol=1e-6, atol=1e-12)
    np.testing.assert_allclose(K.propagate_layer(csr, dict(rng, transpose=1), x[:, None, :])['x'][:, 0],
                               (a_d(m1).to_dense().T @ torch.from_numpy(x).double()).numpy(), rtol=1e-6, atol=1e-12)


def test_views_residual_sum_src_views_and_reduction():
    """Per-view inputs, a residual, sum_src of 1 and of V views, then reduce_views with both regulariser rows: each view
    is the single-view statement on its own slices; the reduction is their sum plus reg_coef * reg_coef_dev * reg_src
    + reg_src2.  Restating only a subset of the rows gives those rows of the full result."""
    adj = _adj(6)
    csr = _csr(adj)
    rs = np.random.RandomState(4)
    V, d, n = 3, 8, adj.n
    x, res = rs.randn(n, V, d), rs.randn(n, V, d)
    s1, sv = rs.randn(n, 1, d), rs.randn(n, V, d)
    reg, reg2 = rs.randn(n, d), rs.randn(n, d)
    a = _args(d, V, in_views=V, sum_src_views=[1, V], edge_mode=[0, 1, 0], edge_keep=[1.0, 0.5, 1.0], edge_scale=[1.0, 2.0, 1.0],
              seed=[0, 9, 0], edge_stream_id=1)
    full = K.propagate_layer(csr, a, x, residual=res, sum_src=[s1, sv])
    A = adj.torch_coo(torch.float64).to_dense().numpy()
    m1 = P.edge_keep(9, 1, adj.rows, adj.cols, 0.5)
    A1 = O.edge_dropped(adj, m1, 0.5, True, torch.float64).to_dense().numpy()
    for v, Av in enumerate((A, A1, A)):
        xv = Av @ x[:, v] + res[:, v]
        np.testing.assert_allclose(full['x'][:, v], xv, rtol=1e-6, atol=1e-12)
        np.testing.assert_allclose(full['sum'][:, v], xv + s1[:, 0] + sv[:, v], rtol=1e-6, atol=1e-12)
    red = K.propagate_layer(csr, dict(a, reduce_views=1, reg_coef=2.0, reg_coef_dev=0.25), x, residual=res, sum_src=[s1, sv],
                            reg_src=reg, reg_src2=reg2)
    np.testing.assert_allclose(red['sum'], full['sum'].sum(1) + 0.5 * reg + reg2, rtol=1e-12, atol=1e-12)
    owned = np.concatenate([np.arange(10, 50), np.arange(150, 200)])
    part = K.propagate_layer(_csr(adj, owned), a, x, residual=res, sum_src=[s1, sv])
    np.testing.assert_array_equal(part['x'], full['x'][owned])


def test_tf32_rounding_tile_permutation_and_split_order():
    one = np.float32(1.0)
    t = lambda k: np.float32(2.0 ** -k)
    x = np.array([one, one + t(11), one + t(12), -(one + t(11)), one + t(11) + t(20), np.float32(-3.0) * t(100), 0.0], dtype=np.float32)
    want = np.array([1.0, 1.0 + 2 ** -10, 1.0, -(1.0 + 2 ** -10), 1.0 + 2 ** -10, -3.0 * 2 ** -100, 0.0], dtype=np.float32)
    np.testing.assert_array_equal(K.tf32_rna(x), want)                    # to nearest, ties away from zero
    y = np.random.RandomState(5).randn(1000).astype(np.float32)
    hi, lo = K.tf32_split(y)
    assert ((hi.view(np.uint32) | lo.view(np.uint32)) & 0x1FFF == 0).all()
    assert (np.abs(hi.astype(np.float64) + lo - y) <= 2.0 ** -21 * np.abs(y)).all()
    tab = np.arange(128 * 3, dtype=np.float32).reshape(128, 3)
    tiles = K.k_major_tiles(tab)
    assert tiles.shape == (2, 3, 64) and tiles[1, 2, 5] == tab[64 + 1 + 16, 2]      # q = 5 -> c = 1 + 16
    assert K.split_tiles(64 * 9 + 1, 3) == [(0, 3), (3, 6), (6, 10)]
