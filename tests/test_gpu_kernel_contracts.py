"""Kernel contracts through the C ABI (ctypes), launch variant by launch variant, against the float64 restatements of
include/sslrec_b200.h in oracle/kernel_ref.py:

  ssl_propagate_layer     a seeded set of configurations that reaches every (G, V, MODE, VM) template instance in both
                          directions on one graph with rows of degree 0, 1, 128, 129, 256, 257 and a hub of 5 200 entries;
                          plus the bit-exact relations between variants, the two-range plan, the peer stores and the
                          argument checks
  ssl_spmm_exact          float64, the sequential fp32 FMA chain, and ssl_propagate_layer on rows that are never split
  ssl_rows_normalize      all four norm modes: rinv, gather, scale, padding rows, the K-major tile copy, the tf32 split
  ssl_softmax_gemm[_tf32x3]  every n_split partition checked split by split on ragged shapes, colscale with zeros, and
                          finite garbage in the padding rows of the streamed operand
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import kernel_ref as K

pytestmark = pytest.mark.gpu

DEV = 'cuda'
SSL_E_ARG = -1
LOG2E = 1.4426950408889634


def _lib():
    from sslrec_b200 import _lib
    return _lib


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ================================================================================================================
# the graph: rows of degree 0, 1, 128, 129 (the first split row), 256, 257 and a hub of ~20 segments
# ================================================================================================================

N_USER, N = 1400, 2400            # side_split = N_USER: the work list runs the rows below it first
SPECIAL = {0: 5200, 1: 0, 2: 1, 3: 128, 4: 129, 5: 256, 6: 257, 1400: 257, 1401: 256, 1402: 129, 1403: 128, 1404: 1, 1405: 0,
           1406: 300, 2399: 130}
RANGES = ((0, 700), (1500, 2100))  # the two-range plan: the hub and a share of both sides


def _build_graph():
    """Symmetric multigraph in CSR order (row, col, edge id): every undirected edge is stored as (a, b) and (b, a) with one
    value, so rev (the position of the reverse entry) is a true involution even where a pair repeats (the hub has more
    entries than there are nodes)."""
    rs = np.random.RandomState(2024)
    background = np.setdiff1d(np.arange(N), list(SPECIAL))
    ea, eb = [], []
    for node, deg in SPECIAL.items():
        ea.append(np.full(deg, node))
        eb.append(rs.choice(background, deg))
    m = 9000
    a, b = rs.choice(background, m), rs.choice(background, m)
    keep = a != b
    ea.append(a[keep])
    eb.append(b[keep])
    ea, eb = np.concatenate(ea), np.concatenate(eb)
    val = rs.uniform(0.02, 0.3, ea.shape[0]).astype(np.float32)
    ne = ea.shape[0]
    rows, cols = np.concatenate([ea, eb]), np.concatenate([eb, ea])
    eid = np.concatenate([np.arange(ne), np.arange(ne)])
    direction = np.concatenate([np.zeros(ne, np.int64), np.ones(ne, np.int64)])
    order = np.lexsort((direction, eid, cols, rows))
    rows, cols, eid, direction = rows[order], cols[order], eid[order], direction[order]
    pos = np.empty((ne, 2), dtype=np.int64)
    pos[eid, direction] = np.arange(2 * ne)
    rev = pos[eid, 1 - direction]
    rowptr = np.zeros(N + 1, dtype=np.int64)
    rowptr[1:] = np.cumsum(np.bincount(rows, minlength=N))
    deg = np.diff(rowptr)
    assert all(deg[k] == v for k, v in SPECIAL.items()) and np.array_equal(rev[rev], np.arange(2 * ne))
    return dict(rowptr=rowptr, colidx=cols.astype(np.int32), vals=val[eid], rows=np.arange(N), rev=rev, n=N, row_ids=rows)


class _RawPlan:
    """ssl_plan_create on a ready CSR with the caller's rev array (GraphPlan derives rev by a search that assumes unique pairs)."""

    def __init__(self, g):
        L = _lib()
        self.colidx = torch.from_numpy(g['colidx']).to(DEV)
        self.vals = torch.from_numpy(g['vals']).to(DEV)
        self.rev = torch.from_numpy(g['rev'].astype(np.int32)).to(DEV)
        self.h_rowptr = np.ascontiguousarray(g['rowptr'].astype(np.int32))
        self.handle = C.c_void_p()
        L.check(L.lib.ssl_plan_create(C.byref(self.handle), self.h_rowptr.ctypes.data, self.colidx.data_ptr(), self.vals.data_ptr(),
                                      self.rev.data_ptr(), N, N, self.colidx.numel(), 0, N_USER, _stream()), 'ssl_plan_create')

    def stats(self):
        out = (C.c_int64 * 4)()
        _lib().check(_lib().lib.ssl_plan_stats(self.handle, out))
        return list(out)

    def close(self):
        _lib().lib.ssl_plan_destroy(self.handle)


@pytest.fixture(scope='module')
def graph():
    from sslrec_b200.graph import GraphPlan
    g = _build_graph()
    full = _RawPlan(g)
    ranged = GraphPlan(g['row_ids'], g['colidx'], g['vals'], N, torch.device(DEV), row_ranges=RANGES, side_split=N_USER)
    items, split_rows, segments, max_deg = full.stats()
    assert max_deg == 5200 and split_rows == 1 + sum(d > 128 for d in np.diff(g['rowptr'])[1:]) and segments >= 20 + 2 * (split_rows - 1)
    yield dict(g=g, full=full, ranged=ranged)
    full.close()


# ================================================================================================================
# configurations and the dispatch rule of ssl_propagate_layer
# ================================================================================================================

DIMS_BY_G = {4: (4, 8, 12, 16), 8: (20, 32), 16: (48, 64), 32: (100, 128)}
DIMS = sorted(d for ds in DIMS_BY_G.values() for d in ds)


def lane_group(dim):
    q = dim // 4
    return 4 if q <= 4 else 8 if q <= 8 else 16 if q <= 16 else 32


def instance(dim, n_views, in_views, masked, reduce_views, view_major_opt):
    """The template instance prop_kernel<G, V, MODE, VM> that ssl_propagate_layer launches for these arguments."""
    mode = 2 if masked else (0 if in_views == 1 else 1)
    vm = bool(view_major_opt) and n_views > 1 and not reduce_views and (mode == 2 or in_views == n_views)
    return (lane_group(dim), 1 if vm else n_views, mode, vm)


def cfg_instance(c):
    return instance(c['dim'], c['V'], c['in_views'], any(m != 0 for m in c['edge_mode']), c['reduce'], c['vm_opt'])


def reachable_instances():
    out = set()
    for dim in DIMS:
        for V in range(1, 5):
            for iv in sorted({1, V}):
                for masked in (False, True):
                    for red in (False, True):
                        for opt in (False, True):
                            out.add(instance(dim, V, iv, masked, red, opt))
    return out


def make_configs(seed=20260417):
    """One configuration per (reachable instance, transpose), every other field drawn from one seeded stream."""
    rs = np.random.RandomState(seed)
    dim_turn = {g: 0 for g in DIMS_BY_G}
    cfgs = []
    for (G, Vi, mode, vm) in sorted(reachable_instances()):
        for transpose in (0, 1):
            dim = DIMS_BY_G[G][dim_turn[G] % len(DIMS_BY_G[G])]
            dim_turn[G] += 1
            V = int(rs.randint(2, 5)) if vm else Vi
            in_views = 1 if mode == 0 else V if mode == 1 else int(rs.choice(sorted({1, V})))
            edge_mode = [0] * V
            if mode == 2:
                edge_mode = [int(m) for m in rs.choice(3, V, p=[0.3, 0.4, 0.3])]
                if not any(edge_mode):
                    edge_mode[int(rs.randint(V))] = int(rs.randint(1, 3))
            keep = [float(np.round(rs.uniform(0.3, 0.95), 3)) for _ in range(V)]
            scale = [float(rs.choice([1.0, 1.0 / k, rs.uniform(0.5, 2.0)])) for k in keep]
            sum_out = bool(rs.rand() < 0.6)
            reduce = False
            opt = True if vm else bool(rs.rand() < 0.5)
            if not vm and opt and instance(dim, V, in_views, mode == 2, False, True)[3]:
                reduce = True                       # the option is on but a view reduction keeps the interleaved kernel
            elif not vm and sum_out and V > 1:
                reduce = bool(rs.rand() < 0.3)
            sum_out = sum_out or reduce
            x_out = bool(rs.rand() < 0.6) or not sum_out
            n_src = int(rs.randint(0, 7)) if sum_out else 0
            c = dict(idx=len(cfgs), dim=dim, V=V, in_views=in_views, transpose=transpose, vm_opt=opt, reduce=reduce,
                     edge_mode=edge_mode, keep=keep, scale=scale,
                     noise_mode=[int(m) for m in rs.choice(3, V, p=[0.5, 0.25, 0.25])], eps=float(np.round(rs.uniform(0.05, 0.5), 3)),
                     residual=bool(rs.rand() < 0.5), x_out=x_out, sum_out=sum_out,
                     sum_src_views=[int(rs.choice(sorted({1, V}))) for _ in range(n_src)],
                     reg=reduce and bool(rs.rand() < 0.7), reg_dev=bool(rs.rand() < 0.5), reg2=reduce and bool(rs.rand() < 0.5),
                     reg_coef=float(np.round(rs.uniform(-2, 2), 3)),
                     seed=[int(s) for s in rs.randint(0, 2 ** 62, V, dtype=np.int64)],
                     seed_dev=[int(s) if rs.rand() < 0.25 else None for s in rs.randint(0, 2 ** 62, V, dtype=np.int64)],
                     edge_stream=int(rs.randint(0, 2 ** 32, dtype=np.int64)), noise_stream=int(rs.randint(0, 2 ** 32, dtype=np.int64)),
                     data_seed=int(rs.randint(0, 2 ** 31)))
            c['reg_dev'] = c['reg_dev'] and c['reg']
            assert cfg_instance(c) == (G, Vi, mode, vm)
            cfgs.append(c)
    return cfgs


CONFIGS = make_configs()


def _cfg_id(c):
    G, V, M, vm = cfg_instance(c)
    return f"c{c['idx']:03d}-G{G}V{V}M{M}{'VM' if vm else ''}-T{c['transpose']}-d{c['dim']}"


def test_configurations_reach_every_instance_in_both_directions():
    want = {(i, t) for i in reachable_instances() for t in (0, 1)}
    got = {(cfg_instance(c), c['transpose']) for c in CONFIGS}
    print('reached (G, V, MODE, VM) instances:', sorted(reachable_instances()))
    assert got == want, sorted(want - got)
    assert len(reachable_instances()) == 52                   # 4 lane groups x (11 interleaved + 2 view-major)
    assert {c['dim'] for c in CONFIGS} == set(DIMS)
    assert max(len(c['sum_src_views']) for c in CONFIGS) == 6 and any(c['reg_dev'] and c['reg2'] for c in CONFIGS)


# ================================================================================================================
# launching a configuration
# ================================================================================================================

def _data(c, g):
    """Seeded host inputs of a configuration (float32 / uint8)."""
    rs = np.random.RandomState(c['data_seed'])
    V, d, nnz = c['V'], c['dim'], g['colidx'].shape[0]
    f = lambda *s: (rs.randn(*s) * 0.5).astype(np.float32)
    return dict(x_in=f(N, c['in_views'], d), residual=f(N, V, d) if c['residual'] else None,
                sum_src=[f(N, sv, d) for sv in c['sum_src_views']],
                reg_src=f(N, d) if c['reg'] else None, reg_coef_dev=np.float32(rs.uniform(-1, 1)) if c['reg_dev'] else None,
                reg_src2=f(N, d) if c['reg2'] else None,
                noise_u=[rs.rand(N, d).astype(np.float32) if m == 2 else None for m in c['noise_mode']],
                edge_mask=[(rs.rand(nnz) < k).astype(np.uint8) if m == 2 else None for m, k in zip(c['edge_mode'], c['keep'])])


def _dev(x):
    return None if x is None else torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def launch(handle, c, data, view_major, fill=float('nan'), n_peers=0):
    """One ssl_propagate_layer call -> (x_out [N, V, d] | None, sum_out | None, peer tables) as host arrays."""
    L = _lib()
    V, d = c['V'], c['dim']
    keep_alive = []

    def ptr(x):
        t = _dev(x) if isinstance(x, np.ndarray) else x
        if t is None:
            return None
        keep_alive.append(t)
        return t.data_ptr()
    a = L.PropArgs()
    a.dim, a.n_views, a.in_views, a.transpose = d, V, c['in_views'], c['transpose']
    a.x_in = ptr(data['x_in'])
    x_out = torch.full((N, V, d), fill, device=DEV) if c['x_out'] else None
    sum_out = torch.full((N, d) if c['reduce'] else (N, V, d), fill, device=DEV) if c['sum_out'] else None
    a.x_out, a.sum_out = ptr(x_out), ptr(sum_out)
    a.residual = ptr(data['residual'])
    a.reduce_views, a.n_sum_src = int(c['reduce']), len(c['sum_src_views'])
    for i, (sv, src) in enumerate(zip(c['sum_src_views'], data['sum_src'])):
        a.sum_src[i], a.sum_src_views[i] = ptr(src), sv
    a.reg_coef, a.reg_src, a.reg_src2 = c['reg_coef'], ptr(data['reg_src']), ptr(data['reg_src2'])
    a.reg_coef_dev = ptr(None if data['reg_coef_dev'] is None else np.array([data['reg_coef_dev']], np.float32))
    for v in range(V):
        a.edge_mode[v], a.edge_keep[v], a.edge_scale[v] = c['edge_mode'][v], c['keep'][v], c['scale'][v]
        a.edge_mask[v] = ptr(data['edge_mask'][v])
        a.noise_mode[v], a.noise_u[v] = c['noise_mode'][v], ptr(data['noise_u'][v])
        a.seed[v] = c['seed'][v]
        if c['seed_dev'][v] is not None:
            a.seed_ptr[v] = ptr(np.array([c['seed_dev'][v]], np.int64))
    a.noise_eps, a.edge_stream_id, a.noise_stream_id = c['eps'], c['edge_stream'], c['noise_stream']
    peers = []
    a.n_peers = n_peers
    for q in range(n_peers):
        px = torch.full_like(x_out, -5.0) if x_out is not None else None
        ps = torch.full_like(sum_out, -5.0) if sum_out is not None else None
        a.x_out_peers[q], a.sum_out_peers[q] = ptr(px), ptr(ps)
        peers.append((px, ps))
    L.check(L.lib.ssl_set_option(b'prop_view_major', int(view_major)), 'ssl_set_option')
    try:
        L.check(L.lib.ssl_propagate_layer(handle, C.byref(a), _stream()), 'ssl_propagate_layer ' + _cfg_id(c))
    finally:
        L.check(L.lib.ssl_set_option(b'prop_view_major', 0), 'ssl_set_option')
    torch.cuda.synchronize()
    host = lambda t: None if t is None else t.cpu().numpy()
    return host(x_out), host(sum_out), [(host(px), host(ps)) for px, ps in peers]


def reference(c, g, data):
    a = dict(dim=c['dim'], n_views=c['V'], in_views=c['in_views'], transpose=c['transpose'], reduce_views=c['reduce'],
             sum_src_views=c['sum_src_views'], reg_coef=c['reg_coef'],
             reg_coef_dev=None if data['reg_coef_dev'] is None else float(data['reg_coef_dev']),
             edge_mode=c['edge_mode'], edge_keep=c['keep'], edge_scale=c['scale'], edge_mask=data['edge_mask'],
             noise_mode=c['noise_mode'], noise_eps=c['eps'], seed=[sd if sd is not None else s for s, sd in zip(c['seed'], c['seed_dev'])],
             edge_stream_id=c['edge_stream'], noise_stream_id=c['noise_stream'])
    return K.propagate_layer(g, a, data['x_in'], residual=data['residual'], sum_src=data['sum_src'], reg_src=data['reg_src'],
                             reg_src2=data['reg_src2'], noise_u=data['noise_u'])


def _close(got, ref, tol, what):
    err = np.abs(got.astype(np.float64) - ref)
    bad = ~(err <= tol)                                      # NaN (a row the kernel never wrote) fails
    assert not bad.any(), f'{what}: {bad.sum()} / {bad.size} off, first at {np.argwhere(bad)[0]}: got {got[bad][0]!r} want {ref[bad][0]!r}'


def check_against_reference(c, g, data, x_out, sum_out):
    """rtol 1e-5 plus an absolute floor of 2e-6 times the largest magnitude of the (row, view): the fp32 evaluation
    rounds every partial sum, so its error scales with sum |terms|, not with the (possibly cancelling) result.  The noise
    term follows sign(x): where |x| < 1e-6 max|x| the fp32 and fp64 signs may differ, so there the noise term is
    excluded from the check (twice its magnitude is added to the tolerance)."""
    r = reference(c, g, data)
    ambiguous = np.abs(r['pre']) < 1e-6 * np.abs(r['pre']).max()
    slack = np.where(ambiguous, 2 * r['noise_abs'], 0.0)
    if x_out is not None:
        floor = r['mag_x'].max(axis=2, keepdims=True)
        _close(x_out, r['x'], 1e-5 * np.abs(r['x']) + 2e-6 * floor + slack, 'x_out ' + _cfg_id(c))
    if sum_out is not None:
        floor = r['mag_sum'].max(axis=-1, keepdims=True)
        _close(sum_out, r['sum'], 1e-5 * np.abs(r['sum']) + 2e-6 * floor + (slack.sum(1) if c['reduce'] else slack), 'sum_out ' + _cfg_id(c))
    return r


def single_view(c, data, v):
    """The 1-view configuration of view v of c and its inputs (slices of the V-view tensors)."""
    pick = lambda xs: [xs[v]]
    c1 = dict(c, V=1, in_views=1, reduce=False, reg=False, reg2=False, reg_dev=False, edge_mode=pick(c['edge_mode']), keep=pick(c['keep']),
              scale=pick(c['scale']), noise_mode=pick(c['noise_mode']), seed=pick(c['seed']), seed_dev=pick(c['seed_dev']),
              sum_src_views=[1] * len(c['sum_src_views']))
    sl = lambda x, views: x[:, (0 if views == 1 else v):(0 if views == 1 else v) + 1, :]
    d1 = dict(data, x_in=sl(data['x_in'], c['in_views']), residual=None if data['residual'] is None else sl(data['residual'], c['V']),
              sum_src=[sl(s, sv) for s, sv in zip(data['sum_src'], c['sum_src_views'])], reg_src=None, reg_src2=None, reg_coef_dev=None,
              noise_u=pick(data['noise_u']), edge_mask=pick(data['edge_mask']))
    return c1, d1


def _same(a, b, what):
    assert a is not None and b is not None and a.shape == b.shape, what
    assert np.array_equal(a, b), f'{what}: {(a != b).sum()} elements differ, first at {np.argwhere(a != b)[0]}'


# ================================================================================================================
# propagation tests
# ================================================================================================================

@pytest.mark.parametrize('c', CONFIGS, ids=_cfg_id)
def test_propagation_variant_matches_float64_and_its_bit_exact_relatives(graph, c):
    g, plan = graph['g'], graph['full'].handle
    data = _data(c, g)
    vm = cfg_instance(c)[3]
    x_out, sum_out, _ = launch(plan, c, data, c['vm_opt'])
    r = check_against_reference(c, g, data, x_out, sum_out)
    # in-kernel keep tests: the launch with edge_mode 1 equals, bit for bit, edge_mode 2 with the restated mask injected
    # (transposed launches read mask[rev[p]]; rev is an involution, so the injected array is keep[rev])
    if 1 in c['edge_mode']:
        inj = dict(c, edge_mode=[2 if m == 1 else m for m in c['edge_mode']])
        masks = [(r['keep'][v][g['rev']] if c['transpose'] else r['keep'][v]).astype(np.uint8) if c['edge_mode'][v] == 1 else data['edge_mask'][v]
                 for v in range(c['V'])]
        xi, si, _ = launch(plan, inj, dict(data, edge_mask=masks), c['vm_opt'])
        for a_, b_, name in ((x_out, xi, 'x_out'), (sum_out, si, 'sum_out')):
            if a_ is not None:
                _same(a_, b_, f'{name}: RNG keep test vs its restated mask injected, {_cfg_id(c)}')
    # view-major and interleaved: every output element is the same FMA chain in both mappings
    if instance(c['dim'], c['V'], c['in_views'], 2 in c['edge_mode'] or 1 in c['edge_mode'], c['reduce'], True)[3]:
        xo, so, _ = launch(plan, c, data, not vm)
        for a_, b_, name in ((x_out, xo, 'x_out'), (sum_out, so, 'sum_out')):
            if a_ is not None:
                _same(a_, b_, f'{name}: view-major vs interleaved, {_cfg_id(c)}')
    # view v of the V-view launch is the 1-view launch of that view's spec
    if c['V'] > 1 and not c['reduce']:
        for v in range(c['V']):
            c1, d1 = single_view(c, data, v)
            x1, s1, _ = launch(plan, c1, d1, False)
            if x_out is not None:
                _same(x_out[:, v], x1[:, 0], f'x_out view {v} vs its 1-view launch, {_cfg_id(c)}')
            if sum_out is not None:
                _same(sum_out[:, v], s1[:, 0], f'sum_out view {v} vs its 1-view launch, {_cfg_id(c)}')


def test_relaunch_after_other_variants_is_bit_identical(graph):
    """Every configuration launched twice, the second time after all other variants ran on the same plan in another
    order: a split-row ticket or partial left behind by one variant would change the next launch that uses it."""
    import hashlib
    g, plan = graph['g'], graph['full'].handle
    digest = lambda outs: [None if t is None else hashlib.sha256(t.tobytes()).hexdigest() for t in outs]
    first = [digest(launch(plan, c, _data(c, g), c['vm_opt'])[:2]) for c in CONFIGS]
    for i in np.random.RandomState(5).permutation(len(CONFIGS)):
        again = digest(launch(plan, CONFIGS[i], _data(CONFIGS[i], g), CONFIGS[i]['vm_opt'])[:2])
        assert again == first[i], 'relaunch changed the output of ' + _cfg_id(CONFIGS[i])


@pytest.mark.parametrize('view_major', [False, True])
@pytest.mark.parametrize('transpose', [0, 1])
def test_two_range_plan_writes_only_its_rows(graph, transpose, view_major):
    """V = 4, dim 100 on the plan owning [0, 700) + [1500, 2100) (the hub and split rows included): the owned rows equal the
    full plan's bit for bit, every other row keeps its sentinel."""
    g = graph['g']
    rs = np.random.RandomState(7 + transpose)
    c = dict(CONFIGS[0], idx=900 + transpose, dim=100, V=4, in_views=4, transpose=transpose, vm_opt=view_major, reduce=False,
             edge_mode=[1, 0, 1, 1], keep=[0.5, 1.0, 0.7, 0.9], scale=[2.0, 1.0, 1.0, 1.3], noise_mode=[1, 2, 0, 1], eps=0.2,
             residual=True, x_out=True, sum_out=True, sum_src_views=[4, 1], reg=False, reg_dev=False, reg2=False,
             seed=[int(s) for s in rs.randint(0, 2 ** 62, 4, dtype=np.int64)], seed_dev=[None] * 4, data_seed=31 + transpose)
    data = _data(c, g)
    want = launch(graph['full'].handle, c, data, view_major)[:2]
    got = launch(graph['ranged'].handle, c, data, view_major, fill=-7.0)[:2]
    own = np.zeros(N, dtype=bool)
    for a0, a1 in RANGES:
        own[a0:a1] = True
    for w, t in zip(want, got):
        _same(t[own], w[own], 'owned rows of the two-range plan')
        assert (t[~own] == -7.0).all(), 'a row the plan does not own was written'


def test_seven_peer_tables_equal_the_own_table(graph):
    g, plan = graph['g'], graph['full'].handle
    base = [c for c in CONFIGS if c['V'] == 2 and not c['reduce']][0]
    c = dict(base, x_out=True, sum_out=True)
    red = dict([c_ for c_ in CONFIGS if c_['reduce']][0], x_out=True)
    for cc in (c, red):
        data = _data(cc, g)
        x_out, sum_out, peers = launch(plan, cc, data, cc['vm_opt'], n_peers=7)
        assert len(peers) == 7
        for px, ps in peers:
            _same(px, x_out, 'x_out peer table ' + _cfg_id(cc))
            _same(ps, sum_out, 'sum_out peer table ' + _cfg_id(cc))


def test_rejected_arguments_launch_nothing(graph):
    L = _lib()
    x = torch.zeros(N, 4, 132, device=DEV)
    out = torch.zeros(N, 4, 132, device=DEV)
    mask = torch.ones(graph['g']['colidx'].shape[0], dtype=torch.uint8, device=DEV)

    def args(**kw):
        a = L.PropArgs()
        a.dim, a.n_views, a.in_views, a.transpose = 64, 2, 1, 0
        a.x_in, a.x_out = x.data_ptr(), out.data_ptr()
        for k, v in kw.items():
            setattr(a, k, v)
        return a
    sum_bad = args(sum_out=out.data_ptr(), n_sum_src=1, n_views=3)
    sum_bad.sum_src[0], sum_bad.sum_src_views[0] = x.data_ptr(), 2
    inj = args(transpose=1)
    inj.edge_mode[0], inj.edge_mask[0], inj.edge_keep[0], inj.edge_scale[0] = 2, mask.data_ptr(), 0.5, 1.0
    cases = [('dim 6', graph['full'], args(dim=6)), ('dim 132', graph['full'], args(dim=132)), ('5 views', graph['full'], args(n_views=5)),
             ('reg_src without reduce_views', graph['full'], args(sum_out=out.data_ptr(), reg_src=x.data_ptr())),
             ('injected mask + transpose without rev', graph['ranged'], inj),
             ('sum_src_views 2 of 3 views', graph['full'], sum_bad)]
    torch.cuda.synchronize()
    n0 = L.launch_count()
    for what, plan, a in cases:
        assert L.lib.ssl_propagate_layer(plan.handle, C.byref(a), _stream()) == SSL_E_ARG, what
    assert L.launch_count() == n0
    good = args()
    L.check(L.lib.ssl_propagate_layer(graph['full'].handle, C.byref(good), _stream()))      # the same arguments, fixed, launch
    assert L.launch_count() == n0 + 1


# ================================================================================================================
# ssl_spmm_exact
# ================================================================================================================

@pytest.mark.parametrize('dim', [1, 3, 4, 33, 128])
def test_spmm_exact_float64_fma_chain_and_unsplit_propagation(graph, dim):
    import scipy.sparse as sp
    L = _lib()
    g = graph['g']
    rowptr = torch.from_numpy(g['rowptr'].astype(np.int32)).to(DEV)
    colidx, vals = graph['full'].colidx, graph['full'].vals
    xb = torch.randn(N, dim + 5, generator=torch.Generator().manual_seed(dim)).to(DEV)
    x = xb[:, 2:2 + dim]                                                   # strided rows, offset start
    yb = torch.full((N, dim + 3), -7.0, device=DEV)
    y = yb[:, 1:1 + dim]
    L.check(L.lib.ssl_spmm_exact(rowptr.data_ptr(), colidx.data_ptr(), vals.data_ptr(), N, x.data_ptr(), x.stride(0), dim, y.data_ptr(),
                                 y.stride(0), _stream()), 'ssl_spmm_exact')
    torch.cuda.synchronize()
    got, yh = y.cpu().numpy(), yb.cpu().numpy()
    assert (yh[:, 0] == -7.0).all() and (yh[:, 1 + dim:] == -7.0).all()
    xh = x.cpu().numpy()
    csr = lambda v: sp.csr_matrix((v, g['colidx'].copy(), g['rowptr'].copy()), shape=(N, N))     # copies: scipy may sort in place
    ref = csr(g['vals'].astype(np.float64)) @ xh.astype(np.float64)
    mag = csr(np.abs(g['vals'].astype(np.float64))) @ np.abs(xh.astype(np.float64))
    _close(got, ref, 1e-5 * np.abs(ref) + 1e-6 * mag, f'spmm_exact dim {dim}')
    chain = K.spmm_fma_chain(g['rowptr'], g['colidx'], g['vals'], xh)
    equal = float((got == chain).mean())
    print(f'spmm_exact dim {dim}: {equal:.6f} of the elements bit-equal to the sequential fp32 FMA chain')
    assert equal >= 0.9999, equal
    if dim % 4 == 0:            # rows of <= 128 entries are never split: ssl_propagate_layer evaluates the same chain
        xc = x.contiguous().cpu().numpy()[:, None, :]
        c = dict(CONFIGS[0], idx=990, dim=dim, V=1, in_views=1, transpose=0, reduce=False, edge_mode=[0], keep=[1.0], scale=[1.0],
                 noise_mode=[0], residual=False, x_out=True, sum_out=False, sum_src_views=[], reg=False, reg_dev=False, reg2=False,
                 seed=[0], seed_dev=[None])
        prop = launch(graph['full'].handle, c, dict(x_in=xc, residual=None, sum_src=[], reg_src=None, reg_coef_dev=None, reg_src2=None,
                                                     noise_u=[None], edge_mask=[None]), False)[0][:, 0]
        short = np.diff(g['rowptr']) <= 128
        assert np.array_equal(prop[short], got[short])
    # an empty launch succeeds and touches nothing
    n0 = L.launch_count()
    L.check(L.lib.ssl_spmm_exact(rowptr.data_ptr(), colidx.data_ptr(), vals.data_ptr(), 0, x.data_ptr(), x.stride(0), dim, y.data_ptr(),
                                 y.stride(0), _stream()))
    torch.cuda.synchronize()
    assert L.launch_count() == n0 and np.array_equal(yb.cpu().numpy(), yh)


# ================================================================================================================
# ssl_rows_normalize
# ================================================================================================================

def _u32(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize('norm_mode', [0, 1, 2, 3])
@pytest.mark.parametrize('n,dim', [(1, 4), (63, 36), (64, 64), (130, 128), (200, 20)])
def test_rows_normalize_contract(norm_mode, n, dim):
    L = _lib()
    rs = np.random.RandomState(n * 7 + dim + norm_mode)
    n_src = n + 5
    src = (rs.randn(n_src, dim + 4) * 0.7).astype(np.float32)
    src[3] = 0.0                                                           # an all-zero row, gathered at least once
    idx = rs.randint(0, n_src, n).astype(np.int64)
    idx[n // 2] = 3
    alpha = 1.7
    npad = (n + 63) // 64 * 64
    pitch = npad + 68
    xb = torch.from_numpy(src).to(DEV)
    x = xb[:, :dim]
    nan = float('nan')
    out = torch.full((npad + 64, dim), nan, device=DEV)
    out_t = torch.full((npad // 64 + 1, dim, 64), nan, device=DEV)
    rinv = torch.full((n + 8,), nan, device=DEV)
    hi, lo = torch.full((npad + 64, dim), nan, device=DEV), torch.full((npad + 64, dim), nan, device=DEV)
    thi, tlo = torch.full((dim, pitch), nan, device=DEV), torch.full((dim, pitch), nan, device=DEV)
    idx_d = torch.from_numpy(idx).to(DEV)
    L.check(L.lib.ssl_rows_normalize(x.data_ptr(), x.stride(0), idx_d.data_ptr(), n, dim, norm_mode, alpha, out.data_ptr(), out_t.data_ptr(),
                                     rinv.data_ptr(), hi.data_ptr(), lo.data_ptr(), thi.data_ptr(), tlo.data_ptr(), pitch, _stream()),
            'ssl_rows_normalize')
    torch.cuda.synchronize()
    out, out_t, rinv, hi, lo, thi, tlo = (t.cpu().numpy() for t in (out, out_t, rinv, hi, lo, thi, tlo))
    want, want_rinv = K.rows_normalize(src[:, :dim], idx, norm_mode, alpha)
    _close(rinv[:n], want_rinv, 2e-6 * want_rinv, 'rinv')
    assert np.isnan(rinv[n:]).all()
    _close(out[:n], want, 2e-6 * np.abs(want) + 1e-30, 'out')
    assert (out[n:npad] == 0).all() and np.isnan(out[npad:]).all()             # rows n .. ceil64(n) are zeros, nothing beyond
    _same(out_t[:npad // 64], K.k_major_tiles(out[:npad]), 'K-major tile copy')
    assert np.isnan(out_t[npad // 64:]).all()
    y = out[:npad]
    want_hi, want_lo = K.tf32_split(y)
    assert ((_u32(hi[:npad]) | _u32(lo[:npad])) & 0x1FFF == 0).all(), 'tf32 parts with low mantissa bits set'
    _same(_u32(hi[:npad]), _u32(want_hi), 'out_hi = tf32_rna(out)')
    _same(_u32(lo[:npad]), _u32(want_lo), 'out_lo = tf32_rna(out - out_hi)')
    assert np.isnan(hi[npad:]).all() and np.isnan(lo[npad:]).all()
    _same(_u32(thi[:, :npad]), _u32(hi[:npad].T), 'out_thi = out_hi^T')
    _same(_u32(tlo[:, :npad]), _u32(lo[:npad].T), 'out_tlo = out_lo^T')
    assert np.isnan(thi[:, npad:]).all() and np.isnan(tlo[:, npad:]).all()      # t_pitch > ceil64(n): the tail stays untouched


# ================================================================================================================
# ssl_softmax_gemm / ssl_softmax_gemm_tf32x3
# ================================================================================================================

N_R = (1, 127, 128, 129, 300)
N_C = (1, 31, 32, 33, 64, 65, 64 * 9 + 1, 5000)


def _splits(n_c):
    n_ct = (n_c + 63) // 64
    return sorted(set(range(1, min(n_ct, 8) + 1)) | {n_ct})


def _colscale(n_c, rs):
    cs = rs.uniform(0.25, 2.0, n_c).astype(np.float32)
    cs[rs.rand(n_c) < 0.2] = 0.0
    return cs


def _producer(x_np, n, dim, tc, pitch_extra=0):
    """Operand copies written by ssl_rows_normalize (norm_mode 3: the rows themselves, alpha 1), padded to ceil64(n) rows."""
    L = _lib()
    npad = max(64, (n + 63) // 64 * 64)
    pitch = npad + pitch_extra
    x = torch.from_numpy(np.ascontiguousarray(x_np[:n])).to(DEV)
    out = torch.empty(npad, dim, device=DEV)
    out_t = None if tc else torch.empty(npad // 64, dim, 64, device=DEV)
    hi, lo = (torch.empty(npad, dim, device=DEV), torch.empty(npad, dim, device=DEV)) if tc else (None, None)
    thi, tlo = (torch.empty(dim, pitch, device=DEV), torch.empty(dim, pitch, device=DEV)) if tc else (None, None)
    p = lambda t: None if t is None else t.data_ptr()
    L.check(L.lib.ssl_rows_normalize(x.data_ptr(), dim, None, n, dim, 3, 1.0, out.data_ptr(), p(out_t), None, p(hi), p(lo), p(thi), p(tlo),
                                     pitch, _stream()), 'ssl_rows_normalize')
    return dict(out=out, out_t=out_t, hi=hi, lo=lo, thi=thi, tlo=tlo, pitch=pitch, npad=npad)


def _gemm(tc, R, n_r, Cp, n_c, dim, cs, offset, n_split):
    L = _lib()
    rs_part = torch.full((n_split, n_r), float('nan'), device=DEV)
    o_part = torch.full((n_split, n_r, dim), float('nan'), device=DEV)
    csp = None if cs is None else cs.data_ptr()
    if tc:
        rc = L.lib.ssl_softmax_gemm_tf32x3(R['hi'].data_ptr(), R['lo'].data_ptr(), n_r, Cp['hi'].data_ptr(), Cp['lo'].data_ptr(),
                                           Cp['thi'].data_ptr(), Cp['tlo'].data_ptr(), Cp['pitch'], n_c, dim, csp, offset, n_split,
                                           rs_part.data_ptr(), o_part.data_ptr(), _stream())
    else:
        rc = L.lib.ssl_softmax_gemm(R['out'].data_ptr(), n_r, Cp['out'].data_ptr(), Cp['out_t'].data_ptr(), n_c, dim, csp, offset, n_split,
                                    rs_part.data_ptr(), o_part.data_ptr(), _stream())
    L.check(rc, 'softmax gemm')
    torch.cuda.synchronize()
    return rs_part.cpu().numpy(), o_part.cpu().numpy()


def _sentinel_padding(Cp, n_c, dim, tc, cs_pad):
    """The same operands with 7.0 in every padding row / column of the streamed copies (and of colscale's padded tail)."""
    q = dict(Cp)
    rows = torch.arange(Cp['npad'], device=DEV) >= n_c
    for k in ('out', 'hi', 'lo'):
        if Cp[k] is not None:
            q[k] = Cp[k].clone()
            q[k][rows] = 7.0
    if not tc:
        pad = K.k_major_tiles(np.broadcast_to(rows.cpu().numpy()[:, None], (Cp['npad'], dim)).astype(np.float32)) > 0
        q['out_t'] = Cp['out_t'].clone()
        q['out_t'][torch.from_numpy(pad).to(DEV)] = 7.0
    else:
        for k in ('thi', 'tlo'):
            q[k] = Cp[k].clone()
            q[k][:, n_c:] = 7.0
    return q, (None if cs_pad is None else torch.cat([cs_pad[:n_c], torch.full((cs_pad.numel() - n_c,), 7.0, device=DEV)]))


def _run_contraction(tc, dim, R_all, C_all, offset, rtol_fn, seed):
    """Every (n_r, n_c, n_split, colscale) case: each split's partials against float64 over exactly its columns; the
    padding of the streamed operand filled with 7.0 gives bit-identical results (checked at the smallest and the largest
    split)."""
    rs = np.random.RandomState(seed)
    cs_all = _colscale(max(N_C), rs)
    nrm = max(N_R)
    R = _producer(R_all, nrm, dim, tc)
    for n_c in N_C:
        Cp = _producer(C_all, n_c, dim, tc, pitch_extra=64 if n_c % 2 else 0)
        for use_cs in (False, True):
            cs_np = cs_all[:n_c] if use_cs else None
            cs_pad = None
            if use_cs:            # readable up to ceil64(n_c): the tf32x3 kernel loads the tail with the tile and masks it
                cs_pad = torch.zeros(Cp['npad'], device=DEV)
                cs_pad[:n_c] = torch.from_numpy(cs_np).to(DEV)
            rsum_t, o_t, mag_t = K.softmax_gemm_tiles(R['out'][:nrm].cpu().numpy(), Cp['out'][:n_c].cpu().numpy(), cs_np, offset)
            for n_r in N_R:
                Rn = dict(R)
                for n_split in _splits(n_c):
                    rsum, o = _gemm(tc, Rn, n_r, Cp, n_c, dim, cs_pad, offset, n_split)
                    for s, (t0, t1) in enumerate(K.split_tiles(n_c, n_split)):
                        what = f'dim {dim} n_r {n_r} n_c {n_c} colscale {use_cs} split {s}/{n_split} tiles [{t0},{t1})'
                        want_rs, want_o = rsum_t[t0:t1, :n_r].sum(0), o_t[t0:t1, :n_r].sum(0)
                        tol_rs, tol_o = rtol_fn(want_rs, want_rs, t1 - t0), rtol_fn(want_o, mag_t[t0:t1, :n_r].sum(0), t1 - t0)
                        _close(rsum[s], want_rs, tol_rs, 'rowsum_part ' + what)
                        _close(o[s], want_o, tol_o, 'o_part ' + what)
                    if n_split in (1, _splits(n_c)[-1]) and n_r == nrm:
                        Cs, cs_s = _sentinel_padding(Cp, n_c, dim, tc, cs_pad)
                        rsum2, o2 = _gemm(tc, Rn, n_r, Cs, n_c, dim, cs_s, offset, n_split)
                        _same(rsum2, rsum, f'rowsum_part with 7.0 padding, dim {dim} n_c {n_c} split {n_split}')
                        _same(o2, o, f'o_part with 7.0 padding, dim {dim} n_c {n_c} split {n_split}')


@pytest.mark.parametrize('dim', [4, 20, 32, 36, 48, 64, 100, 128])
def test_softmax_gemm_every_split_against_float64(dim):
    """FP32-FMA contraction.  Operands are multiples of 1/8 small enough that every dot product is exact in fp32, so the
    exponents are exact and each e carries only the ex2.approx and colscale roundings.  What remains is the fp32
    accumulation, 64 terms per tile and thread, whose error is a random walk relative to the magnitude sum e |C|: the
    tolerance is 2e-6 * sqrt(tiles of the split) of that magnitude per split (about 7 standard deviations; a dropped or
    unmasked column moves a partial by far more).  Exponents lie in about [-45, 0] (offset = the largest dot product)."""
    rs = np.random.RandomState(dim)
    a = int(np.ceil(np.sqrt(10368.0 / dim)))                    # std of a dot product ~ 4.5
    R_all = (rs.randint(-a, a + 1, (max(N_R), dim)) / 8.0).astype(np.float32)
    C_all = (rs.randint(-8, 9, (max(N_C), dim)) / 8.0).astype(np.float32)
    offset = float((R_all.astype(np.float64) @ C_all.T.astype(np.float64)).max())
    assert offset == float(np.float32(offset))
    _run_contraction(False, dim, R_all, C_all, offset, lambda ref, mag, nt: 2e-6 * np.sqrt(max(nt, 1)) * mag + 1e-30, seed=dim + 1)


@pytest.mark.parametrize('dim', [32, 64])
def test_softmax_gemm_tf32x3_every_split_against_float64(dim):
    """tcgen05 3xTF32 contraction on unit rows (R scaled by log2(e)/0.2, offset the same: exponents in [-14.4, 0]), operands
    from ssl_rows_normalize; the tolerance of test_infonce_term_forward_backward: 2e-4 relative + 1e-5 of the largest entry
    of the split's output (the tensor cores' fp32 accumulators round toward zero)."""
    rs = np.random.RandomState(100 + dim)
    unit = lambda m: (lambda x: (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32))(rs.randn(m, dim))
    off = LOG2E / 0.2
    R_all = (unit(max(N_R)) * np.float32(off)).astype(np.float32)
    C_all = unit(max(N_C))
    _run_contraction(True, dim, R_all, C_all, off, lambda ref, mag, nt: 2e-4 * np.abs(ref) + 1e-5 * np.abs(ref).max(), seed=dim + 2)


def test_softmax_gemm_rejects_bad_splits_and_misaligned_operands():
    L = _lib()
    dim, n_c, n_r = 32, 65, 10
    z = lambda *s: torch.zeros(*s, device=DEV)
    R, Cm, Ct, o, rsum = z(n_r + 1, dim), z(128, dim), z(2, dim, 64), z(4, n_r + 1, dim), z(4, n_r)
    hi, ct = z(128, dim), z(dim, 128)
    torch.cuda.synchronize()
    n0 = L.launch_count()
    ffma = lambda r, c, t, ns: L.lib.ssl_softmax_gemm(r, n_r, c, t, n_c, dim, None, 0.0, ns, rsum.data_ptr(), o.data_ptr(), _stream())
    tc = lambda r, c, t, op, ns: L.lib.ssl_softmax_gemm_tf32x3(r, r, n_r, c, c, t, t, 128, n_c, dim, None, 0.0, ns, rsum.data_ptr(), op, _stream())
    assert ffma(R.data_ptr(), Cm.data_ptr(), Ct.data_ptr(), 3) == SSL_E_ARG                 # 65 columns = 2 tiles
    assert ffma(R.data_ptr() + 4, Cm.data_ptr(), Ct.data_ptr(), 1) == SSL_E_ARG
    assert ffma(R.data_ptr(), Cm.data_ptr() + 8, Ct.data_ptr(), 1) == SSL_E_ARG
    assert ffma(R.data_ptr(), Cm.data_ptr(), Ct.data_ptr() + 4, 1) == SSL_E_ARG
    assert tc(hi.data_ptr(), hi.data_ptr(), ct.data_ptr(), o.data_ptr(), 3) == SSL_E_ARG
    assert tc(hi.data_ptr() + 4, hi.data_ptr(), ct.data_ptr(), o.data_ptr(), 1) == SSL_E_ARG
    assert tc(hi.data_ptr(), hi.data_ptr(), ct.data_ptr() + 4, o.data_ptr(), 1) == SSL_E_ARG
    assert tc(hi.data_ptr(), hi.data_ptr(), ct.data_ptr(), o.data_ptr() + 4, 1) == SSL_E_ARG
    assert L.launch_count() == n0
