"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol the header
declares, the host logic that needs no GPU (config mirror, data handler, generators, seed streams)."""
import os
import re
import types

import numpy as np
import pytest
import scipy.sparse as sp
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import ctypes
    from sslrec_b200 import _lib
    hdr = open(os.path.join(ROOT, 'include', 'sslrec_b200.h')).read()
    declared = set(re.findall(r'SSL_API\s+[\w\s\*]+?\b(ssl_\w+)\s*\(', hdr))
    assert len(declared) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(_lib.EXPORTS)
    assert _lib.lib.ssl_version() >= 100


def test_prop_args_struct_matches_header_layout():
    """ctypes mirror vs the C struct: compile a tiny C program against the header and compare sizeof/offsetof."""
    import ctypes, subprocess, tempfile
    from sslrec_b200 import _lib
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "sslrec_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(ssl_prop_args), offsetof(ssl_prop_args, sum_src), offsetof(ssl_prop_args, edge_mask), offsetof(ssl_prop_args, seed), offsetof(ssl_prop_args, noise_stream_id), offsetof(ssl_prop_args, sum_out_peers), offsetof(ssl_prop_args, reg_src2), offsetof(ssl_prop_args, seed_ptr));return 0;}'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, 't.c'), 'w').write(src)
        subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), os.path.join(d, 't.c'), '-o', os.path.join(d, 't')], check=True)
        out = subprocess.run([os.path.join(d, 't')], capture_output=True, text=True, check=True).stdout.split()
    P = _lib.PropArgs
    assert [int(x) for x in out] == [ctypes.sizeof(P), P.sum_src.offset, P.edge_mask.offset, P.seed.offset, P.noise_stream_id.offset, P.sum_out_peers.offset, P.reg_src2.offset, P.seed_ptr.offset]


def test_normalized_adjacency_matches_oracle_bits():
    from oracle import cf_oracle as O
    from oracle import inputs
    from sslrec_b200.data_handler import normalized_adjacency
    case = inputs.make_case('small')
    trn = sp.coo_matrix((np.ones(len(case['rows'])), (case['rows'], case['cols'])), shape=(case['n_user'], case['n_item']))
    rows, cols, vals, n = normalized_adjacency(trn)
    adj = O.normalized_adjacency(case['rows'], case['cols'], case['n_user'], case['n_item'])
    o = np.lexsort((cols, rows))
    assert n == adj.n and np.array_equal(rows[o], adj.rows) and np.array_equal(cols[o], adj.cols)
    assert np.array_equal(vals[o].view(np.uint32), adj.vals.view(np.uint32))


def test_vectorised_negative_sampler():
    from sslrec_b200.config import default_config, load_config
    from sslrec_b200.data_handler import PairwiseTrnData
    from oracle import inputs
    load_config(base=default_config('lightgcn'), device='cpu')
    case = inputs.make_case('small')
    trn = sp.coo_matrix((np.ones(len(case['rows'])), (case['rows'], case['cols'])), shape=(case['n_user'], case['n_item']))
    ds = PairwiseTrnData(trn)
    np.random.seed(1)
    ds.sample_negs()
    pos = set(zip(case['rows'].tolist(), case['cols'].tolist()))
    assert all((u, j) not in pos for u, j in zip(ds.rows.tolist(), ds.negs.tolist()))
    assert ds.negs.min() >= 0 and ds.negs.max() < case['n_item'] and len(set(ds.negs.tolist())) > case['n_item'] // 2


def test_synthetic_graph_generator_is_deterministic_and_exact():
    from synth_graphs import bipartite_graph
    r1, c1 = bipartite_graph(2000, 1500, 30000, seed=5, zipf_alpha=0.5)
    r2, c2 = bipartite_graph(2000, 1500, 30000, seed=5, zipf_alpha=0.5)
    assert np.array_equal(r1, r2) and np.array_equal(c1, c2) and len(r1) == 30000
    assert len(set(zip(r1.tolist(), c1.tolist()))) == 30000
    assert r1.max() < 2000 and c1.max() < 1500


def test_models_refuse_to_run_without_cuda():
    from sslrec_b200 import engine as E
    with pytest.raises(RuntimeError, match='CUDA'):
        E._require_cuda(torch.zeros(2, 4), 'table')


def test_choose_split_fills_waves():
    from sslrec_b200.engine import choose_split
    assert choose_split(32, 1309) == 37          # 32 * 37 = 1184 = 4 waves of 296 CTA slots
    assert choose_split(32, 1) == 1
    s = choose_split(655, 64)
    assert 1 <= s <= 16 and (655 * s) / (296 * -(-655 * s // 296)) > 0.95
    # the tcgen05 kernel (1 CTA per SM): waves x (tiles per CTA + per-CTA overhead), fitted to the B200 sweep (tools/perf_tc.py sweep)
    assert choose_split(32, 1195, slots=148, prefer_few=True) == 9          # forward role at the amazon shape: measured optimum
    assert choose_split(598, 64, slots=148, prefer_few=True) == 2           # backward role: measured optimum (the wave-efficiency rule said 4)
    assert choose_split(200, 64, slots=148, prefer_few=True) == 2 and choose_split(1, 1, slots=148, prefer_few=True) == 1


def test_device_side_components_fail_loudly_without_cuda():
    """No host fallback: the device loader, the native k-means and the DirectAU losses refuse CPU inputs."""
    from sslrec_b200 import loss_utils as LU
    from sslrec_b200.data_handler import DeviceTrnData
    from sslrec_b200.kmeans import KMeansClustering
    trn = sp.coo_matrix((np.ones(3), ([0, 1, 2], [1, 0, 2])), shape=(3, 3))
    with pytest.raises(RuntimeError, match='CUDA'):
        DeviceTrnData(trn, 'cpu')
    with pytest.raises(RuntimeError, match='CUDA'):
        KMeansClustering(2, 4)(torch.zeros(8, 4))
    with pytest.raises(RuntimeError, match='CUDA'):
        LU.uniformity(torch.randn(8, 4))
    with pytest.raises(RuntimeError, match='CUDA'):
        LU.alignment(torch.randn(8, 4), torch.randn(8, 4))


def test_batch_shard_coalesce_orders_by_parameter_position():
    """Collectives must be issued in the same order on every rank although buffer addresses differ per process."""
    from sslrec_b200.parallel import BatchShard
    flat = torch.zeros(10, 2)
    a, b, c = flat[:6], flat[6:], torch.zeros(5)
    for order in ([c, a, b], [b, c, a], [a, b, c]):
        bufs = BatchShard.coalesce(order)
        pos_c = [i for i, t in enumerate(order) if t is c][0]
        first = min(i for i, t in enumerate(order) if t is not c)
        want = [20, 5] if first < pos_c else [5, 20]
        assert [x.numel() for x in bufs] == want, [x.numel() for x in bufs]
    nc = torch.zeros(4, 6)[:, :3]                                 # non-contiguous gradients travel alone
    assert [x.numel() for x in BatchShard.coalesce([nc, a])] == [12, 12]


def test_device_loader_shares_and_flags_with_a_stub_dataset():
    """DeviceLoader's shuffling / sharding / epoch-flag bookkeeping is device-agnostic: exercised here with a CPU stub in
    place of DeviceTrnData (whose kernels are covered by the GPU tests)."""
    from sslrec_b200.data_handler import DeviceLoader, DeviceTrnData

    class Stub:
        device, epoch_period, epoch_flag_counter = torch.device('cpu'), 2, -1
        rows = torch.arange(103) * 10
        cols = negs = torch.arange(103)
        __len__ = lambda self: 103
        batch = DeviceTrnData.batch
    full = DeviceLoader(Stub(), 16, seed=3)
    assert len(full) == 7
    got = torch.cat([b[0] for b in full])
    assert sorted(got.tolist()) == (torch.arange(103) * 10).tolist()
    first, second = torch.cat([b[0] for b in full]), torch.cat([b[0] for b in full])
    assert not torch.equal(first, second)                          # a fresh permutation per epoch
    shares = [torch.cat([b[0] for b in DeviceLoader(Stub(), 16, rank=r, world=3, seed=5)]) for r in range(3)]
    assert [len(s) for s in shares] == [35, 35, 35] and len(DeviceLoader(Stub(), 16, rank=0, world=3)) == 3
    assert set(torch.cat(shares).tolist()) == set((torch.arange(103) * 10).tolist())    # padded by wrap-around, nothing lost
    ds = Stub()
    loader = DeviceLoader(ds, 16, seed=4)
    flags = [int(torch.cat([b[3] for b in loader]).sum()) for _ in range(5)]
    assert flags == [1, 1, 0, 1, 0]                                # first sample ever, then pair 0 on every 2nd visit


def test_trainer_early_stop_restores_best_state_tests_and_saves(tmp_path, monkeypatch):
    """Trainer.train (trainer.py:86-137): patience counting on the first metric @ k[0], best state_dict restored into a
    freshly built model, final evaluate + test, checkpoint under ./checkpoint/{model}/{model}-{data}-{ts}.pth."""
    import torch
    from sslrec_b200.config import configs, default_config, load_config
    from sslrec_b200.trainer import Trainer
    cfg = default_config('lightgcn')
    cfg['train'].update(epoch=20, test_step=1, patience=2, save_model=True)
    cfg['data']['name'] = 'gowalla'
    load_config(base=cfg, device='cpu')
    assert configs['train']['early_stop'] is True
    monkeypatch.chdir(tmp_path)

    class Model(torch.nn.Module):
        def __init__(self, data_handler=None):
            super().__init__()
            self.w = torch.nn.Parameter(torch.zeros(3))
    scores = [0.10, 0.30, 0.20, 0.25, 0.90]            # best at epoch 1; epochs 2, 3 do not improve -> stop after epoch 3
    log = []
    tr = Trainer(types.SimpleNamespace(test_dataloader='tst', valid_dataloader='val'))
    monkeypatch.setattr(tr, 'create_optimizer', lambda m: None)

    def train_epoch(model, e):
        with torch.no_grad():
            model.w.fill_(float(e))
        log.append(('train', e))

    def evaluate(model, epoch_idx=None, loader=None, data_type=None):
        log.append(('eval', epoch_idx, data_type, float(model.w[0])))
        return {'recall': [scores[epoch_idx] if epoch_idx is not None else -1.0], 'ndcg': [0.0]}
    monkeypatch.setattr(tr, 'train_epoch', train_epoch)
    monkeypatch.setattr(tr, 'evaluate', evaluate)
    best = tr.train(Model())
    assert [x for x in log if x[0] == 'train'] == [('train', e) for e in range(4)]          # stopped by patience, not by epoch count
    assert float(best.w[0]) == 1.0                                                           # epoch 1's parameters came back
    assert log[-2][:3] == ('eval', None, None) and log[-2][3] == 1.0                         # final evaluate on the restored model
    assert log[-1][:3] == ('eval', None, 'Test set')                                         # then test()
    saved = list((tmp_path / 'checkpoint' / 'lightgcn').glob('lightgcn-gowalla-*.pth'))
    assert len(saved) == 1 and float(torch.load(saved[0])['w'][0]) == 1.0
    # without patience: every epoch runs, then test + save
    cfg2 = default_config('lightgcn')
    cfg2['train'].update(epoch=3, test_step=2)
    load_config(base=cfg2, device='cpu')
    log.clear()
    tr.train(Model())
    assert [x[1] for x in log if x[0] == 'train'] == [0, 1, 2] and [x[1] for x in log if x[0] == 'eval'] == [0, 2, None]
    # unknown metric names are an error, not zeros
    cfg2['test']['metrics'] = ['recall', 'auc']
    load_config(base=cfg2, device='cpu')
    import pytest
    with pytest.raises(ValueError):
        Trainer(types.SimpleNamespace(test_dataloader=[])).evaluate(Model())


def test_vectorised_evaluation_metrics_match_the_per_user_loop_and_do_not_depend_on_batching():
    """trainer.batch_metric_rows (recall / ndcg / precision / mrr, metrics.py:11-45) against the per-user loop form of the same
    formulas: truth lists with duplicates and with more entries than the cut-off, several hits per row; summed over all users in
    loader order the result is bit-identical for any batch size."""
    from sslrec_b200.trainer import batch_metric_rows, truth_csr
    rs = np.random.RandomState(0)
    n_users, n_item, kmax, ks = 700, 900, 40, [10, 20, 40]
    top = np.stack([rs.permutation(n_item)[:kmax] for _ in range(n_users)])
    truths = [rs.choice(n_item, size=rs.randint(1, 60), replace=True).tolist() for _ in range(n_users)]
    for u in range(n_users):
        for _ in range(rs.randint(0, 4)):
            top[u, rs.randint(0, kmax)] = truths[u][rs.randint(len(truths[u]))]
    mets = ('recall', 'ndcg', 'precision', 'mrr')
    want = {m: np.zeros(len(ks)) for m in mets}
    for u in range(n_users):
        hit = np.isin(top[u], truths[u]).astype(np.float64)
        for ki, k in enumerate(ks):
            want['recall'][ki] += hit[:k].sum() / len(truths[u]) / n_users
            idcg = (1.0 / np.log2(np.arange(2, min(k, len(truths[u])) + 2))).sum()
            want['ndcg'][ki] += (hit[:k] / np.log2(np.arange(2, k + 2))).sum() / idcg / n_users
            want['precision'][ki] += hit[:k].sum() / k / n_users
            want['mrr'][ki] += (hit[:k] / np.arange(1, k + 1)).sum() / n_users
    ptr, flat = truth_csr(types.SimpleNamespace(user_pos_lists=truths))
    order = rs.permutation(n_users)                              # loaders serve test_users, not 0..n-1

    def run(batch):
        per = {m: [] for m in mets}
        for lo in range(0, n_users, batch):
            rows = batch_metric_rows(top[order[lo:lo + batch]], order[lo:lo + batch], ptr, flat, ks, mets)
            for m in mets:
                per[m].append(rows[m])
        return {m: np.concatenate(per[m]).sum(0) / n_users for m in mets}
    a, b = run(1024), run(96)
    for m in mets:
        assert np.abs(a[m] - want[m]).max() < 1e-13, m
        assert np.array_equal(a[m], b[m]), m
    assert want['recall'][0] > 0 and want['mrr'][2] > 0


def test_trainer_evaluate_end_to_end_with_a_stub_model(monkeypatch):
    """Trainer.evaluate's plumbing on the CPU (the kernels behind full_predict / topk are covered by the GPU tests): loader batches ->
    full_predict -> top-k -> vectorised metrics, for the dense-mask loader of the reference and the lean (device-CSR) loader, against
    the loop form of metrics.py:82-127 on the same scores."""
    import scipy.sparse as sp
    import torch.utils.data as tdata
    from sslrec_b200 import trainer as T
    from sslrec_b200.config import default_config, load_config
    from sslrec_b200.data_handler import AllRankTstData
    load_config(base=default_config('lightgcn'), device='cpu')
    rs = np.random.RandomState(4)
    U, I = 333, 150
    trn = sp.coo_matrix((np.ones(900), (rs.randint(0, U, 900), rs.randint(0, I, 900))), shape=(U, I))
    val = sp.coo_matrix((np.ones(500), (rs.randint(0, U - 20, 500), rs.randint(0, I, 500))), shape=(U, I))      # the last users have no held-out item
    scores = torch.from_numpy(rs.rand(U, I).astype(np.float32))
    trn_mask = torch.from_numpy((trn.tocsr().toarray() != 0))

    class Model(torch.nn.Module):
        def full_predict(self, batch_data):
            users, mask = batch_data
            s = scores[users]
            m = trn_mask[users] if isinstance(mask, str) else mask.bool()
            return torch.where(m, torch.full_like(s, -1e8), s)
    monkeypatch.setattr(T, 'topk', lambda preds, k: torch.topk(preds, k).indices)
    tr = T.Trainer(types.SimpleNamespace())
    res = {}
    for dense in (True, False):
        ds = AllRankTstData(val, trn, dense_mask=dense)
        res[dense] = tr.evaluate(Model(), loader=tdata.DataLoader(ds, batch_size=64, shuffle=False))
    for m in ('recall', 'ndcg'):
        assert np.array_equal(res[True][m], res[False][m])
    ds = AllRankTstData(val, trn)
    ks, n = [10, 20, 40], len(ds.test_users)
    want = {'recall': np.zeros(3), 'ndcg': np.zeros(3)}
    for u in ds.test_users:
        s = torch.where(trn_mask[u], torch.tensor(-1e8), scores[u])
        top = torch.topk(s, 40).indices.numpy()
        truth = ds.user_pos_lists[u]
        hit = np.isin(top, truth).astype(np.float64)
        for ki, k in enumerate(ks):
            want['recall'][ki] += hit[:k].sum() / len(truth) / n
            want['ndcg'][ki] += (hit[:k] / np.log2(np.arange(2, k + 2))).sum() / (1.0 / np.log2(np.arange(2, min(k, len(truth)) + 2))).sum() / n
    for m in want:
        assert np.abs(res[True][m] - want[m]).max() < 1e-12 and want[m][2] > 0


def test_host_batch_loader_is_the_torch_dataloader_batch_for_batch():
    """data_handler.HostBatchLoader against torch.utils.data.DataLoader(trn_data, batch_size, shuffle=True) (data_handler_general_cf.py:95)
    under the same global seed: identical batches (values and dtypes) over several epochs, identical epoch flags of NCL's dataset, and
    the same state of torch's global generator afterwards."""
    import scipy.sparse as sp
    import torch.utils.data as tdata
    from sslrec_b200.config import default_config, load_config
    from sslrec_b200.data_handler import HostBatchLoader, PairwiseTrnData, PairwiseWEpochFlagTrnData
    load_config(base=default_config('ncl', epoch_period=2), device='cpu')
    rs = np.random.RandomState(0)
    U, I = 300, 200
    key = np.unique(rs.randint(0, U, 5000).astype(np.int64) * I + rs.randint(0, I, 5000))
    m = sp.coo_matrix((np.ones(len(key)), (key // I, key % I)), shape=(U, I))
    for cls in (PairwiseTrnData, PairwiseWEpochFlagTrnData):
        runs = []
        for make in (lambda d: tdata.DataLoader(d, batch_size=256, shuffle=True, num_workers=0), lambda d: HostBatchLoader(d, 256)):
            d = cls(m)
            loader = make(d)
            torch.manual_seed(5)
            np.random.seed(1)
            epochs = []
            for _ in range(5):
                d.sample_negs()
                epochs.append([[t.clone() for t in batch] for batch in loader])
            runs.append((len(loader), epochs, torch.get_rng_state()))
        (la, ea, ra), (lb, eb, rb) = runs
        assert la == lb and torch.equal(ra, rb)
        for x, y in zip(ea, eb):
            assert len(x) == len(y)
            for bx, by in zip(x, y):
                assert isinstance(by, list) and len(bx) == len(by)
                assert all(t.dtype == u.dtype and torch.equal(t, u) for t, u in zip(bx, by))
        if cls is PairwiseWEpochFlagTrnData:
            assert [int(sum(b[3].sum() for b in e)) for e in eb] == [1, 1, 0, 1, 0]


def test_data_handler_default_train_loader():
    import scipy.sparse as sp
    import torch.utils.data as tdata
    from sslrec_b200.config import default_config, load_config
    from sslrec_b200.data_handler import DataHandlerGeneralCF, HostBatchLoader
    rs = np.random.RandomState(1)
    m = sp.coo_matrix((np.ones(400), (rs.randint(0, 50, 400), rs.randint(0, 40, 400))), shape=(50, 40))
    cfg = default_config('lightgcn')
    cfg['train']['batch_size'] = 64
    load_config(base=cfg, device='cpu')
    dh = DataHandlerGeneralCF(m, m, m)
    dh.load_data()
    assert isinstance(dh.train_dataloader, HostBatchLoader) and len(dh.train_dataloader) == (len(dh.train_dataloader.dataset) + 63) // 64
    cfg['train']['torch_dataloader'] = True
    load_config(base=cfg, device='cpu')
    dh = DataHandlerGeneralCF(m, m, m)
    dh.load_data()
    assert isinstance(dh.train_dataloader, tdata.DataLoader)


def test_trainer_tensorboard_scalars(tmp_path, monkeypatch):
    """train.tensorboard: true -> the scalars of trainer.py:78,144 ('Loss/train' per epoch, 'HR/test' per evaluate, none for test)."""
    from sslrec_b200 import trainer as T
    from sslrec_b200.config import default_config, load_config
    cfg = default_config('lightgcn')
    cfg['train']['tensorboard'] = True
    load_config(base=cfg, device='cpu')
    calls = []

    class Writer:
        def add_scalar(self, tag, value, step):
            calls.append((tag, round(float(value), 6), step))
    monkeypatch.setattr(T, '_summary_writer', lambda: Writer())
    tr = T.Trainer(types.SimpleNamespace())
    tr._scalar('Loss/train', 0.5, 3)
    assert calls == [('Loss/train', 0.5, 3)]
    cfg['train']['tensorboard'] = False
    load_config(base=cfg, device='cpu')
    tr2 = T.Trainer(types.SimpleNamespace())
    tr2._scalar('Loss/train', 0.5, 3)
    assert len(calls) == 1 and tr2._writer is None


def test_lean_evaluation_batches_equal_the_dataloader_batches():
    import scipy.sparse as sp
    import torch.utils.data as tdata
    from sslrec_b200.config import default_config, load_config
    from sslrec_b200.data_handler import AllRankTstData
    from sslrec_b200.trainer import _eval_batches
    load_config(base=default_config('lightgcn'), device='cpu')
    rs = np.random.RandomState(1)
    U, I = 500, 80
    trn = sp.coo_matrix((np.ones(900), (rs.randint(0, U, 900), rs.randint(0, I, 900))), shape=(U, I))
    val = sp.coo_matrix((np.ones(300), (rs.randint(0, U, 300), rs.randint(0, I, 300))), shape=(U, I))
    lean = tdata.DataLoader(AllRankTstData(val, trn, dense_mask=False), batch_size=64, shuffle=False, num_workers=0)
    a, b = [x.clone() for x in lean], list(_eval_batches(lean))
    assert len(a) == len(b) and all(x.dtype == y.dtype and torch.equal(x, y) for x, y in zip(a, b))
    dense = tdata.DataLoader(AllRankTstData(val, trn, dense_mask=True), batch_size=64, shuffle=False)
    first = next(iter(_eval_batches(dense)))
    assert isinstance(first, list) and len(first) == 2 and first[1].shape == (64, I)          # the reference's [users, mask] batches untouched


def test_vectorised_metrics_match_the_reference_metric_class():
    """trainer.batch_metric_rows against the reference's own ``Metric.eval_batch`` (trainer/metrics.py:11-80) on random top-k lists and ground
    truths, all four metrics.  The inputs and the reference's per-k sums are stored in tests/golden/ref_metric_eval_batch.npz
    (oracle/gen_host_golden.py)."""
    from sslrec_b200.trainer import batch_metric_rows, truth_csr
    z = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_metric_eval_batch.npz'))
    top, tp, tf = z['top'].astype(np.int64), z['truth_ptr'], z['truth_flat']
    truths = [tf[tp[u]:tp[u + 1]].tolist() for u in range(top.shape[0])]
    ks, metrics = [int(k) for k in z['ks']], [str(m) for m in z['metrics']]
    assert set(metrics) == {'recall', 'ndcg', 'precision', 'mrr'}
    ptr, flat = truth_csr(types.SimpleNamespace(user_pos_lists=truths))
    got = batch_metric_rows(top, np.arange(top.shape[0]), ptr, flat, ks, metrics)
    for m in metrics:
        want = z['want_' + m]
        assert np.allclose(want, got[m].sum(0), rtol=1e-12, atol=1e-12), (m, want, got[m].sum(0))
        assert want[-1] > 0


def test_host_data_path_reproduces_the_reference_batches_draw_for_draw():
    """The reference's own training data path (data_utils/datasets_general_cf.py:6-26 ``PairwiseTrnData`` with its per-pair rejection loop, served by
    ``DataLoader(trn_data, batch_size, shuffle=True)``, data_handler_general_cf.py:95) against this repository's default host path (vectorised
    ``sample_negs`` + ``HostBatchLoader``) under the same numpy / torch seeds: identical (user, positive, negative) batches over two epochs and the
    same generator states afterwards -- a graph dense enough that a third of the first draws are rejected.  The reference's batches and states are
    stored in tests/golden/ref_pairwise_batches.npz (oracle/gen_host_golden.py)."""
    from sslrec_b200.data_handler import HostBatchLoader, PairwiseTrnData
    z = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_pairwise_batches.npz'))
    rs = np.random.RandomState(0)
    U, I = 90, 30
    key = np.unique(rs.randint(0, U, 1500).astype(np.int64) * I + rs.randint(0, I, 1500))
    assert int(z['n_user']) == U and int(z['n_item']) == I and np.array_equal(key, z['key'])       # the graph the reference was given
    m = sp.coo_matrix((np.ones(len(key)), (key // I, key % I)), shape=(U, I))
    ds = PairwiseTrnData(m)
    loader = HostBatchLoader(ds, int(z['batch_size']))
    np.random.seed(11)
    torch.manual_seed(12)
    for epoch in range(2):
        ds.sample_negs()
        batches = [[t.long().numpy() for t in b] for b in loader]
        assert np.array_equal([len(b[0]) for b in batches], z[f'epoch{epoch}_batch_len']), epoch
        triples = np.stack([np.concatenate([b[i] for b in batches]) for i in range(3)])
        assert np.array_equal(triples, z[f'epoch{epoch}_triples']), epoch
    assert np.array_equal(np.random.get_state()[1][:8], z['numpy_state_head'])
    assert np.array_equal(torch.get_rng_state()[:16].numpy(), z['torch_state_head'])
    assert len(z['epoch0_batch_len']) >= 5 and len(key) / (U * I) > 0.3
