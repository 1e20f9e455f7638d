"""Model-level parity on the GPU: the drop-in classes against the golden vectors of the unmodified
reference (same weights, same batch, injected masks / noise), through the C ABI.
Tolerances: loss terms |d| <= 1e-5 (BASELINE.json), gradients / Adam rtol 2e-4 + 5e-6 * max|g|
(fp32 reassociation between torch's CPU kernels and the CUDA summation order)."""
import numpy as np
import pytest
import torch

from oracle import cf_oracle as O
from oracle import inputs, replay
import ssl_test_helpers as H

pytestmark = pytest.mark.gpu

CASES = [('lightgcn', 'tiny'), ('simgcl', 'tiny'), ('sgl', 'tiny'), ('sgl_nd', 'tiny'), ('ncl', 'tiny'), ('hccf', 'tiny'),
         ('lightgcn', 'small'), ('simgcl', 'small'), ('sgl', 'small'), ('simgcl', 'mid'),
         ('directau', 'tiny'), ('directau', 'small'), ('lightgcl', 'tiny'), ('lightgcl', 'small'),
         ('ncl_k50', 'small'), ('hccf_h128', 'small')]        # the YAML sizes: ncl.yml cluster_num 50, hccf.yml hyper_num 128


def _run(model_key, case_name):
    g = replay.load_golden(model_key, case_name)
    hp = g['hp']
    case = inputs.make_case(case_name)
    adj = O.normalized_adjacency(case['rows'], case['cols'], case['n_user'], case['n_item'])
    dr = replay.draws(model_key, case, hp, adj)
    model, dh = H.make_model(model_key, case, hp, inject=H.gpu_injection(model_key, case, hp, adj, dr))
    sd = {'user_embeds': case['user_e'], 'item_embeds': case['item_e']}
    if 'user_w' in dr:
        sd['user_hyper_embeds'], sd['item_hyper_embeds'] = dr['user_w'], dr['item_w']
    if model_key == 'lightgcl':
        for i, w in enumerate(dr['ws']):
            sd[f'Ws.{i}.W'] = w
        # the t.svd_lowrank factors of the reference run (random projections: injected, like every other draw)
        model.ut, model.vt, model.u_mul_s, model.v_mul_s = (torch.from_numpy(g['svd_' + k]).cuda() for k in ('ut', 'vt', 'u_mul_s', 'v_mul_s'))
        if 'lgcl_vals' in g:       # R / sqrt(rowD colD): bit-identical values (float32 arithmetic as lightgcl.py:16-20)
            r, c, v = model._ui
            o, og = np.lexsort((c, r)), np.lexsort((g['lgcl_cols'], g['lgcl_rows']))
            assert np.array_equal(r[o], g['lgcl_rows'][og]) and np.array_equal(c[o], g['lgcl_cols'][og])
            assert np.array_equal(v[o].view(np.uint32), g['lgcl_vals'][og].view(np.uint32))
    model.load_state_dict(sd)
    if model_key.split('_')[0] == 'ncl':
        model.user_centroids = torch.from_numpy(g['user_centroids']).cuda()
        model.item_centroids = torch.from_numpy(g['item_centroids']).cuda()
        model.user2cluster = torch.from_numpy(g['user2cluster']).cuda()
        model.item2cluster = torch.from_numpy(g['item2cluster']).cuda()
    batch = [torch.from_numpy(case[k]).cuda() for k in ('ancs', 'poss', 'negs')]
    if model_key.split('_')[0] == 'ncl':
        batch.append(torch.zeros(case['batch'], dtype=torch.int64).cuda())
    return g, case, model, batch


@pytest.mark.parametrize('model_key,case_name', CASES)
def test_cal_loss_backward_adam_match_reference(model_key, case_name):
    from sslrec_b200.optim import FusedAdam
    g, case, model, batch = _run(model_key, case_name)
    wd = float(g.get('opt_weight_decay', 0.0))            # directau.yml: 1e-6; the other YAMLs: 0
    opt = FusedAdam(model.parameters(), lr=float(g.get('opt_lr', 1e-3)), weight_decay=wd)
    opt.zero_grad()
    loss, parts = model.cal_loss(batch)
    assert abs(loss.item() - float(g['loss'])) <= 1e-5 * max(1.0, abs(float(g['loss']))), (loss.item(), float(g['loss']))
    for k, v in parts.items():
        assert abs(float(v) - float(g['part_' + k])) <= 1e-5 * max(1.0, abs(float(g['part_' + k]))), (k, float(v), float(g['part_' + k]))
    loss.backward()
    for name, p in model.named_parameters():
        gr = p.grad
        if 'grad_' + name in g:
            ref = g['grad_' + name]
            H.close(gr, ref, 2e-4, 5e-6 * np.abs(ref).max() + 1e-9, 'grad_' + name)
        else:
            ref = g['grad_' + name + '_head']
            scale = g['grad_' + name + '_abssum'] / gr.numel()
            H.close(gr[:32], ref, 2e-4, 2e-4 * scale + 1e-9, 'grad_' + name + '_head')
            H.close(gr.double().sum(1), g['grad_' + name + '_rowsum'], 1e-3, 1e-3 * scale * gr.shape[1], 'grad_' + name + '_rowsum')
            assert abs(gr.double().abs().sum().item() - g['grad_' + name + '_abssum']) <= 1e-4 * g['grad_' + name + '_abssum']
    opt.step()
    for name, p in model.named_parameters():
        full = 'new_' + name in g
        ref = g['new_' + name] if full else g['new_' + name + '_head']
        gref = g['grad_' + name] if full else (g['grad_' + name + '_head'] if 'grad_' + name + '_head' in g else g['grad_' + name][:32])
        got = (p if full else p[:32]).detach().cpu().numpy()
        # entries whose reference gradient is rounding noise have no defined Adam sign (see test_oracle_golden.py)
        case_p = case[{'user_embeds': 'user_e', 'item_embeds': 'item_e'}[name]].numpy() if name in ('user_embeds', 'item_embeds') else 0.0
        gtot = gref + wd * (case_p if full or np.isscalar(case_p) else case_p[:32])       # Adam folds weight decay into g
        noise = np.abs(gtot) <= 1e-5 * np.abs(gtot).max()
        H.close(np.where(noise, ref, got), ref, 1e-5, 2e-6, 'new_' + name)
        assert (np.abs(got - ref)[noise] <= 2.1e-3).all(), name


@pytest.mark.parametrize('model_key,case_name', CASES)
def test_full_predict_topk_match_reference(model_key, case_name):
    from sslrec_b200.trainer import topk
    g, case, model, batch = _run(model_key, case_name)
    U, I = case['n_user'], case['n_item']
    bt = min(64, U)
    users = torch.arange(bt).cuda()
    mask = torch.zeros(bt, I, dtype=torch.int64)
    sel = case['rows'] < bt
    mask[torch.from_numpy(case['rows'][sel]), torch.from_numpy(case['cols'][sel])] = 1
    model.eval()
    with torch.no_grad():
        preds = model.full_predict([users, mask.cuda()])
    if 'preds' in g:
        H.close(preds, g['preds'], 1e-5, 1e-6, 'preds')
    k = min(40, I)
    idx, val = topk(preds, k, return_values=True)
    # identical to torch.topk on the same scores (ties -> lower index, which torch does not promise: compare values)
    tv, ti = torch.topk(preds, k)
    assert torch.equal(val, tv)
    gv, gi = g['topk_val'], g['topk_idx']
    H.close(val, gv, 1e-5, 1e-6, 'topk_val')
    gap = np.abs(np.diff(gv, axis=1))
    near = gap <= 2e-6 * np.maximum(1.0, np.abs(gv[:, :-1]))
    ok = np.ones_like(gi, dtype=bool)
    ok[:, :-1] &= ~near
    ok[:, 1:] &= ~near
    ok[:, -1] = False
    assert (idx.cpu().numpy()[ok] == gi[ok]).all()      # bit-exact indices wherever the reference's own gap is not a near-tie
    assert ok.mean() > 0.9


@pytest.mark.parametrize('name', ['lightgcn', 'simgcl', 'ncl', 'directau', 'lightgcl'])
def test_trainer_epochs_and_evaluate(name):
    """The Trainer mirror end to end on a small graph: train_epoch (sample_negs, DataLoader, cal_loss, backward, FusedAdam,
    asynchronous loss reads), evaluate (full_predict -> native top-k -> recall / ndcg); the loss goes down and the
    logged epoch loss equals the sum of the per-step losses."""
    import scipy.sparse as sp
    from sslrec_b200.config import default_config, load_config
    from sslrec_b200.data_handler import DataHandlerGeneralCF
    from sslrec_b200.trainer import Trainer, init_seed
    import importlib
    case = inputs.make_case('small')
    hp = dict(layer_num=2, embedding_size=32, reg_weight=1e-6, keep_rate=0.8, cl_weight=1e-2, temperature=0.2, eps=0.2)
    if name == 'ncl':
        hp.update(high_order=1, proto_weight=1e-3, struct_weight=1e-3, cluster_num=8, epoch_period=1, keep_rate=1.0)
    if name == 'directau':
        hp.update(gamma=2.0)
    if name == 'lightgcl':
        hp.update(dropout=0.1, temp=0.2, svd_q=5)                # dropout > 0: the in-kernel per-layer value dropout
    cfg = default_config(name, **hp)
    cfg['train'].update(batch_size=1024, epoch=2, loss='pairwise_with_epoch_flag' if name == 'ncl' else 'pairwise')
    if name in ('directau', 'ncl'):
        cfg['train']['device_loader'] = True                     # pairs, negative sampling and batching on the device
    cfg['optimizer']['lr'] = 5e-3
    cfg['test']['batch_size'] = 256
    cfg['test']['dense_mask'] = True                             # the reference's dense train-mask rows; the lean loader is compared below
    load_config(base=cfg, device='cuda')
    init_seed()
    U, I = case['n_user'], case['n_item']
    trn = sp.coo_matrix((np.ones(len(case['rows']), dtype=np.float32), (case['rows'], case['cols'])), shape=(U, I))
    rs = np.random.RandomState(0)
    val = sp.coo_matrix((np.ones(400), (rs.randint(0, U, 400), rs.randint(0, I, 400))), shape=(U, I))
    dh = DataHandlerGeneralCF(trn, val, val)
    dh.load_data()
    mod = importlib.import_module('sslrec_b200.general_cf.' + name)
    model = [getattr(mod, a) for a in dir(mod) if a.lower() == name][0](dh).cuda()
    tr = Trainer(dh)
    tr.create_optimizer(model)
    losses = [tr.train_epoch(model, e)[0] for e in range(3)]
    assert all(np.isfinite(losses)) and losses[-1] < losses[0]
    res = tr.evaluate(model)
    assert set(res) == {'recall', 'ndcg'} and all(0.0 <= v <= 1.0 for m in res.values() for v in m)
    assert res['recall'][2] >= res['recall'][0]          # recall@40 >= recall@10
    # the device-CSR mask (no dense host rows) gives exactly the same scores and metrics as the reference's dense mask
    from sslrec_b200.data_handler import AllRankTstData
    import torch.utils.data as tdata
    lean = tdata.DataLoader(AllRankTstData(val, trn, dense_mask=False), batch_size=256, shuffle=False)
    res2 = tr.evaluate(model, loader=lean)
    for m in res:
        assert np.array_equal(res[m], res2[m])
    users = torch.arange(64).cuda()
    dense = torch.from_numpy((trn.tocsr()[:64].toarray() != 0).astype(np.int64)).cuda()
    with torch.no_grad():
        assert torch.equal(model.full_predict([users, dense]), model.full_predict([users, 'train']))


@pytest.mark.parametrize('name', ['lightgcn', 'simgcl', 'sgl', 'sgl_nd'])
def test_cuda_graph_step_equals_eager_step(name):
    """graphed.GraphedStep: the captured step replayed on new batches with device-resident seeds / step count trains exactly like
    the eager loop -- same in-kernel masks and noise (the SeedStream sequence is shared), same losses, same parameters."""
    from sslrec_b200.graphed import GraphedStep
    from sslrec_b200.optim import FusedAdam
    size = 'tiny' if name == 'sgl_nd' else 'small'
    g = replay.load_golden(name, size)
    case = inputs.make_case(size)
    rs = np.random.RandomState(3)
    B = case['batch']
    batches = []
    for _ in range(5):
        pick = rs.randint(0, len(case['rows']), size=B)
        batches.append([torch.from_numpy(np.asarray(a)).long().cuda() for a in (case['rows'][pick], case['cols'][pick], rs.randint(0, case['n_item'], size=B))])
    out = {}
    for mode in ('eager', 'graph'):
        model, _ = H.make_model(name, case, g['hp'])
        model.load_state_dict({'user_embeds': case['user_e'], 'item_embeds': case['item_e']})
        opt = FusedAdam(model.parameters(), lr=1e-2)
        losses = []
        if mode == 'eager':
            for b in [batches[0]] * 2 + batches[1:]:
                opt.zero_grad()
                loss, parts = model.cal_loss(b)
                loss.backward()
                opt.step()
                losses.append(loss.item())
        else:
            step = GraphedStep(model, opt, batches[0], warmup=2)          # two eager steps on batch 0, then the capture
            losses += [float('nan')] * 2
            assert step.n_seeds == {'lightgcn': 1, 'simgcl': 2, 'sgl': 2, 'sgl_nd': 2}[name]
            for b in batches[1:]:
                loss, parts = step(b)
                losses.append(loss.item())
            step.close()
            assert all(int(st['step']) == 6 for st in opt.state.values())          # the device counter came back to the host
            # and the eager path continues from the same seed sequence afterwards
        out[mode] = (losses, torch.cat([model.user_embeds.detach(), model.item_embeds.detach()]).clone())
    for a, b in zip(out['graph'][0][2:], out['eager'][0][2:]):
        assert abs(a - b) <= 1e-6 * max(1.0, abs(b)), (name, out['graph'][0], out['eager'][0])
    assert torch.allclose(out['graph'][1], out['eager'][1], rtol=1e-5, atol=3e-4), (name, (out['graph'][1] - out['eager'][1]).abs().max().item())


def test_trainer_cuda_graph_epoch_matches_eager_epoch():
    """Trainer.train_epoch with train.cuda_graph: the same per-epoch loss as the eager loop on the same loader order (device loader,
    fixed seed), including the epoch's last, smaller batch."""
    import types
    from sslrec_b200.config import configs
    from sslrec_b200.data_handler import DeviceLoader, DeviceTrnData
    from sslrec_b200.trainer import Trainer
    g = replay.load_golden('simgcl', 'small')
    case = inputs.make_case('small')
    res = {}
    for graph in (False, True):
        model, dh = H.make_model('simgcl', case, g['hp'])
        model.load_state_dict({'user_embeds': case['user_e'], 'item_embeds': case['item_e']})
        configs['train']['cuda_graph'] = graph
        configs['train']['batch_size'] = 512
        loader = DeviceLoader(DeviceTrnData(dh.trn_mat, 'cuda', 2023), 512, seed=2023)
        tr = Trainer(types.SimpleNamespace(train_dataloader=loader))
        tr.create_optimizer(model)
        ep = [tr.train_epoch(model, e)[0] for e in range(2)]
        res[graph] = (ep, model.user_embeds.detach().clone())
        assert len(loader) >= 3 and len(loader.dataset) % 512 != 0          # the last batch is smaller: eager path inside the graphed epoch
    configs['train']['cuda_graph'] = False
    for a, b in zip(res[True][0], res[False][0]):
        assert abs(a - b) <= 1e-5 * max(1.0, abs(b)), res
    assert torch.allclose(res[True][1], res[False][1], rtol=1e-5, atol=3e-4)


def _reference_chains_full_predict(case, layer_num, n_users_scored):
    """The reference's CPU full_predict (lightgcn.py:31-43,58-66 without a mask) restated as the FMA chains its operators evaluate (pinned by
    tests/test_host_emulation.py), emulated in float64 (a product of two floats is exact in double; one extra rounding per step)."""
    adj = O.normalized_adjacency(case['rows'], case['cols'], case['n_user'], case['n_item'])
    order = np.lexsort((adj.cols, adj.rows))
    r, c, w = adj.rows[order], adj.cols[order], adj.vals[order].astype(np.float64)
    n = adj.n
    start = np.zeros(n + 1, dtype=np.int64)
    start[1:] = np.cumsum(np.bincount(r, minlength=n))
    deg = np.diff(start)
    x = np.concatenate([case['user_e'].numpy(), case['item_e'].numpy()], 0).astype(np.float32)
    total = x.copy()
    for _ in range(layer_num):
        y = np.zeros_like(x)
        for k in range(int(deg.max())):                          # the k-th stored entry of every row that has one: per row still sequential
            rows = np.flatnonzero(deg > k)
            e = start[rows] + k
            y[rows] = (w[e, None] * x[c[e]].astype(np.float64) + y[rows].astype(np.float64)).astype(np.float32)
        x = y
        total = total + x                                        # ((E0 + X1) + X2) + ...
    a, b = total[:n_users_scored], total[case['n_user']:]
    s = np.zeros((a.shape[0], b.shape[0]), dtype=np.float32)
    for q in range(a.shape[1]):
        s = (a[:, q:q + 1].astype(np.float64) * b[:, q].astype(np.float64)[None, :] + s.astype(np.float64)).astype(np.float32)
    return s


def test_exact_order_full_predict_reproduces_the_reference_cpu_scores_bit_for_bit():
    from sslrec_b200.config import configs
    g = replay.load_golden('lightgcn', 'small')
    case = inputs.make_case('small')
    model, _ = H.make_model('lightgcn', case, g['hp'])
    model.load_state_dict({'user_embeds': case['user_e'], 'item_embeds': case['item_e']})
    n_scored = min(64, case['n_user'])
    configs['test']['exact_order'] = True
    try:
        model.eval()
        with torch.no_grad():
            preds = model.full_predict([torch.arange(n_scored).cuda(), None]).cpu().numpy()
    finally:
        configs['test']['exact_order'] = False
    want = _reference_chains_full_predict(case, g['hp']['layer_num'], n_scored)
    equal = float((preds == want).mean())
    print(f'exact-order full_predict: {equal:.6f} of {want.size} scores bit-equal to the reference operators\' chains')
    assert equal >= 0.9999, equal
