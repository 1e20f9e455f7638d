"""Generate the two host-side golden files of tests/test_host.py by running the UNMODIFIED reference (HKUDS/SSLRec) on CPU.
TEST INFRASTRUCTURE ONLY: the outputs are committed, so the tests never need the reference.

    python oracle/gen_host_golden.py --reference PATH/TO/SSLRec

tests/golden/ref_metric_eval_batch.npz
    ``trainer.metrics.Metric.eval_batch`` (all four metrics, k = 5 / 20 / 40) on seeded random top-k lists and ground
    truths; the inputs are stored next to the reference's per-k sums.
tests/golden/ref_pairwise_batches.npz
    The reference's training data path -- ``data_utils.datasets_general_cf.PairwiseTrnData`` (per-pair rejection loop of
    ``sample_negs``) served by ``DataLoader(batch_size=128, shuffle=True)`` -- over two epochs after ``np.random.seed(11)``
    and ``torch.manual_seed(12)`` on a dense 90 x 30 graph: every (user, positive, negative) batch and the head of both RNG
    states afterwards.

The reference's config module parses ``sys.argv`` and reads its YAML relative to the working directory at import, so the
reference runs in a subprocess started in its own directory.  No reference source is modified or copied.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, 'tests', 'golden')

BODY = r'''
import os, sys
import numpy as np, scipy.sparse as sp, torch
import torch.utils.data as tdata
ref, out = sys.argv[1], sys.argv[2]
os.chdir(ref)
sys.path.insert(0, ref)
sys.argv = ['main.py', '--model', 'lightgcn', '--device', 'cpu']
from config.configurator import configs

# ---- Metric.eval_batch on seeded top-k lists (the inputs of test_vectorised_metrics_match_the_reference_metric_class) ----
metrics, ks = ['recall', 'ndcg', 'precision', 'mrr'], [5, 20, 40]
configs['test']['metrics'] = metrics
configs['test']['k'] = ks
from trainer.metrics import Metric
rs = np.random.RandomState(5)
n, n_item, kmax = 300, 500, 40
top = np.stack([rs.permutation(n_item)[:kmax] for _ in range(n)])
truths = [rs.choice(n_item, size=rs.randint(1, 50), replace=False).tolist() for _ in range(n)]
for u in range(n):
    for _ in range(rs.randint(0, 5)):
        top[u, rs.randint(0, kmax)] = truths[u][rs.randint(len(truths[u]))]
want = Metric().eval_batch((torch.from_numpy(top), truths), ks)
np.savez_compressed(os.path.join(out, 'ref_metric_eval_batch.npz'), top=top.astype(np.int32),
                    truth_ptr=np.cumsum([0] + [len(t) for t in truths]).astype(np.int64),
                    truth_flat=np.concatenate([np.asarray(t, dtype=np.int32) for t in truths]),
                    ks=np.asarray(ks, dtype=np.int64), metrics=np.asarray(metrics),
                    **{'want_' + m: np.asarray(want[m], dtype=np.float64) for m in metrics})

# ---- PairwiseTrnData + DataLoader(shuffle=True): two epochs under fixed numpy / torch seeds ----
rs = np.random.RandomState(0)
U, I = 90, 30
key = np.unique(rs.randint(0, U, 1500).astype(np.int64) * I + rs.randint(0, I, 1500))
m = sp.coo_matrix((np.ones(len(key)), (key // I, key % I)), shape=(U, I))
configs['data']['user_num'], configs['data']['item_num'] = U, I
from data_utils.datasets_general_cf import PairwiseTrnData
ds = PairwiseTrnData(m)
loader = tdata.DataLoader(ds, batch_size=128, shuffle=True, num_workers=0)
np.random.seed(11); torch.manual_seed(12)
rec = {}
for epoch in range(2):
    ds.sample_negs()
    batches = [[t.long().numpy() for t in b] for b in loader]
    rec[f'epoch{epoch}_batch_len'] = np.asarray([len(b[0]) for b in batches], dtype=np.int64)
    rec[f'epoch{epoch}_triples'] = np.stack([np.concatenate([b[i] for b in batches]) for i in range(3)]).astype(np.int32)
np.savez_compressed(os.path.join(out, 'ref_pairwise_batches.npz'), key=key, n_user=U, n_item=I, batch_size=128,
                    numpy_state_head=np.random.get_state()[1][:8].astype(np.int64),
                    torch_state_head=torch.get_rng_state()[:16].numpy().astype(np.int64), **rec)
print('wrote', os.path.join(out, 'ref_metric_eval_batch.npz'), os.path.join(out, 'ref_pairwise_batches.npz'))
'''


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reference', default=os.environ.get('SSLREC_REFERENCE'), help='checkout of the reference (HKUDS/SSLRec)')
    a = ap.parse_args()
    if not a.reference or not os.path.isdir(os.path.join(a.reference, 'trainer')):
        raise SystemExit('--reference must point at a checkout of the reference (HKUDS/SSLRec)')
    os.makedirs(OUT, exist_ok=True)
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE='1')
    subprocess.run([sys.executable, '-c', BODY, os.path.abspath(a.reference), OUT], check=True, env=env)


if __name__ == '__main__':
    main()
