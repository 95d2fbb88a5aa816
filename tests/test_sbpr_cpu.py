"""SBPR drop-in (f-4 sibling model: model/ranking/SBPR.py mirror) on the CPU.

(1) the item sets and the minibatch sampler against the UNMODIFIED reference class, recorded on the same inputs in
    tests/golden/sbpr_reference_sampler.json.xz (oracle/gen_golden.py social): same PositiveSet / FPSet, same
    (u, i, k, j, S_uk) batches from the same `random` state, same generator state afterwards;
    and (portable: no reference checkout needed) against the golden record oracle/gen_golden.py made from the unmodified
    reference class on FilmTrust with its real trust network (tests/golden/sbpr_filmtrust_seed77.npz);
(2) the numpy path stops where the reference's does (SBPR.py:47, TypeError);
(3) trainModel_tf, with the kernels replaced by stand-ins that follow include/qrec.h, against float64 autograd of the
    loss SBPR.py:110-114 states plus the oracle's TF1 Adam (TensorFlow is absent: parity unpinned for this part)."""
import contextlib
import io
import os
import random

import numpy as np
import pytest

from oracle import golden_json
from qrec_b200.util.config import ModelConf
from test_bpr_model_cpu import _stub_engine
from test_tbpr_cpu import _data

CONF = '''ratings=x
social=x
ratings.setup=-columns 0 1 2
social.setup=-columns 0 1
model.name=SBPR
evaluation.setup=-testSet x -b 1.0 -tf
item.ranking=on -topN 10
num.factors=10
num.max.epoch=2
batch_size=700
learnRate=-init 0.005 -max 0.1
reg.lambda=-u 0.01 -i 0.01 -b 0.01 -s 0.2
output.setup=off -dir ./results/
'''


def _model(golden_bpr, n_train=3000):
    from qrec_b200.model.ranking.SBPR import SBPR
    train, test, rel = _data(golden_bpr, n_train)
    m = SBPR(ModelConf.from_string(CONF), train, test, [list(r) for r in rel])
    with contextlib.redirect_stdout(io.StringIO()):
        m.readConfiguration()
        m.initModel()
    return m, train, test, rel


def test_sbpr_item_sets_and_numpy_path_error(golden_bpr, monkeypatch, tmp_path):
    calls = []
    _stub_engine(monkeypatch, calls)
    monkeypatch.chdir(tmp_path)
    m, train, _, _ = _model(golden_bpr)
    assert sum(len(v) for v in m.PositiveSet.values()) == len(train)
    fp_users = [u for u in m.FPSet if len(m.FPSet[u]) > 0]
    assert len(fp_users) > 10
    for u in fp_users[:50]:
        assert not (set(m.FPSet[u]) & set(m.PositiveSet[u]))                    # social feedback excludes the user's own items
        friends = [f for f in m.social.getFollowees(u) if f in m.data.user]
        for item, cnt in list(m.FPSet[u].items())[:20]:
            assert cnt == sum(1 for f in friends if item in m.data.trainSet_u[f]) >= 1
    with contextlib.redirect_stdout(io.StringIO()), pytest.raises(TypeError, match='unhashable'):
        m.trainModel()                                                          # SBPR.py:47
    # batches: training-data order, ragged last batch, negatives outside the rated and the social sets
    random.seed(3)
    m.batch_size = 700
    batches = list(m.next_batch())
    assert [len(b[0]) for b in batches] == [700, 700, 700, 700, 200]
    # the native sampler (qrec_sample_sbpr_batch) and the same loop in Python: same rows, same generator state afterwards
    native_state = random.getstate()
    random.seed(3)
    python_batches = list(m._next_batch_python())
    assert random.getstate() == native_state
    for a, b in zip(batches, python_batches):
        assert all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(a, b))
    flat_u = [x for b in batches for x in b[0]]
    assert flat_u == [m.data.user[r[0]] for r in m.data.trainingData]
    id2item = {v: k for k, v in m.data.item.items()}
    id2user = {v: k for k, v in m.data.user.items()}
    for u, i, k, j, w in zip(*batches[0]):
        user = id2user[u]
        assert id2item[j] not in m.data.trainSet_u[user] and id2item[j] not in m.FPSet[user]
        assert (w == 0 and len(m.FPSet[user]) == 0) or m.FPSet[user][id2item[k]] == w


def test_sbpr_sampler_equals_unmodified_reference_class(golden_bpr, monkeypatch, tmp_path):
    calls = []
    _stub_engine(monkeypatch, calls)
    monkeypatch.chdir(tmp_path)
    m, train, test, rel = _model(golden_bpr)
    ref = golden_json.load(os.path.join(os.path.dirname(__file__), 'golden', 'sbpr_reference_sampler.json.xz'))
    assert ref['positive'] == {u: dict(v) for u, v in m.PositiveSet.items() if v}
    assert {u: v for u, v in ref['fp'].items() if v} == {u: dict(v) for u, v in m.FPSet.items() if v}
    for u in ref['fp']:
        assert list(ref['fp'][u].keys()) == list(m.FPSet[u].keys())          # `choice(list(keys))` depends on the order
    random.seed(77)
    m.batch_size = 700
    ours = [tuple(list(x) for x in b) for b in m.next_batch()]
    assert random.getstate() == ref['state']
    assert len(ours) == len(ref['batches']) == 5
    for a, b in zip(ours, ref['batches']):
        assert a == b


def test_sbpr_trainModel_tf_composition_equals_autograd_restatement(golden_bpr, monkeypatch, tmp_path):
    import torch
    from oracle import bpr_oracle as O, tf_models as T
    from qrec_b200 import engine as E
    calls = []
    _stub_engine(monkeypatch, calls)

    def grad_scaled(U, V, u, i, j, y_scale, eps, reg, gU, gV, loss):
        """include/qrec.h: -ln(sigmoid(c_k y_k) + eps), dL/dy = -c s(1-s)/(s+eps); float64 numpy restatement."""
        calls.append(('grad_scaled', len(u)))
        Un, Vn = U.numpy().astype(np.float64), V.numpy().astype(np.float64)
        un, inn, jn, c = u.numpy(), i.numpy(), j.numpy(), y_scale.numpy().astype(np.float64)
        y = c * ((Un[un] * (Vn[inn] - Vn[jn])).sum(1))
        s = 1.0 / (1.0 + np.exp(-y))
        gy = (-s * (1.0 - s) / (s + eps) * c)[:, None]
        a, b = np.zeros_like(Un), np.zeros_like(Vn)
        np.add.at(a, un, gy * (Vn[inn] - Vn[jn]))
        np.add.at(b, inn, gy * Un[un])
        np.add.at(b, jn, -gy * Un[un])
        assert reg == 0.0
        gU += torch.from_numpy(a).float(); gV += torch.from_numpy(b).float()
        loss += float(-np.log(s + eps).sum())
    monkeypatch.setattr(E, 'bpr_grad_scatter_scaled', grad_scaled)
    monkeypatch.chdir(tmp_path)
    m, train, test, rel = _model(golden_bpr)
    random.seed(21); torch.manual_seed(5)
    with contextlib.redirect_stdout(io.StringIO()):
        m.trainModel_tf()
    assert [c[1] for c in calls if c[0] == 'grad_scaled'] == [700, 700, 700, 700, 200] * 2
    assert [c[1] for c in calls if c[0] == 'grad'] == [700, 700, 700, 700, 200] * 2
    # restatement: same initial tables, same batches, autograd of the stated loss (no regulariser: SBPR.py:115 is a
    # statement of its own), TF1 Adam
    torch.manual_seed(5)
    d, nu, ni = m.emb_size, m.num_users, m.num_items
    U = torch.nn.init.trunc_normal_(torch.empty(nu, d), std=0.005, a=-0.01, b=0.01).numpy().copy()
    V = torch.nn.init.trunc_normal_(torch.empty(ni, d), std=0.005, a=-0.01, b=0.01).numpy().copy()
    mU, vU, mV, vV = (np.zeros_like(x) for x in (U, U, V, V))
    random.seed(21)
    t = 0
    for epoch in range(2):
        for u, i, k, j, w in m.next_batch():
            t += 1
            _, gU, gV = T.sbpr_loss_and_grad(U, V, u, i, k, j, w)           # oracle/tf_models.py (SBPR.py:103-115)
            O.adam_tf1(U, mU, vU, gU.astype(np.float32), m.lRate, t)
            O.adam_tf1(V, mV, vV, gV.astype(np.float32), m.lRate, t)
    np.testing.assert_allclose(m.P, U, rtol=1e-3, atol=1e-5)
    np.testing.assert_allclose(m.Q, V, rtol=1e-3, atol=1e-5)
    assert float(np.abs(m.P).max()) > 0.01


def test_sbpr_sets_and_sampler_equal_golden_reference_record(golden_bpr, monkeypatch, tmp_path):
    """FilmTrust + its trust network: FPSet (sizes, count sums, first key = insertion order) and the first eight
    512-sample minibatches (u, i, k, j, S_uk) from random.seed(77), and the generator state after them, equal what the
    unmodified reference class produced (oracle/gen_golden.py gen_sbpr)."""
    from qrec_b200.model.ranking.SBPR import SBPR
    calls = []
    _stub_engine(monkeypatch, calls)
    monkeypatch.chdir(tmp_path)
    gs = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'sbpr_filmtrust_seed77.npz'), allow_pickle=False)
    g = golden_bpr
    train = [[u, i, float(r)] for u, i, r in zip(g['train_users'].tolist(), g['train_items'].tolist(), g['train_rating'].tolist())]
    rel = [[a, b, w] for a, b, w in zip(gs['relation_from'].tolist(), gs['relation_to'].tolist(), gs['relation_w'].tolist())]
    conf = str(gs['conf']).replace('./dataset/FilmTrust/ratings.txt', 'x').replace('./dataset/FilmTrust/trust.txt', 'x') \
                          .replace('./dataset/FilmTrust/testset.txt', 'x')
    np.random.seed(0); random.seed(0)
    m = SBPR(ModelConf.from_string(conf), train, [], rel)
    with contextlib.redirect_stdout(io.StringIO()):
        m.readConfiguration()
        m.initModel()
    users = list(m.data.user.keys())
    assert np.array_equal(np.array([len(m.FPSet[u]) for u in users]), gs['fp_sizes'])
    assert np.array_equal(np.array([sum(m.FPSet[u].values()) for u in users]), gs['fp_sums'])
    assert [next(iter(m.FPSet[u])) if len(m.FPSet[u]) else '' for u in users] == gs['fp_first'].tolist()
    m.batch_size = 512
    random.seed(77)
    for n, b in enumerate(m.next_batch()):
        assert np.array_equal(np.array(b, dtype=np.int64), gs['batches'][n]), 'batch %d' % n
        if n == 7:
            break
    assert np.array_equal(np.array(random.getstate()[1], dtype=np.uint32), gs['mt_state_after_8_batches'])
