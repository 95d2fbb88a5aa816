"""Host-side logic of the drop-in class surface (no GPU): config parsing quirks, id mapping,
metrics, top-K, the data pipeline against the reference's recorded split."""
import os
import random

import numpy as np
import pytest

from conftest import adjacency_kernel_stand_ins

from qrec_b200.util.config import ModelConf, OptionConf
from qrec_b200.util.measure import Measure
from qrec_b200.util.qmath import find_k_largest, _heap_top_k
from qrec_b200.data.rating import Rating


def test_option_conf_behaviour_table():
    # SURVEY.md App. B6, observed on the reference's util/config.py
    assert OptionConf('-cv 5 -b 1.0 -tf').options == {'-cv': '5', '-b': '1.0', '-tf': ''}
    o = OptionConf('on -topN 10')
    assert o.isMainOn() and o.options == {'-topN': '10'}
    o = OptionConf('off -topN -1')
    assert not o.isMainOn() and o['-topN'] == '-1'
    assert OptionConf(' -n_layer 2')['-n_layer'] == '2'
    assert OptionConf('-columns 0 1 2')['-columns'] == '0 1 2'
    assert OptionConf('-n_layer 2 -lambda 0.5 -eps 0.1').options == {'-n_layer': '2', '-lambda': '0.5', '-eps': '0.1'}
    with pytest.raises(SystemExit):
        OptionConf('-a 1')['-missing']


def test_model_conf(tmp_path):
    p = tmp_path / 'm.conf'
    p.write_text('ratings=./x.txt\n\nmodel.name=BPR\nbroken line\nlearnRate=-init 0.01 -max 1\n')
    c = ModelConf(str(p))
    assert c['model.name'] == 'BPR' and c.contains('learnRate') and not c.contains('broken line')
    with pytest.raises(SystemExit):
        c['nope']
    with pytest.raises(IOError):
        ModelConf(str(tmp_path / 'absent.conf'))


def _conf(text):
    return ModelConf.from_string(text)


def test_rating_id_space_matches_reference(golden_bpr):
    g = golden_bpr
    train = [[u, i, r] for u, i, r in zip(g['train_users'].tolist(), g['train_items'].tolist(), g['train_rating'].tolist())]
    test = [[u, i, r] for u, i, r in zip(g['test_users'].tolist(), g['test_items'].tolist(), g['test_rating'].tolist())]
    data = Rating(_conf(str(g['conf'])), train, test)
    assert data.trainingSize() == (1484, 1891, 27555)
    assert [data.id2user[k] for k in range(len(data.user))] == g['user_names'].tolist()
    assert [data.id2item[k] for k in range(len(data.item))] == g['item_names'].tolist()
    csr = data.rated_csr()
    assert csr.num_positives == g['triples_epoch'].shape[1]
    # CSR order of positives == the (u, i) columns of the reference's first-epoch stream
    t = g['triples_epoch'][0]
    assert np.array_equal(csr.pos_cols, t[:, 1])
    assert np.array_equal(np.repeat(np.arange(1484), np.diff(csr.pos_rowptr)), t[:, 0])
    assert data.globalMean == 1.0 and data.rScale == [1.0]
    u, i, r = data.training_ids()
    assert len(u) == 27555 and u.dtype == np.int32


def test_find_k_largest_same_as_heap_algorithm():
    rng = np.random.default_rng(0)
    for trial in range(50):
        n = int(rng.integers(5, 400))
        K = int(rng.integers(1, 12))
        s = rng.standard_normal(n).round(1 if trial % 2 else 6)      # odd trials: many ties
        s[rng.integers(0, n, n // 4)] = 0.0
        ids, vals = find_k_largest(K, s.copy())
        rid, rval = _heap_top_k(K, s.copy())
        assert ids == rid and vals == rval
    assert find_k_largest(3, np.array([1.0, 5.0, 2.0, 4.0]))[0] == [1, 3, 2]


def test_measure_definitions():
    origin = {'a': {'x': 1, 'y': 1}, 'b': {'z': 1}}
    res = {'a': [('x', .9), ('q', .8), ('y', .7)], 'b': [('q', .5), ('w', .4), ('z', .3)]}
    m = Measure.rankingMeasure(origin, res, [3])
    import math
    assert m[0] == 'Top 3\n'
    assert m[1] == 'Precision:' + str(3 / 6) + '\n'
    assert m[2] == 'Recall:' + str((2 / 2 + 1 / 1) / 2) + '\n'
    ndcg_a = (1 / math.log(2) + 1 / math.log(4)) / (1 / math.log(2) + 1 / math.log(3))
    ndcg_b = (1 / math.log(4)) / (1 / math.log(2))
    assert m[4] == 'NDCG:' + str((ndcg_a + ndcg_b) / 2) + '\n'
    assert Measure.ratingMeasure([['u', 'i', 3.0, 2.0], ['u', 'j', 1.0, 2.0]]) == ['MAE:1.0\n', 'RMSE:1.0\n']


def test_loader_and_split_reproduce_reference_split(golden_bpr, tmp_path, monkeypatch):
    """QRec.__init__ (QRec.py:8-47): loadDataSet + seeded -ap split of FilmTrust's ratings file
    (tests/golden/filmtrust_ratings.txt.xz) give the recorded training list and leave Python's MT19937
    in the recorded state."""
    import lzma
    from conftest import GOLDEN
    from qrec_b200.QRec import QRec
    monkeypatch.chdir(tmp_path)
    os.makedirs('dataset/FilmTrust')
    with lzma.open(os.path.join(GOLDEN, 'filmtrust_ratings.txt.xz')) as f:
        (tmp_path / 'dataset' / 'FilmTrust' / 'ratings.txt').write_bytes(f.read())
    random.seed(0)
    q = QRec(_conf(str(golden_bpr['conf'])))
    assert [r[0] for r in q.trainingData] == golden_bpr['train_users'].tolist()
    assert [r[1] for r in q.trainingData] == golden_bpr['train_items'].tolist()
    assert [r[0] for r in q.testData] == golden_bpr['test_users'].tolist()
    assert np.array_equal(np.array(random.getstate()[1], dtype=np.uint32), golden_bpr['mt_state_after_split'])


def test_shuffle_training_data_equals_random_shuffle(golden_bpr):
    from qrec_b200.base.iterativeRecommender import IterativeRecommender
    g = golden_bpr
    train = [[u, i, r] for u, i, r in zip(g['train_users'].tolist()[:500], g['train_items'].tolist()[:500], [1.0] * 500)]
    m = IterativeRecommender(_conf(str(g['conf'])), train, [])
    random.seed(5)
    expect = m.data.trainingData[:]
    random.shuffle(expect)
    st = random.getstate()
    random.seed(5)
    m.shuffle_training_data()
    assert m.data.trainingData == expect and random.getstate() == st


def test_device_adjacency_builder_equals_reference_matrix(golden_graph, graph_ids, monkeypatch):
    """graph_build.norm_adjacency_csr (structure by sort + run-length, here on CPU tensors; the value kernels
    replaced by numpy stand-ins) reproduces the scipy matrix of base/graphRecommender.py:10-29 recorded from
    the reference -- structure exactly, values to fp32 rounding -- including summed duplicate interactions and
    an isolated node."""
    import torch
    from qrec_b200.graph_build import norm_adjacency_csr
    adjacency_kernel_stand_ins(monkeypatch)
    g = golden_graph
    u, i, nu, ni = graph_ids
    rowptr, cols, vals = norm_adjacency_csr(torch.from_numpy(u), torch.from_numpy(i), nu, ni)
    assert np.array_equal(rowptr.numpy(), g['adj_indptr'])
    assert np.array_equal(cols.numpy(), g['adj_indices'])
    np.testing.assert_allclose(vals.numpy(), g['adj_data'], rtol=5e-7, atol=0)       # <= 2 ulp of fp32
    # duplicates are summed before normalisation; node without edges keeps an empty row
    from oracle import bpr_oracle as O
    uu = np.array([0, 0, 1, 1, 1, 3]); ii = np.array([2, 2, 0, 2, 0, 1])
    ref = O.norm_adjacency(5, 3, uu, ii)
    rp, co, va = norm_adjacency_csr(torch.from_numpy(uu), torch.from_numpy(ii), 5, 3)
    assert np.array_equal(rp.numpy(), ref.indptr) and np.array_equal(co.numpy(), ref.indices)
    np.testing.assert_allclose(va.numpy(), ref.data, rtol=5e-7)
    assert rp[3] == rp[2] and rp[5] == rp[4] + 0                       # users 2 and 4 are isolated


def test_device_csr_constructors_agree():
    """DeviceCSR from a scipy matrix and from device-built arrays expose the same fields (CPU tensors
    here; the kernels are exercised by the GPU suites)."""
    import scipy.sparse as sp
    import torch
    from qrec_b200.base.graphRecommender import DeviceCSR
    A = sp.random(30, 30, density=0.2, format='csr', dtype=np.float32, random_state=0)
    a = DeviceCSR(A, 'cpu')
    b = DeviceCSR.from_tensors(A.shape, a.rowptr, a.cols, a.vals)
    assert (a.nnz, a.shape, a.rowsplit) == (b.nnz, b.shape, b.rowsplit) and a.nnz == A.nnz
    for name in ('matmul', 'matmul_sparse_rows'):
        assert hasattr(b, name)
    long_row = sp.csr_matrix((np.ones(5000, np.float32), (np.zeros(5000, int), np.arange(5000))), shape=(2, 5000))
    assert DeviceCSR(long_row, 'cpu').rowsplit is False


def test_graph_recommender_adj_tensor_method_on_cpu_tensors(golden_graph, tmp_path, monkeypatch):
    """GraphRecommender.create_joint_sparse_adj_tensor end to end with the device stubbed to 'cpu':
    the DeviceCSR it returns holds the reference's matrix."""
    import torch
    from qrec_b200.base.graphRecommender import GraphRecommender
    g = golden_graph
    monkeypatch.chdir(tmp_path)
    train = [[u, i, 1.0] for u, i in zip(g['train_users'].tolist(), g['train_items'].tolist())]
    m = GraphRecommender(_conf(str(g['conf'])), train, [])
    monkeypatch.setattr(GraphRecommender, '_device', lambda self: torch.device('cpu'))
    adjacency_kernel_stand_ins(monkeypatch)
    adj = m.create_joint_sparse_adj_tensor()
    assert adj.shape == tuple(g['adj_shape']) and adj.nnz == len(g['adj_indices']) and adj.rowsplit
    assert np.array_equal(adj.rowptr.numpy(), g['adj_indptr']) and np.array_equal(adj.cols.numpy(), g['adj_indices'])
    np.testing.assert_allclose(adj.vals.numpy(), g['adj_data'], rtol=5e-7)
    # and the scipy-returning method is still the reference's matrix
    sp_adj = m.create_joint_sparse_adjaceny().tocsr(); sp_adj.sort_indices()
    assert np.array_equal(sp_adj.indices, g['adj_indices'])
    np.testing.assert_allclose(sp_adj.data, g['adj_data'], rtol=1e-6)


def test_vectorised_measures_equal_measure_class():
    """util/fastmeasure.ranking_measures == Measure.rankingMeasure (hence the reference's) on random
    rankings: same strings up to the last printed digit of the float sums."""
    import random as pyrandom
    from qrec_b200.util.fastmeasure import ranking_measures
    rng = pyrandom.Random(0)
    n_items = 80
    for trial in range(30):
        n_users = rng.randint(1, 25)
        tests = [rng.sample(range(n_items), rng.randint(1, 18)) for _ in range(n_users)]
        top = np.array([rng.sample(range(n_items), 20) for _ in range(n_users)])
        rowptr = np.zeros(n_users + 1, np.int64); rowptr[1:] = np.cumsum([len(t) for t in tests])
        cols = np.concatenate([np.array(t) for t in tests]).astype(np.int32)
        origin = {'u%d' % k: {'i%d' % it: 1.0 for it in tests[k]} for k in range(n_users)}
        res = {'u%d' % k: [('i%d' % it, 0.0) for it in top[k]] for k in range(n_users)}
        tops = sorted(rng.sample([1, 5, 10, 20], rng.randint(1, 3)))
        fast = ranking_measures(top, rowptr, cols, tops)
        slow = Measure.rankingMeasure(origin, res, tops)
        assert len(fast) == len(slow)
        for a, b in zip(fast, slow):
            if ':' not in a:
                assert a == b
            else:
                (ka, va), (kb, vb) = a.strip().split(':'), b.strip().split(':')
                assert ka == kb and abs(float(va) - float(vb)) <= 1e-12 * max(1.0, abs(float(vb)))
