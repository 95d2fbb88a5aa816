"""Differential tests of the Python drop-in surface against the UNMODIFIED reference modules, on
randomised inputs.  The reference's outputs on the same seeded inputs are recorded in
tests/golden/differential_reference.json.xz (oracle/gen_golden.py differential); FilmTrust's ratings file
is tests/golden/filmtrust_ratings.txt.xz.  Nothing here is imported by the product."""
import lzma
import os
import random

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import golden_json


@pytest.fixture(scope='module')
def ref():
    """What the reference modules returned, one entry per test below."""
    return golden_json.load(os.path.join(GOLDEN, 'differential_reference.json.xz'))


@pytest.fixture(scope='module')
def filmtrust_ratings(tmp_path_factory):
    path = tmp_path_factory.mktemp('filmtrust') / 'ratings.txt'
    with lzma.open(os.path.join(GOLDEN, 'filmtrust_ratings.txt.xz')) as f:
        path.write_bytes(f.read())
    return str(path)


def test_option_conf_equals_reference_on_random_strings(ref):
    from qrec_b200.util.config import OptionConf
    rng = random.Random(0)
    vocab = ['on', 'off', '-a', '-b', '--c', '-topN', '-1', '-12', '-0.5', '5', '10,20', 'x', '0.1', '-tf', '', '-n_layer', '2']
    for options, main_on, line in ref['option_conf']:
        s = ' '.join(rng.choice(vocab) for _ in range(rng.randint(1, 8)))
        if rng.random() < 0.2:
            s = ' ' + s + ' '
        mine = OptionConf(s)
        assert mine.options == options, repr(s)
        assert mine.isMainOn() == main_on and mine.line == line
    assert len(ref['option_conf']) == 3000


def test_model_conf_equals_reference(ref, tmp_path):
    from qrec_b200.util.config import ModelConf
    assert len(ref['model_conf']) == 46                # every config/*.conf of the reference
    for name, text, config in ref['model_conf']:
        path = tmp_path / name
        path.write_text(text)
        assert ModelConf(str(path)).config == config, name
    bad = tmp_path / 'bad.conf'
    bad.write_text('a=1\nnot a pair\nb=2=3\n\nc=x y\n')
    assert ModelConf(str(bad)).config == ref['model_conf_bad'] == {'a': '1', 'c': 'x y'}


def test_measures_equal_reference_on_random_rankings(ref):
    from qrec_b200.util.measure import Measure
    rng = random.Random(1)
    items = ['i%d' % k for k in range(60)]
    for case in range(200):
        users = ['u%d' % k for k in range(rng.randint(1, 12))]
        origin = {u: {it: 1.0 for it in rng.sample(items, rng.randint(1, 15))} for u in users}
        res = {u: [(it, rng.random()) for it in rng.sample(items, 20)] for u in users}
        tops = sorted(rng.sample([1, 3, 5, 10, 20], rng.randint(1, 3)))
        assert Measure.rankingMeasure(origin, res, tops) == ref['ranking_measure'][case]
    rows = [['u', 'i', rng.random() * 5, rng.random() * 5] for _ in range(50)]
    assert Measure.ratingMeasure(rows) == ref['rating_measure'][0]
    assert Measure.ratingMeasure([]) == ref['rating_measure'][1]


def test_find_k_largest_equals_reference_numba_heap(ref):
    from qrec_b200.util.qmath import find_k_largest, sigmoid
    rng = np.random.default_rng(2)
    for trial in range(120):
        n, K = int(rng.integers(3, 300)), int(rng.integers(1, 15))
        s = rng.standard_normal(n).round(1 if trial % 3 == 0 else 7)
        s[rng.integers(0, n, n // 5)] = 0.0                       # rated items are overwritten with 0
        ids, vals = find_k_largest(K, s.copy())
        rid, rvals = ref['find_k_largest'][trial]
        assert list(ids) == list(rid) and list(vals) == list(rvals), (trial, n, K)
    assert sigmoid(0.3) == ref['sigmoid_0.3']


def test_rating_equals_reference_on_random_data(ref):
    from qrec_b200.data.rating import Rating
    from qrec_b200.util.config import ModelConf
    rng = random.Random(3)
    for ev, theirs in zip(('-ap 0.2', '-ap 0.2 -b 1', '-cold 2', '-val 0.25'), ref['rating']):
        conf_text = 'ratings=x\nevaluation.setup=%s\n' % ev
        train = [['u%d' % rng.randint(0, 30), 'i%d' % rng.randint(0, 40), float(rng.randint(1, 5))] for _ in range(400)]
        test = [['u%d' % rng.randint(0, 35), 'i%d' % rng.randint(0, 45), float(rng.randint(1, 5))] for _ in range(120)]
        random.seed(11)
        mine = Rating(ModelConf.from_string(conf_text), [r[:] for r in train], [r[:] for r in test])
        for attr in ('user', 'item', 'id2user', 'id2item', 'userMeans', 'itemMeans', 'globalMean', 'rScale',
                     'trainingData', 'testData'):
            assert getattr(mine, attr) == theirs[attr], (ev, attr)
        assert dict(mine.trainSet_u) == theirs['trainSet_u'] and dict(mine.testSet_u) == theirs['testSet_u']
        assert dict(mine.trainSet_i) == theirs['trainSet_i'] and dict(mine.testSet_i) == theirs['testSet_i']
        assert mine.trainingSize() == theirs['trainingSize'] and mine.testSize() == theirs['testSize']
        u0 = next(iter(mine.user))
        assert u0 == theirs['u0']
        assert mine.userRated(u0) == theirs['userRated'] and np.array_equal(mine.row(u0), theirs['row'])


def test_data_split_and_cv_equal_reference(ref):
    from qrec_b200.util.dataSplit import DataSplit
    split, cv = ref['data_split']
    rng = random.Random(5)
    data = [['u%d' % rng.randint(0, 9), 'i%d' % rng.randint(0, 9), float(rng.randint(0, 1))] for _ in range(300)]
    for (ratio, binar), (b, st_b) in zip(((0.2, False), (0.2, True), (1.5, False), (0.0, True)), split):
        random.seed(7)
        a = DataSplit.dataSplit(data, test_ratio=ratio, binarized=binar)
        assert a == b and random.getstate() == st_b
    for (k, binar), b in zip(((5, False), (3, True), (1, False), (11, False)), cv):
        assert list(DataSplit.crossValidation(data, k, binarized=binar)) == b


def test_loader_equals_reference_on_shipped_datasets(ref, filmtrust_ratings):
    from qrec_b200.util.io import FileIO
    from qrec_b200.util.config import ModelConf
    path = filmtrust_ratings
    for (setup, kw), (n, head, digest) in zip((('-columns 0 1 2', {}), ('-columns 0 1 2', {'binarized': True, 'threshold': 3.0}),
                                               ('-columns 1 0', {}), ('-columns 0 1 2 -header', {'bTest': True})),
                                              ref['load_filmtrust']):
        mine_conf = ModelConf.from_string('ratings.setup=%s\n' % setup)
        import contextlib, io
        with contextlib.redirect_stdout(io.StringIO()):
            a = FileIO.loadDataSet(mine_conf, path, **kw)
        assert len(a) == n and a[:5] == head, setup
        assert golden_json.digest(a) == digest, setup


def test_eval_ranking_and_lr_schedule_equal_reference(ref, tmp_path, monkeypatch):
    """Recommender.evalRanking / IterativeRecommender.isConverged of the mirror classes against the
    reference classes, both fed the same numpy P, Q: identical recommendation lines, metric strings,
    learning-rate updates and generator state."""
    import contextlib
    import io
    from qrec_b200.base.iterativeRecommender import IterativeRecommender as Mine
    from qrec_b200.util.config import ModelConf
    monkeypatch.chdir(tmp_path)
    rng = random.Random(9)
    conf_text = ('ratings=x\nratings.setup=-columns 0 1 2\nmodel.name=BPR\nevaluation.setup=-ap 0.2 -b 1\n'
                 'item.ranking=on -topN 5,10\nnum.factors=8\nnum.max.epoch=3\nlearnRate=-init 0.01 -max 0.0105\n'
                 'reg.lambda=-u 0.001 -i 0.001 -b 0.2 -s 0.2\noutput.setup=on -dir ./results/\n')
    train = [['u%d' % rng.randint(0, 40), 'i%d' % rng.randint(0, 60), 1.0] for _ in range(900)]
    test = [['u%d' % rng.randint(0, 45), 'i%d' % rng.randint(0, 60), 1.0] for _ in range(200)]
    m = Mine(ModelConf.from_string(conf_text), [r[:] for r in train], [r[:] for r in test])
    with contextlib.redirect_stdout(io.StringIO()):
        m.readConfiguration()
        m.initializing_log()
        np.random.seed(4)
        m.initModel()
        random.seed(21)
        conv = []
        for epoch, loss in enumerate([100.0, 90.0, 95.0, 94.9995], 1):
            m.loss = loss
            conv.append((m.isConverged(epoch), m.lRate))
        m.evalRanking()
    outs = [(conv, m.recOutput, m.measure, random.getstate(), [r[:] for r in m.data.trainingData]), ref['eval_ranking']]
    assert outs[0][0] == outs[1][0]                 # convergence flags + lr after 1.05x / 0.5x / clamp
    assert outs[0][1] == outs[1][1]                 # every recommendation line, scores included
    assert outs[0][2] == outs[1][2]                 # metric strings
    assert outs[0][3] == outs[1][3] and outs[0][4] == outs[1][4]   # MT19937 state and shuffled list


@pytest.mark.parametrize('seed', [0, 7, 2024])
def test_minibatch_samplers_equal_reference_on_random_data(ref, tmp_path, monkeypatch, seed):
    """DeepRecommender.next_batch_pairwise / next_batch_pointwise (C MT19937 clone underneath) against
    the reference generators (Python `random`) on random interaction lists with duplicates and
    non-binary ratings: every batch, the shuffled list and the generator state afterwards."""
    import contextlib
    import io
    from qrec_b200.base.deepRecommender import DeepRecommender as Mine
    from qrec_b200.util.config import ModelConf
    monkeypatch.chdir(tmp_path)
    rng = random.Random(seed)
    conf_text = ('ratings=x\nratings.setup=-columns 0 1 2\nmodel.name=LightGCN\nevaluation.setup=-ap 0.2\n'
                 'item.ranking=on -topN 10\nnum.factors=8\nnum.max.epoch=1\nbatch_size=128\n'
                 'learnRate=-init 0.01 -max 1\nreg.lambda=-u 0.001 -i 0.001 -b 0.2 -s 0.2\noutput.setup=off -dir ./results/\n')
    train = [['u%d' % rng.randint(0, 50), 'i%d' % rng.randint(0, 80), float(rng.randint(1, 5))] for _ in range(1000)]
    m = Mine(ModelConf.from_string(conf_text), [r[:] for r in train], [])
    with contextlib.redirect_stdout(io.StringIO()):
        m.readConfiguration()
    random.seed(seed)
    pair = [tuple(np.asarray(x).tolist() for x in batch) for batch in m.next_batch_pairwise()]
    point = [tuple(np.asarray(x).tolist() for x in batch) for batch in m.next_batch_pointwise()]
    n_pair, pair_digest, point_digest, train_digest, state = ref['minibatch'][seed]
    assert len(pair) == n_pair == 8 and len(pair[-1][0]) == 1000 - 7 * 128
    assert golden_json.digest(pair) == pair_digest          # pairwise batches (u, i, j)
    assert golden_json.digest(point) == point_digest        # pointwise batches (u, i, y), 5 rows per interaction
    assert golden_json.digest([r[:] for r in m.data.trainingData]) == train_digest and random.getstate() == state


def test_interaction_table_equals_reference_loader_and_rating(ref, filmtrust_ratings):
    """f-3: the array-backed table built from the shipped FilmTrust file has the reference's id space."""
    from qrec_b200.data.interactions import InteractionTable
    data = ref['table_filmtrust']
    t = InteractionTable.from_text(filmtrust_ratings, binarize_threshold=1.0)
    assert len(t) == data['n'] == 34437
    assert t.user_names.tolist() == data['user_names']
    assert t.item_names.tolist() == data['item_names']
    assert golden_json.digest(t.u.tolist()) == data['u_digest'] and golden_json.digest(t.i.tolist()) == data['i_digest']
