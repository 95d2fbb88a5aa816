#!/usr/bin/env python
"""Golden-vector generator: runs the UNMODIFIED reference (a Coder-Yu/QRec checkout, found at
$QREC_REFERENCE_DIR) and records what the hot path consumed and produced.  TEST INFRASTRUCTURE
ONLY -- nothing in the product path imports this file, and no test needs the reference checkout:
the tests read only what this file wrote under tests/golden/.

What is exercised (reference file:line):
  * QRec.__init__            QRec.py:8-47        load FilmTrust, `-ap 0.2 -b 1` split
  * Rating.__generateSet     data/rating.py:33-67   first-appearance id maps
  * IterativeRecommender.initModel  base/iterativeRecommender.py:36-39
  * BPR.trainModel / optimization   model/ranking/BPR.py:19-53   (numpy float64 SGD)
  * IterativeRecommender.isConverged / updateLearningRate  base/iterativeRecommender.py:56-63,82-102
  * Recommender.evalRanking  base/recommender.py:127-179
  * DeepRecommender.next_batch_pairwise / next_batch_pointwise  base/deepRecommender.py:29-77
  * GraphRecommender.create_joint_sparse_adjaceny / create_sparse_rating_matrix
                              base/graphRecommender.py:10-29,41-51
  * BasicMF / PMF / SVD .trainModel   model/rating/BasicMF.py:9-25, PMF.py:9-28, SVD.py:9-36
    (pointwise sequential SGD; §8 f-4), with the per-epoch shuffle of isConverged and the
    MAE / RMSE of evalRatings (base/recommender.py:95-125, util/measure.py)
  * SBPR.initModel / next_batch   model/ranking/SBPR.py:12-29, 69-101 (social-feedback sets, minibatch sampler)
  * the host-side modules under differential test (gen_differential) and TBPR / SBPR on the inputs of
    their CPU tests (gen_social)

`tensorflow` and `mkl` are absent from this image; both are stubbed with empty
modules because the reference imports them at module level (model/ranking/BPR.py:7,
QRec.py:6).  The numpy path never calls into either.

Usage:  QREC_REFERENCE_DIR=<QRec checkout> python oracle/gen_golden.py [bpr] [mf] [sbpr] [differential] [social]
        (default: all sections; writes tests/golden/*.npz, *.json.xz, *.txt.xz; needs the built package for `social`)
"""
import os
import sys
import types
import random
import tempfile
import contextlib
import io

import numpy as np

REF = os.environ.get('QREC_REFERENCE_DIR', '')
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(REPO, 'tests', 'golden')

CONF_BPR = """ratings=./dataset/FilmTrust/ratings.txt
ratings.setup=-columns 0 1 2
model.name=BPR
evaluation.setup=-ap 0.2 -b 1
item.ranking=on -topN 10
num.factors=64
num.max.epoch=3
batch_size=2048
learnRate=-init 0.01 -max 1
reg.lambda=-u 0.001 -i 0.001 -b 0.2 -s 0.2
output.setup=on -dir ./results/
"""

CONF_LGCN = """ratings=./dataset/FilmTrust/ratings.txt
ratings.setup=-columns 0 1 2
model.name=LightGCN
evaluation.setup=-ap 0.2 -b 1
item.ranking=on -topN 10
num.factors=64
num.max.epoch=2
batch_size=2048
learnRate=-init 0.001 -max 1
LightGCN=-n_layer 3
reg.lambda=-u 0.001 -i 0.001 -b 0.2 -s 0.2
output.setup=on -dir ./results/
"""

CONF_MF = """ratings=./dataset/FilmTrust/trainset.txt
ratings.setup=-columns 0 1 2
model.name=%(name)s
evaluation.setup=-testSet ./dataset/FilmTrust/testset.txt
item.ranking=off -topN 10
num.factors=%(d)d
num.max.epoch=3
batch_size=1024
learnRate=-init %(lr)s -max 1
reg.lambda=-u 0.01 -i 0.02 -b 0.03 -s 0.1
output.setup=on -dir ./results/
"""
MF_RUNS = (('BasicMF', 20, '0.03', 11), ('PMF', 10, '0.02', 12), ('SVD', 20, '0.005', 13))   # name, d, lr, seed


def _stub_modules():
    sys.modules.setdefault('tensorflow', types.ModuleType('tensorflow'))
    mkl = types.ModuleType('mkl')
    mkl.set_num_threads = lambda n: None
    mkl.get_max_threads = lambda: 1
    sys.modules.setdefault('mkl', mkl)


def _state_to_array(state):
    """random.getstate() -> uint32[625] (624 words + index)."""
    version, internal, gauss = state
    assert version == 3 and gauss is None
    return np.array(internal, dtype=np.uint32)


def _enter_workdir():
    assert os.path.isdir(REF), 'reference checkout not mounted'
    _stub_modules()
    sys.path.insert(0, REF)
    work = tempfile.mkdtemp(prefix='qrec_golden_')
    os.chdir(work)
    os.symlink(os.path.join(REF, 'dataset'), 'dataset')
    os.makedirs('log', exist_ok=True)
    os.makedirs('results', exist_ok=True)


def gen_bpr():
    with open('BPR_ft.conf', 'w') as f:
        f.write(CONF_BPR)
    with open('LGCN_ft.conf', 'w') as f:
        f.write(CONF_LGCN)

    from util.config import ModelConf
    from QRec import QRec
    from model.ranking.BPR import BPR

    # ------------------------------------------------------------------ BPR numpy path
    random.seed(0)
    np.random.seed(0)
    conf = ModelConf('BPR_ft.conf')
    with contextlib.redirect_stdout(io.StringIO()):
        q = QRec(conf)
    train, test = q.trainingData, q.testData
    state_after_split = _state_to_array(random.getstate())

    model = BPR(conf, train, test)
    # training list exactly as the model holds it at construction (data/rating.py:27)
    train_users = np.array([e[0] for e in model.data.trainingData])
    train_items = np.array([e[1] for e in model.data.trainingData])
    train_rating = np.array([e[2] for e in model.data.trainingData], dtype=np.float64)
    test_users = np.array([e[0] for e in model.data.testData])
    test_items = np.array([e[1] for e in model.data.testData])
    test_rating = np.array([e[2] for e in model.data.testData], dtype=np.float64)
    user_names = np.array([model.data.id2user[k] for k in range(len(model.data.user))])
    item_names = np.array([model.data.id2item[k] for k in range(len(model.data.item))])

    rec = dict(triples=[], cur=[], P=[], Q=[], loss=[], lrate=[], states=[])
    orig_opt = BPR.optimization
    orig_conv = BPR.isConverged

    def spy_opt(self, u, i, j):
        rec['cur'].append((u, i, j))
        return orig_opt(self, u, i, j)

    def spy_conv(self, epoch):
        rec['triples'].append(np.array(rec['cur'], dtype=np.int32))
        rec['cur'] = []
        rec['P'].append(self.P.copy())
        rec['Q'].append(self.Q.copy())
        rec['loss'].append(float(self.loss))
        lr_before = self.lRate
        r = orig_conv(self, epoch)
        rec['lrate'].append((lr_before, self.lRate))
        rec['states'].append(_state_to_array(random.getstate()))
        return r

    BPR.optimization = spy_opt
    BPR.isConverged = spy_conv
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            model.readConfiguration()
            model.initializing_log()
            state_before_init = _state_to_array(random.getstate())
            model.initModel()
            P0, Q0 = model.P.copy(), model.Q.copy()
            model.trainModel()
            model.evalRanking()
    finally:
        BPR.optimization = orig_opt
        BPR.isConverged = orig_conv
    measure = [m.strip() for m in model.measure]
    print('BPR FilmTrust: train', model.data.trainingSize(), 'losses', rec['loss'], 'measure', measure)

    # check the regenerable init: legacy numpy stream is stable across versions
    np.random.seed(0)
    P0r = np.random.rand(len(model.data.user), 64) / 3
    Q0r = np.random.rand(len(model.data.item), 64) / 3
    assert np.array_equal(P0r, P0) and np.array_equal(Q0r, Q0)
    assert np.array_equal(state_before_init, state_after_split)

    # top-10 recommendation lists (ids) for the first 64 test users, for the eval parity test
    rec_lines = model.recOutput[1:65]

    np.savez_compressed(
        os.path.join(OUT, 'bpr_filmtrust_seed0.npz'),
        user_names=user_names, item_names=item_names,
        train_users=train_users, train_items=train_items, train_rating=train_rating,
        test_users=test_users, test_items=test_items, test_rating=test_rating,
        mt_state_after_split=state_after_split,
        mt_state_after_epoch=np.stack(rec['states']),
        triples_epoch=np.stack(rec['triples']),            # [3, n, 3] int32 (u,i,j) in reference order
        P_epoch1=rec['P'][0], Q_epoch1=rec['Q'][0],        # float64
        P_epoch3=rec['P'][2].astype(np.float32), Q_epoch3=rec['Q'][2].astype(np.float32),
        loss=np.array(rec['loss']), lrate=np.array(rec['lrate']),
        measure=np.array(measure), rec_lines=np.array(rec_lines),
        conf=np.array(CONF_BPR),
    )

    # ------------------------------------------------------------------ samplers (TF-style path)
    from base.deepRecommender import DeepRecommender
    from base.graphRecommender import GraphRecommender
    random.seed(1234)
    np.random.seed(1234)
    lconf = ModelConf('LGCN_ft.conf')
    with contextlib.redirect_stdout(io.StringIO()):
        q2 = QRec(lconf)
    g = GraphRecommender(lconf, q2.trainingData, q2.testData)
    with contextlib.redirect_stdout(io.StringIO()):
        g.readConfiguration()
    g_train_users = np.array([e[0] for e in g.data.trainingData])
    g_train_items = np.array([e[1] for e in g.data.trainingData])
    g_user_names = np.array([g.data.id2user[k] for k in range(len(g.data.user))])
    g_item_names = np.array([g.data.id2item[k] for k in range(len(g.data.item))])
    st_pair = _state_to_array(random.getstate())
    pair_batches = [np.array(b, dtype=np.int32) for b in DeepRecommender.next_batch_pairwise(g)]
    st_after_pair = _state_to_array(random.getstate())
    # the list was shuffled in place by the generator; record the new order as (u,i) ids
    shuffled_u = np.array([g.data.user[e[0]] for e in g.data.trainingData], dtype=np.int32)
    shuffled_i = np.array([g.data.item[e[1]] for e in g.data.trainingData], dtype=np.int32)
    st_point = _state_to_array(random.getstate())
    point_batches = []
    for n, b in enumerate(DeepRecommender.next_batch_pointwise(g)):
        point_batches.append(np.array(b, dtype=np.int32))
        if n == 1:
            break
    st_after_point = _state_to_array(random.getstate())

    adj = g.create_joint_sparse_adjaceny().tocsr()
    adj.sort_indices()
    rmat = g.create_sparse_rating_matrix().tocsr()
    rmat.sort_indices()
    np.savez_compressed(
        os.path.join(OUT, 'sampler_graph_filmtrust_seed1234.npz'),
        user_names=g_user_names, item_names=g_item_names,
        train_users=g_train_users, train_items=g_train_items,
        mt_state_before_pairwise=st_pair, mt_state_after_pairwise=st_after_pair,
        pair_first=pair_batches[0], pair_last=pair_batches[-1],
        pair_all_j=np.concatenate([b[2] for b in pair_batches]),
        pair_num_batches=np.array(len(pair_batches)),
        shuffled_u=shuffled_u, shuffled_i=shuffled_i,
        mt_state_before_pointwise=st_point, mt_state_after_pointwise=st_after_point,
        point_b0=point_batches[0], point_b1=point_batches[1],
        adj_indptr=adj.indptr.astype(np.int64), adj_indices=adj.indices.astype(np.int32),
        adj_data=adj.data.astype(np.float32), adj_shape=np.array(adj.shape),
        rmat_indptr=rmat.indptr.astype(np.int64), rmat_indices=rmat.indices.astype(np.int32),
        rmat_data=rmat.data.astype(np.float32), rmat_shape=np.array(rmat.shape),
        conf=np.array(CONF_LGCN),
    )
    print('samplers: pairwise batches', len(pair_batches), 'last', pair_batches[-1].shape,
          'pointwise b0', point_batches[0].shape, 'adj nnz', adj.nnz, 'rmat nnz', rmat.nnz)


def gen_mf():
    """One fixture per rating-prediction MF model: the order the entries were visited in each epoch
    (a permutation of the initial training list), the tables after every epoch, the epoch losses,
    the learning-rate schedule, the MT19937 state after every epoch's shuffle and the final
    MAE / RMSE lines."""
    import importlib
    from util.config import ModelConf
    from QRec import QRec
    for name, d, lr, seed in MF_RUNS:
        cname = '%s_ft.conf' % name
        with open(cname, 'w') as f:
            f.write(CONF_MF % dict(name=name, d=d, lr=lr))
        random.seed(seed)
        np.random.seed(seed)
        conf = ModelConf(cname)
        with contextlib.redirect_stdout(io.StringIO()):
            q = QRec(conf)
        cls = getattr(importlib.import_module('model.rating.' + name), name)
        model = cls(conf, q.trainingData, q.testData)
        first = list(model.data.trainingData)
        where = {id(e): k for k, e in enumerate(first)}
        rec = dict(order=[], P=[], Q=[], Bu=[], Bi=[], loss=[], lrate=[], states=[], rmse=[])
        orig_conv = cls.isConverged

        def spy_conv(self, epoch):
            rec['order'].append(np.array([where[id(e)] for e in self.data.trainingData], dtype=np.int32))
            rec['P'].append(self.P.copy())
            rec['Q'].append(self.Q.copy())
            if hasattr(self, 'Bu'):
                rec['Bu'].append(self.Bu.copy())
                rec['Bi'].append(self.Bi.copy())
            rec['loss'].append(float(self.loss))
            lr_before = self.lRate
            r = orig_conv(self, epoch)
            rec['rmse'].append([m.strip() for m in self.measure])
            rec['lrate'].append((lr_before, self.lRate))
            rec['states'].append(_state_to_array(random.getstate()))
            return r

        cls.isConverged = spy_conv
        try:
            with contextlib.redirect_stdout(io.StringIO()):
                model.readConfiguration()
                model.initializing_log()
                state_before = _state_to_array(random.getstate())
                model.initModel()
                init = dict(P0=model.P.copy(), Q0=model.Q.copy())
                if hasattr(model, 'Bu'):
                    init.update(Bu0=model.Bu.copy(), Bi0=model.Bi.copy())
                model.trainModel()
                model.evalRatings()
        finally:
            cls.isConverged = orig_conv
        measure = [m.strip() for m in model.measure]
        print(name, 'FilmTrust: train', model.data.trainingSize(), 'losses', rec['loss'], 'measure', measure)
        extra = {}
        if rec['Bu']:
            extra = dict(Bu_last=rec['Bu'][-1], Bi_last=rec['Bi'][-1])
        np.savez_compressed(
            os.path.join(OUT, 'mf_%s_filmtrust.npz' % name.lower()),
            user_names=np.array([model.data.id2user[k] for k in range(len(model.data.user))]),
            item_names=np.array([model.data.id2item[k] for k in range(len(model.data.item))]),
            train_users=np.array([e[0] for e in first]), train_items=np.array([e[1] for e in first]),
            train_rating=np.array([e[2] for e in first], dtype=np.float64),
            test_users=np.array([e[0] for e in model.data.testData]),
            test_items=np.array([e[1] for e in model.data.testData]),
            test_rating=np.array([e[2] for e in model.data.testData], dtype=np.float64),
            test_pred=np.array([e[3] for e in model.data.testData], dtype=np.float64),
            global_mean=np.array(model.data.globalMean),
            mt_state_before=state_before, mt_state_after_epoch=np.stack(rec['states']),
            order_epoch=np.stack(rec['order']),               # [E, n] indices into the initial list
            # tables after the first epoch (fp32 copy, loose checks) and after the last (float64, exact)
            P_epoch1=rec['P'][0].astype(np.float32), Q_epoch1=rec['Q'][0].astype(np.float32),
            P_last=rec['P'][-1], Q_last=rec['Q'][-1],
            loss=np.array(rec['loss']), lrate=np.array(rec['lrate']),
            epoch_measure=np.array(rec['rmse']), measure=np.array(measure),
            seed=np.array(seed), conf=np.array(CONF_MF % dict(name=name, d=d, lr=lr)),
            **init, **extra)


CONF_SBPR = """ratings=./dataset/FilmTrust/ratings.txt
social=./dataset/FilmTrust/trust.txt
ratings.setup=-columns 0 1 2
social.setup=-columns 0 1
model.name=SBPR
evaluation.setup=-testSet ./dataset/FilmTrust/testset.txt -b 1.0 -tf
item.ranking=on -topN 10
num.factors=16
num.max.epoch=2
batch_size=512
learnRate=-init 0.005 -max 0.1
reg.lambda=-u 0.01 -i 0.01 -b 0.01 -s 0.2
output.setup=off -dir ./results/
"""


def gen_sbpr():
    """model/ranking/SBPR.py:12-29 (PositiveSet / FPSet from FilmTrust's trust network) and :69-101 (next_batch): the
    social-feedback sets and the first minibatches of the UNMODIFIED reference class on the training split recorded in
    bpr_filmtrust_seed0.npz.  Only dicts are involved (no sets), so the stream does not depend on the hash seed."""
    from util.config import ModelConf
    from util.io import FileIO
    from model.ranking.SBPR import SBPR
    g = np.load(os.path.join(OUT, 'bpr_filmtrust_seed0.npz'), allow_pickle=True)
    train = [[u, i, float(r)] for u, i, r in zip(g['train_users'].tolist(), g['train_items'].tolist(), g['train_rating'].tolist())]
    with open('SBPR_ft.conf', 'w') as f:
        f.write(CONF_SBPR)
    conf = ModelConf('SBPR_ft.conf')
    relation = FileIO.loadRelationship(conf, conf['social'])
    np.random.seed(0)
    random.seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        m = SBPR(conf, [list(r) for r in train], [], [list(r) for r in relation])
        m.readConfiguration()
        m.initModel()
    m.batch_size = 512
    users = list(m.data.user.keys())
    fp_sizes = np.array([len(m.FPSet[u]) if u in m.FPSet else 0 for u in users], dtype=np.int64)
    fp_sums = np.array([sum(m.FPSet[u].values()) if u in m.FPSet else 0 for u in users], dtype=np.int64)
    fp_first = np.array([(next(iter(m.FPSet[u])) if (u in m.FPSet and len(m.FPSet[u])) else '') for u in users])
    random.seed(77)
    batches = []
    for n, b in enumerate(m.next_batch()):
        batches.append(np.array(b, dtype=np.int64))                  # [5, batch]: u, i, k, j, S_uk
        if n == 7:
            break
    state = _state_to_array(random.getstate())
    np.savez_compressed(
        os.path.join(OUT, 'sbpr_filmtrust_seed77.npz'),
        relation_from=np.array([r[0] for r in relation]), relation_to=np.array([r[1] for r in relation]),
        relation_w=np.array([float(r[2]) for r in relation]),
        fp_sizes=fp_sizes, fp_sums=fp_sums, fp_first=fp_first,
        batches=np.stack(batches), mt_state_after_8_batches=state, conf=np.array(CONF_SBPR))
    print('sbpr: %d relations, %d users with social feedback, 8 batches of 512' % (len(relation), int((fp_sizes > 0).sum())))


def _quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **kw)


def gen_differential():
    """Inputs and outputs of the reference's host-side surface for tests/test_differential_reference.py, plus
    FilmTrust's ratings file itself (tests/golden/filmtrust_ratings.txt.xz, read by the loader tests).  The tests
    draw the same seeded random inputs again, so only the reference's outputs are stored:
      * util/config.py OptionConf / ModelConf   on random option strings and on every config/*.conf
      * util/measure.py rankingMeasure / ratingMeasure, util/qmath.py find_k_largest / sigmoid
      * data/rating.py Rating under four evaluation setups, util/dataSplit.py dataSplit / crossValidation
      * util/io.py loadDataSet on FilmTrust (digests: the full lists are 35K records each) and the id space of
        Rating over it
      * base/iterativeRecommender.py isConverged + base/recommender.py evalRanking, and
        base/deepRecommender.py next_batch_pairwise / next_batch_pointwise on random interaction lists (digests)"""
    import importlib
    import lzma
    from oracle import golden_json
    M = {n: importlib.import_module(n) for n in ('util.config', 'util.measure', 'util.qmath', 'util.io', 'util.dataSplit',
                                                 'data.rating', 'base.iterativeRecommender', 'base.deepRecommender')}
    RConf = M['util.config'].ModelConf

    def conf_of(config):
        c = RConf.__new__(RConf)
        c.config = dict(config)
        return c
    rec = {}

    rng = random.Random(0)
    vocab = ['on', 'off', '-a', '-b', '--c', '-topN', '-1', '-12', '-0.5', '5', '10,20', 'x', '0.1', '-tf', '', '-n_layer', '2']
    rows = []
    for _ in range(3000):
        s = ' '.join(rng.choice(vocab) for _ in range(rng.randint(1, 8)))
        if rng.random() < 0.2:
            s = ' ' + s + ' '
        o = M['util.config'].OptionConf(s)
        rows.append((o.options, o.isMainOn(), o.line))
    rec['option_conf'] = rows

    cdir = os.path.join(REF, 'config')
    rec['model_conf'] = [(name, open(os.path.join(cdir, name)).read(), RConf(os.path.join(cdir, name)).config)
                         for name in sorted(os.listdir(cdir))]
    with open('bad.conf', 'w') as f:
        f.write('a=1\nnot a pair\nb=2=3\n\nc=x y\n')
    rec['model_conf_bad'] = RConf('bad.conf').config

    R = M['util.measure'].Measure
    rng = random.Random(1)
    items = ['i%d' % k for k in range(60)]
    cases = []
    for _ in range(200):
        users = ['u%d' % k for k in range(rng.randint(1, 12))]
        origin = {u: {it: 1.0 for it in rng.sample(items, rng.randint(1, 15))} for u in users}
        res = {u: [(it, rng.random()) for it in rng.sample(items, 20)] for u in users}
        tops = sorted(rng.sample([1, 3, 5, 10, 20], rng.randint(1, 3)))
        cases.append(R.rankingMeasure(origin, res, tops))
    rows = [['u', 'i', rng.random() * 5, rng.random() * 5] for _ in range(50)]
    rec['ranking_measure'] = cases
    rec['rating_measure'] = (R.ratingMeasure(rows), R.ratingMeasure([]))

    F = M['util.qmath'].find_k_largest
    rng = np.random.default_rng(2)
    trials = []
    for trial in range(120):
        n, K = int(rng.integers(3, 300)), int(rng.integers(1, 15))
        s = rng.standard_normal(n).round(1 if trial % 3 == 0 else 7)
        s[rng.integers(0, n, n // 5)] = 0.0                       # rated items are overwritten with 0
        ids, vals = F(K, s.copy())
        trials.append((list(ids), list(vals)))
    rec['find_k_largest'] = trials
    rec['sigmoid_0.3'] = M['util.qmath'].sigmoid(0.3)

    rng = random.Random(3)
    runs = []
    for ev in ('-ap 0.2', '-ap 0.2 -b 1', '-cold 2', '-val 0.25'):
        train = [['u%d' % rng.randint(0, 30), 'i%d' % rng.randint(0, 40), float(rng.randint(1, 5))] for _ in range(400)]
        test = [['u%d' % rng.randint(0, 35), 'i%d' % rng.randint(0, 45), float(rng.randint(1, 5))] for _ in range(120)]
        random.seed(11)
        d = M['data.rating'].Rating(conf_of({'ratings': 'x', 'evaluation.setup': ev}), [r[:] for r in train], [r[:] for r in test])
        u0 = next(iter(d.user))
        out = {a: getattr(d, a) for a in ('user', 'item', 'id2user', 'id2item', 'userMeans', 'itemMeans', 'globalMean',
                                          'rScale', 'trainingData', 'testData')}
        out.update(trainSet_u=dict(d.trainSet_u), testSet_u=dict(d.testSet_u), trainSet_i=dict(d.trainSet_i),
                   testSet_i=dict(d.testSet_i), trainingSize=d.trainingSize(), testSize=d.testSize(), u0=u0,
                   userRated=d.userRated(u0), row=d.row(u0))
        runs.append(out)
    rec['rating'] = runs

    RS = M['util.dataSplit'].DataSplit
    rng = random.Random(5)
    data = [['u%d' % rng.randint(0, 9), 'i%d' % rng.randint(0, 9), float(rng.randint(0, 1))] for _ in range(300)]
    split = []
    for ratio, binar in ((0.2, False), (0.2, True), (1.5, False), (0.0, True)):
        random.seed(7)
        split.append((RS.dataSplit(data, test_ratio=ratio, binarized=binar), random.getstate()))
    cv = [list(RS.crossValidation(data, k, binarized=binar)) for k, binar in ((5, False), (3, True), (1, False), (11, False))]
    rec['data_split'] = (split, cv)

    path = os.path.join(REF, 'dataset', 'FilmTrust', 'ratings.txt')
    loads = []
    for setup, kw in (('-columns 0 1 2', {}), ('-columns 0 1 2', {'binarized': True, 'threshold': 3.0}),
                      ('-columns 1 0', {}), ('-columns 0 1 2 -header', {'bTest': True})):
        b = _quiet(M['util.io'].FileIO.loadDataSet, conf_of({'ratings.setup': setup}), path, **kw)
        loads.append((len(b), b[:5], golden_json.digest(b)))
    rec['load_filmtrust'] = loads
    rc = conf_of({'ratings.setup': '-columns 0 1 2', 'evaluation.setup': '-ap 0.2 -b 1'})
    recs = _quiet(M['util.io'].FileIO.loadDataSet, rc, path, binarized=True, threshold=1.0)
    d = M['data.rating'].Rating(rc, recs, [])
    rec['table_filmtrust'] = dict(n=len(recs), user_names=[d.id2user[k] for k in range(len(d.user))],
                                  item_names=[d.id2item[k] for k in range(len(d.item))],
                                  u_digest=golden_json.digest([d.user[r[0]] for r in recs]),
                                  i_digest=golden_json.digest([d.item[r[1]] for r in recs]))

    rng = random.Random(9)
    conf_text = ('ratings=x\nratings.setup=-columns 0 1 2\nmodel.name=BPR\nevaluation.setup=-ap 0.2 -b 1\n'
                 'item.ranking=on -topN 5,10\nnum.factors=8\nnum.max.epoch=3\nlearnRate=-init 0.01 -max 0.0105\n'
                 'reg.lambda=-u 0.001 -i 0.001 -b 0.2 -s 0.2\noutput.setup=on -dir ./results/\n')
    train = [['u%d' % rng.randint(0, 40), 'i%d' % rng.randint(0, 60), 1.0] for _ in range(900)]
    test = [['u%d' % rng.randint(0, 45), 'i%d' % rng.randint(0, 60), 1.0] for _ in range(200)]
    with open('eval.conf', 'w') as f:
        f.write(conf_text)
    m = M['base.iterativeRecommender'].IterativeRecommender(RConf('eval.conf'), [r[:] for r in train], [r[:] for r in test])
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
    rec['eval_ranking'] = (conv, m.recOutput, m.measure, random.getstate(), [r[:] for r in m.data.trainingData])

    batches = {}
    for seed in (0, 7, 2024):
        rng = random.Random(seed)
        conf_text = ('ratings=x\nratings.setup=-columns 0 1 2\nmodel.name=LightGCN\nevaluation.setup=-ap 0.2\n'
                     'item.ranking=on -topN 10\nnum.factors=8\nnum.max.epoch=1\nbatch_size=128\n'
                     'learnRate=-init 0.01 -max 1\nreg.lambda=-u 0.001 -i 0.001 -b 0.2 -s 0.2\noutput.setup=off -dir ./results/\n')
        train = [['u%d' % rng.randint(0, 50), 'i%d' % rng.randint(0, 80), float(rng.randint(1, 5))] for _ in range(1000)]
        with open('batch.conf', 'w') as f:
            f.write(conf_text)
        m = M['base.deepRecommender'].DeepRecommender(RConf('batch.conf'), [r[:] for r in train], [])
        _quiet(m.readConfiguration)
        random.seed(seed)
        pair = [tuple(np.asarray(x).tolist() for x in batch) for batch in m.next_batch_pairwise()]
        point = [tuple(np.asarray(x).tolist() for x in batch) for batch in m.next_batch_pointwise()]
        batches[seed] = (len(pair), golden_json.digest(pair), golden_json.digest(point),
                         golden_json.digest([r[:] for r in m.data.trainingData]), random.getstate())
    rec['minibatch'] = batches

    golden_json.save(os.path.join(OUT, 'differential_reference.json.xz'), rec)
    with open(path, 'rb') as f, lzma.open(os.path.join(OUT, 'filmtrust_ratings.txt.xz'), 'wb', preset=9) as g:
        g.write(f.read())
    print('differential: %d option strings, %d config files, %d ranking cases' % (
        len(rec['option_conf']), len(rec['model_conf']), len(rec['ranking_measure'])))


TBPR_ROWS = np.arange(0, 310, 5)          # every 5th row of both tables is stored whole (P has 310 rows)


def gen_social():
    """model/ranking/TBPR.py (whole numpy run) and model/ranking/SBPR.py:12-29,69-101 (item sets + sampler) of the
    UNMODIFIED reference classes on the inputs tests/test_tbpr_cpu.py and tests/test_sbpr_cpu.py build (a FilmTrust
    training prefix + a synthetic trust network).  TBPR iterates a Python set of item names (TBPR.py:122), so its
    stream depends on the string-hash seed: main() runs every section with PYTHONHASHSEED=0 and the TBPR test replays
    the drop-in under the same seed."""
    import importlib
    from oracle import golden_json
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    import test_tbpr_cpu
    import test_sbpr_cpu
    g = np.load(os.path.join(OUT, 'bpr_filmtrust_seed0.npz'))
    RConf = importlib.import_module('util.config').ModelConf

    R = importlib.import_module('model.ranking.TBPR').TBPR
    train, test, rel = test_tbpr_cpu._data(g)
    with open('tbpr.conf', 'w') as f:
        f.write(test_tbpr_cpu.CONF)
    random.seed(11); np.random.seed(11)
    ref = R(RConf('tbpr.conf'), [list(r) for r in train], [list(r) for r in test], [list(r) for r in rel])
    losses = []
    orig = R.isConverged
    R.isConverged = lambda self, epoch: (losses.append((self.loss, self.lRate)), orig(self, epoch))[1]
    try:
        measure = _quiet(ref.execute)
    finally:
        R.isConverged = orig
    np.savez_compressed(os.path.join(OUT, 'tbpr_reference_hashseed0.npz'),
                        theta=np.array(ref.theta), t_s=np.array(ref.t_s), t_w=np.array(ref.t_w),
                        loss=np.array([l[0] for l in losses]), lrate=np.array([l[1] for l in losses]),
                        rows=TBPR_ROWS, P_rows=ref.P[TBPR_ROWS], Q_rows=ref.Q[TBPR_ROWS], P_abs_row_sums=np.abs(ref.P).sum(1),
                        Q_abs_row_sums=np.abs(ref.Q).sum(1), measure=np.array([x.strip() for x in measure]))

    R = importlib.import_module('model.ranking.SBPR').SBPR
    train, test, rel = test_tbpr_cpu._data(g, 3000)
    with open('sbpr.conf', 'w') as f:
        f.write(test_sbpr_cpu.CONF)
    np.random.seed(1)
    ref = R(RConf('sbpr.conf'), [list(r) for r in train], [list(r) for r in test], [list(r) for r in rel])
    _quiet(ref.readConfiguration)
    _quiet(ref.initModel)
    ref.batch_size = 700
    random.seed(77)
    batches = [tuple(list(x) for x in b) for b in ref.next_batch()]
    golden_json.save(os.path.join(OUT, 'sbpr_reference_sampler.json.xz'), dict(
        positive={u: dict(v) for u, v in ref.PositiveSet.items() if v},
        fp={u: dict(v) for u, v in ref.FPSet.items()},
        batches=batches, state=random.getstate()))
    print('social: TBPR losses %s, SBPR %d batches' % ([l[0] for l in losses], len(batches)))


def main():
    if os.environ.get('PYTHONHASHSEED') != '0':      # gen_social's TBPR stream depends on the string-hash seed
        os.execve(sys.executable, [sys.executable] + sys.argv, dict(os.environ, PYTHONHASHSEED='0'))
    what = set(sys.argv[1:]) or {'bpr', 'mf', 'sbpr', 'differential', 'social'}
    sys.path.insert(0, REPO)
    _enter_workdir()
    if 'bpr' in what:
        gen_bpr()
    if 'mf' in what:
        gen_mf()
    if 'sbpr' in what:
        gen_sbpr()
    if 'differential' in what:
        gen_differential()
    if 'social' in what:
        gen_social()


if __name__ == '__main__':
    main()
