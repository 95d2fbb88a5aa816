"""TBPR drop-in (f-4 sibling model: model/ranking/TBPR.py mirror) on the CPU: the device is stubbed and the K1
kernels are replaced by the pinned oracle, so what is checked is the HOST side that is specific to TBPR -- tie
strengths, the per-epoch strong / weak / joint item sets, the preference chains and their draw order from Python's
`random`, the per-user regulariser quirk of the loss, the learning-rate bookkeeping.

(1) differential against the UNMODIFIED reference class, recorded under a fixed string-hash seed (the joint set is
    iterated in Python set order, which depends on it) and replayed under the same seed;
(2) self-consistency that also runs on the GPU box's CPU suite."""
import contextlib
import io
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from qrec_b200.util.config import ModelConf
from test_bpr_model_cpu import _stub_engine

CONF = '''ratings=x
social=x
ratings.setup=-columns 0 1 2
social.setup=-columns 0 1
model.name=TBPR
evaluation.setup=-testSet x -b 1.0
item.ranking=on -topN 10
num.factors=16
num.max.epoch=3
learnRate=-init 0.01 -max 0.1
reg.lambda=-u 0.001 -i 0.001 -b 0.01 -s 0.2
TBPR=-regT 0.01
output.setup=off -dir ./results/
'''


def _data(golden_bpr, n_train=6000):
    g = golden_bpr
    train = [[u, i, 1.0] for u, i in zip(g['train_users'][:n_train].tolist(), g['train_items'][:n_train].tolist())]
    users = sorted({r[0] for r in train}, key=lambda s: int(s))
    test = [[u, i, 1.0] for u, i in zip(g['test_users'].tolist(), g['test_items'].tolist()) if u in set(users)][:400]
    # a synthetic trust network over the training users (FilmTrust's trust.txt does not travel to the GPU box):
    # a ring of cliques gives shared followees (Jaccard > 0, strong ties) next to sparse random edges (weak ties)
    rng = random.Random(5)
    rel = []
    for k, u in enumerate(users):
        for step in (1, 2, 3):
            rel.append([u, users[(k + step) % len(users)], 1])
        for _ in range(2):
            rel.append([u, rng.choice(users), 1])
    rel.append(['stranger', users[0], 1]); rel.append([users[1], 'stranger2', 1])     # cleaned by SocialRecommender
    return train, test, rel


def _run(cls, train, test, rel, conf_text):
    random.seed(11); np.random.seed(11)
    model = cls(ModelConf.from_string(conf_text) if hasattr(ModelConf, 'from_string') else conf_text, train, test, [list(r) for r in rel])
    losses = []
    orig = cls.isConverged

    def spy(self, epoch):
        losses.append((self.loss, self.lRate))
        return orig(self, epoch)
    cls.isConverged = spy
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            measure = model.execute()
    finally:
        cls.isConverged = orig
    return model, losses, measure


def test_tbpr_host_logic_self_consistency(golden_bpr, monkeypatch, tmp_path):
    from qrec_b200.model.ranking.TBPR import TBPR
    calls = []
    _stub_engine(monkeypatch, calls)
    monkeypatch.chdir(tmp_path)
    train, test, rel = _data(golden_bpr)
    m, losses, measure = _run(TBPR, train, test, rel, CONF)
    assert 'stranger' not in m.social.followees and all('stranger2' not in v for v in m.social.followees.values())
    assert len(m.strongTies) > 0 and len(m.weakTies) > 0 and 0.0 <= m.theta <= 1.0
    # every user of positiveSet is one ordered launch per epoch (more when a chain repeats an item: those single
    # steps are applied apart); chains have 2..5 members -> 1..4 steps per positive
    n_pos = sum(len(v) for v in m.positiveSet.values())
    steps = [c[1] for c in calls if c[0] == 'ordered']
    assert 3 * len(m.positiveSet) <= len(steps) <= 4 * len(m.positiveSet) and 0.99 * 3 * n_pos <= sum(steps) <= 3 * 4 * n_pos
    # joint / strong / weak are disjoint per user and never contain the user's own positives
    for u in m.positiveSet:
        j, s, w = set(m.jointSet[u]), set(m.strongSet[u]), set(m.weakSet[u])
        assert not (j & s) and not (j & w) and not (s & w) and not ((j | s | w) & set(m.positiveSet[u]))
    assert len(losses) == 3 and losses[0][0] > losses[-1][0] > 0           # the loss falls
    assert losses[0][1] == 0.01 and losses[2][1] == pytest.approx(0.01 * 1.05)     # epoch 1 never changes lr; epoch 2 raised it
    assert measure[0].startswith('Top 10')
    # the native epoch sampler (qrec_sample_tbpr_epoch) and the same loop in Python: same steps, same generator state
    random.seed(99)
    nat = m._sample_epoch()
    nat_state = random.getstate()
    random.seed(99)
    py = m._sample_epoch_python()
    assert random.getstate() == nat_state
    assert all(np.array_equal(x, y) for x, y in zip(nat, py)) and nat[0].dtype == np.int32 and len(nat[3]) == len(m.positiveSet)
    # same seeds -> same run (the draw order from `random` is deterministic inside one process)
    m2, losses2, _ = _run(TBPR, train, test, rel, CONF)
    assert losses2 == losses and np.array_equal(m.P, m2.P) and np.array_equal(m.Q, m2.Q)
    # fast mode goes through the user-major kernel entry with a CSR over ALL users
    seen = {}

    def usermajor(P, Q, rowptr, i, j, lr, reg_u, reg_i, loss):
        seen['rowptr'] = rowptr.numpy().copy(); seen['n'] = len(i)
        loss += 1.0
    from qrec_b200 import engine as E
    monkeypatch.setattr(E, 'bpr_sgd_usermajor', usermajor)
    _run(TBPR, train, test, rel, CONF.replace('num.max.epoch=3', 'num.max.epoch=1') + 'engine=-mode fast\n')
    assert len(seen['rowptr']) == m.num_users + 1 and seen['rowptr'][-1] == seen['n'] and np.all(np.diff(seen['rowptr']) >= 0)


def _record_dropin(path):
    """The drop-in's side of test_tbpr_equals_unmodified_reference_class, run in a child interpreter."""
    from qrec_b200.model.ranking.TBPR import TBPR
    train, test, rel = _data(np.load(os.path.join(GOLDEN, 'bpr_filmtrust_seed0.npz')))
    with pytest.MonkeyPatch.context() as mp:
        _stub_engine(mp, [])
        m, losses, measure = _run(TBPR, train, test, rel, CONF)
    np.savez(path, theta=m.theta, t_s=m.t_s, t_w=m.t_w, loss=[l[0] for l in losses], lrate=[l[1] for l in losses],
             P=m.P, Q=m.Q, measure=[x.strip() for x in measure])


def test_tbpr_equals_unmodified_reference_class(tmp_path):
    """Same seeds: epoch losses, learning rates, theta, the final tables and the ranking measures of the drop-in equal
    those of the reference's TBPR (numpy path), recorded on the same inputs in tests/golden/tbpr_reference_hashseed0.npz
    -- K1 being the oracle here.  The joint item set is iterated in Python set order, which follows the string-hash
    seed, so the drop-in runs in a child interpreter under PYTHONHASHSEED=0, the seed the record was made under."""
    out = tmp_path / 'dropin.npz'
    code = 'import sys; sys.path[:0] = sys.argv[1:3]; import test_tbpr_cpu; test_tbpr_cpu._record_dropin(sys.argv[3])'
    run = subprocess.run([sys.executable, '-c', code, ROOT, os.path.dirname(__file__), str(out)], cwd=tmp_path,
                         env=dict(os.environ, PYTHONHASHSEED='0'), capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stderr[-3000:]
    m, ref = np.load(out), np.load(os.path.join(GOLDEN, 'tbpr_reference_hashseed0.npz'))
    assert m['theta'] == ref['theta'] and m['t_s'] == ref['t_s'] and m['t_w'] == ref['t_w']
    assert m['lrate'].tolist() == ref['lrate'].tolist()
    np.testing.assert_allclose(m['loss'], ref['loss'], rtol=1e-12)
    # the record holds every 5th row of each table whole and the |.|-sum of every row
    for name in ('P', 'Q'):
        np.testing.assert_allclose(m[name][ref['rows']], ref[name + '_rows'], rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(np.abs(m[name]).sum(1), ref[name + '_abs_row_sums'], rtol=1e-12)
    assert m['measure'].tolist() == ref['measure'].tolist()
