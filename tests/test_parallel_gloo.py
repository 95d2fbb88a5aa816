"""N>1 host logic on CPU: world_size-2 gloo process group (torch.multiprocessing spawn)."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from qrec_b200 import parallel


def test_user_range_partitions_exactly():
    for world in (1, 2, 3, 8):
        for n in (0, 1, 7, 8, 1000, 1_000_003):
            spans = [parallel.user_range(r, world, n) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
    assert parallel.sync_points(10, 4) == [0, 2, 5, 7, 10] and parallel.sync_points(5, 0) == [0, 5]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        torch.manual_seed(0)
        Q0 = torch.randn(50, 8)
        Q = Q0.clone()
        sync = parallel.ReplicatedTableSync(Q)
        # sharding: every triple lands on exactly one rank, with local user ids
        g = torch.Generator().manual_seed(1)
        u = torch.randint(0, 11, (200,), generator=g, dtype=torch.int32)
        i = torch.randint(0, 50, (200,), generator=g, dtype=torch.int32)
        j = torch.randint(0, 50, (200,), generator=g, dtype=torch.int32)
        lu, li, lj = parallel.shard_triples_by_user(u, i, j, rank, world, 11)
        lo, hi = parallel.user_range(rank, world, 11)
        assert int(lu.min()) >= 0 and int(lu.max()) < hi - lo
        cnt = torch.tensor([lu.numel()])
        dist.all_reduce(cnt)
        assert int(cnt) == 200
        # two rounds of "local training" (rank-specific scatter-adds) + delta sync
        expect = Q0.clone()
        for rnd in range(2):
            for r in range(world):
                gg = torch.Generator().manual_seed(100 * rnd + r)
                rows = torch.randint(0, 50, (30,), generator=gg)
                upd = torch.randn(30, 8, generator=gg)
                expect.index_add_(0, rows, upd)
                if r == rank:
                    Q.index_add_(0, rows, upd)
            sync.sync()
            assert torch.allclose(Q, expect, atol=1e-5), 'rank %d round %d' % (rank, rnd)
            assert torch.equal(Q, sync.base)
        out[rank] = 1
    finally:
        dist.destroy_process_group()


def test_replicated_table_delta_sync_world2():
    world = 2
    port = 29500 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
    assert dict(out) == {0: 1, 1: 1}


def test_single_process_sync_is_identity():
    Q = torch.ones(4, 4)
    s = parallel.ReplicatedTableSync(Q)
    Q += 1
    assert s.sync() is Q and bool((Q == 2).all()) and s.world == 1


# ---------------------------------------------------------------------------------------------
# sharded LightGCN: partition / remap logic and the collective schedule, gloo world_size 2.
# The kernels are replaced by CPU stand-ins INSIDE THIS TEST (the product default is the CUDA path).
# ---------------------------------------------------------------------------------------------
def _toy_graph(U, I, seed=0):
    import numpy as np
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    n = U + I
    rows, cols = [], []
    for u in range(U):
        for it in rng.choice(I, size=3, replace=False):
            rows += [u, U + it]; cols += [U + it, u]
    A = sp.csr_matrix((np.ones(len(rows), np.float32), (rows, cols)), shape=(n, n))
    d = np.asarray(A.sum(1)).ravel(); d[d == 0] = 1
    A = sp.diags(d ** -0.5) @ A @ sp.diags(d ** -0.5)
    A = A.tocsr(); A.sort_indices()
    return A.astype(np.float32)


def _cpu_kernels(lrowptr, lcols, lvals, reg, lr):
    import numpy as np
    from oracle import bpr_oracle as O

    def spmm(X, Y, acc, s):
        A = torch.sparse_csr_tensor(lrowptr, lcols.long(), lvals, size=(lrowptr.numel() - 1, X.shape[0]))
        Y.copy_(A @ X)
        if acc is not None:
            acc.add_(Y, alpha=s)

    def grad(Ue, Ve, u, i, j, gU, gV, loss):
        l, a, b = O.bpr_loss_grad(Ue.numpy(), Ve.numpy(), u.numpy(), i.numpy(), j.numpy(), 10e-8, reg)
        gU.add_(torch.from_numpy(a).float()); gV.add_(torch.from_numpy(b).float())   # same buffer: both add
        loss += l

    def adam(var, m, v, g, t):
        O.adam_tf1(var.numpy(), m.numpy(), v.numpy(), g.numpy(), lr, t)

    def scale(dst, src, s):
        dst.copy_(src * s)
    return spmm, grad, adam, scale


def _lgcn_worker(rank, world, port, out):
    import numpy as np
    from oracle import bpr_oracle as O
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        U, I, d, L, lr, reg = 8, 6, 4, 2, 0.01, 0.001
        A = _toy_graph(U, I)
        part = parallel.NodePartition(U, I, world)
        rp, co, va = (torch.from_numpy(x) for x in (A.indptr.astype(np.int64), A.indices.astype(np.int32), A.data))
        lrp, lco, lva = parallel.shard_adjacency(rp, co, va, part, rank)
        rng = np.random.default_rng(1)
        ego = (rng.standard_normal((U + I, d)) * 0.1).astype(np.float32)
        mine = part.local_nodes(rank)
        spmm, grad, adam, scale = _cpu_kernels(lrp, lco, lva, reg, lr)
        m = parallel.ShardedLightGCN(part, rank, lrp, lco, lva, torch.from_numpy(ego[mine.numpy()].copy()), L, lr, reg,
                                     spmm=spmm, grad=grad, adam=adam, scale=scale)
        # single-process reference: oracle.lightgcn_step on the whole graph
        Ur, Vr = ego[:U].copy(), ego[U:].copy()
        mU, vU, mV, vV = (np.zeros_like(x) for x in (Ur, Ur, Vr, Vr))
        for step in range(3):
            u = rng.integers(0, U, 5).astype(np.int32); i = rng.integers(0, I, 5).astype(np.int32)
            j = rng.integers(0, I, 5).astype(np.int32)
            ref_loss = O.lightgcn_step(A, Ur, Vr, mU, vU, mV, vV, u, i, j, L, lr, reg, step + 1)
            loss = m.train_step(torch.from_numpy(u), torch.from_numpy(i), torch.from_numpy(j))
            assert abs(float(loss) - ref_loss) < 1e-4 * abs(ref_loss) + 1e-6
            full_ref = np.concatenate([Ur, Vr])
            assert np.allclose(m.ego.numpy(), full_ref[mine.numpy()], rtol=1e-3, atol=1e-6), (rank, step)
        out[rank] = 1
    finally:
        dist.destroy_process_group()


def test_sharded_lightgcn_matches_single_process_world2():
    port = 31500 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_lgcn_worker, args=(2, port, out), nprocs=2, join=True)
    assert dict(out) == {0: 1, 1: 1}


def test_node_partition_roundtrip():
    part = parallel.NodePartition(8, 4, 2)
    g = part.to_gathered(torch.arange(12))
    assert sorted(g.tolist()) == list(range(12))
    assert g[:8].tolist() == [0, 1, 2, 3, 6, 7, 8, 9] and g[8:].tolist() == [4, 5, 10, 11]
    assert part.local_nodes(1).tolist() == [4, 5, 6, 7, 10, 11]
    with pytest.raises(ValueError):
        parallel.NodePartition(7, 4, 2)


# ---------------------------------------------------------------------------------------------
# K7: row-sharded item table, all-to-all row fetch / gradient return (gloo, CPU stand-in kernels)
# ---------------------------------------------------------------------------------------------
def _sharded_bpr_worker(rank, world, port, out):
    import numpy as np
    from oracle import c_oracle
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        U, I, d, lr, reg = 40, 60, 8, 0.05, 0.01
        rng = np.random.default_rng(0)
        P0 = (rng.random((U, d)) / 3).astype(np.float32)
        Q0 = (rng.random((I, d)) / 3).astype(np.float32)
        # a conflict-free global batch (every user and item once) so that the result equals the
        # sequential oracle exactly, split by user range
        u = rng.permutation(U)[:24].astype(np.int32)
        items = rng.permutation(I)[:48].astype(np.int32)
        i, j = items[:24].copy(), items[24:].copy()
        lo, hi = parallel.user_range(rank, world, U)
        bi = I // world
        lu, li, lj = parallel.shard_triples_by_user(torch.from_numpy(u), torch.from_numpy(i), torch.from_numpy(j), rank, world, U)

        def gather(T, idx, o):                                   # row -1 = empty slot -> zeros (as the kernel does)
            o.copy_(torch.where((idx >= 0)[:, None], T[idx.clamp(min=0).long()], torch.zeros(1)))

        def bucket(ids, cap, count, send, pos, ovf):             # numpy restatement of bucket_requests_kernel
            count.zero_(); send.fill_(-1)
            for k, idv in enumerate(ids.tolist()):
                owner = min(idv // bi, world - 1)
                slot = int(count[owner]); count[owner] += 1
                if slot < cap:
                    send[owner * cap + slot] = idv - owner * bi
                    pos[k] = owner * cap + slot
                else:
                    pos[k] = owner * cap; ovf.fill_(1)

        def staged(P, uu, pi, pj, R, D, loss):
            # the same arithmetic as the kernel, via the oracle's sequential step on private copies
            for k in range(uu.numel()):
                Pk = P[uu[k].long()].numpy()[None].copy()
                Qk = np.stack([R[pi[k].long()].numpy(), R[pj[k].long()].numpy()]).copy()
                q0 = Qk.copy()
                l = c_oracle.bpr_sgd_sequential(Pk, Qk, np.array([0], np.int32), np.array([0], np.int32),
                                                np.array([1], np.int32), lr, reg, reg)
                P[uu[k].long()] = torch.from_numpy(Pk[0])
                D[pi[k].long()] = torch.from_numpy(Qk[0] - q0[0])
                D[pj[k].long()] = torch.from_numpy(Qk[1] - q0[1])
                loss += l

        def scatter(G, idx, src):
            keep = idx >= 0
            G.index_add_(0, idx[keep].long(), src[keep])
        m = parallel.ShardedItemTableBPR(torch.from_numpy(P0[lo:hi].copy()), torch.from_numpy(Q0[rank * bi:(rank + 1) * bi].copy()),
                                         I, rank, world, lr, reg, reg, gather=gather, staged=staged, scatter=scatter, bucket=bucket,
                                         max_batch=64)
        assert m.capacity(12) == 24 and (1 << 20) < m.capacity(1 << 20) < 1.01 * (1 << 20)   # mean + slack*sigma + 64, capped at 2n
        loss = m.epoch(lu, li, lj, batch=5)                          # several minibatches, ragged tail
        m.check()                                                    # no bucket overflowed
        Pr, Qr = P0.copy(), Q0.copy()
        ref_loss = c_oracle.bpr_sgd_sequential(Pr, Qr, u, i, j, lr, reg, reg)
        tot = loss.clone()
        dist.all_reduce(tot)
        assert abs(float(tot) - ref_loss) < 1e-5 * ref_loss
        assert np.allclose(m.P.numpy(), Pr[lo:hi], rtol=1e-6, atol=1e-7)
        assert np.allclose(m.Q.numpy(), Qr[rank * bi:(rank + 1) * bi], rtol=1e-6, atol=1e-7)
        # a bucket that is too small is reported, not silently truncated
        tiny = parallel.ShardedItemTableBPR(m.P, m.Q, I, rank, world, lr, reg, reg, gather=gather, staged=staged, scatter=scatter,
                                            bucket=bucket, max_batch=64)
        tiny.capacity = lambda n: 1
        tiny.step(lu[:6], li[:6], lj[:6])
        flag = tiny.overflow.clone()
        dist.all_reduce(flag)
        assert int(flag) >= 1
        if int(tiny.overflow):
            with pytest.raises(RuntimeError):
                tiny.check()
        out[rank] = 1
    finally:
        dist.destroy_process_group()


def test_sharded_item_table_bpr_world2():
    port = 33500 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_sharded_bpr_worker, args=(2, port, out), nprocs=2, join=True)
    assert dict(out) == {0: 1, 1: 1}


# ---------------------------------------------------------------------------------------------
# LightGCN, user-partitioned / item-replicated: one all-reduce of the item block per layer
# ---------------------------------------------------------------------------------------------
def _user_sharded_worker(rank, world, port, out, blocks=1, row_lists=False):
    import numpy as np
    from oracle import bpr_oracle as O
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        U, I, d, L, lr, reg = 9, 6, 4, 2, 0.01, 0.001          # U not a multiple of the world size
        A = _toy_graph(U, I, seed=3)
        rp, co, va = (torch.from_numpy(x) for x in (A.indptr.astype(np.int64), A.indices.astype(np.int32), A.data))
        A_ui, A_iu, (lo, hi) = parallel.shard_bipartite_by_user(rp, co, va, U, I, rank, world)
        # the two blocks are transposes of each other and together cover the rank's edges
        D_ui = torch.sparse_csr_tensor(A_ui[0], A_ui[1].long(), A_ui[2], size=(hi - lo, I)).to_dense()
        D_iu = torch.sparse_csr_tensor(A_iu[0], A_iu[1].long(), A_iu[2], size=(I, hi - lo)).to_dense()
        assert torch.equal(D_ui.t(), D_iu)
        assert np.allclose(D_ui.numpy(), A.toarray()[lo:hi, U:])
        rng = np.random.default_rng(1)
        ego = (rng.standard_normal((U + I, d)) * 0.1).astype(np.float32)

        def spmm(Ablk, X, Y, acc, s):
            M = torch.sparse_csr_tensor(Ablk[0], Ablk[1].long(), Ablk[2], size=(Ablk[0].numel() - 1, X.shape[0]))
            Y.copy_(M @ X)
            if acc is not None:
                acc.add_(Y, alpha=s)

        def grad(Ue, Ve, u, i, j, gU, gV, loss):
            keep = (u >= 0).numpy()                       # u = -1: another rank's triple (K3 skips it)
            if not keep.any():
                return
            l, a, b = O.bpr_loss_grad(Ue.numpy(), Ve.numpy(), u.numpy()[keep], i.numpy()[keep], j.numpy()[keep], 10e-8, reg)
            gU.add_(torch.from_numpy(a).float()); gV.add_(torch.from_numpy(b).float())
            loss += l
        calls = []

        def dense(Ablk, n_cols):
            return torch.sparse_csr_tensor(Ablk[0], Ablk[1].long(), Ablk[2], size=(Ablk[0].numel() - 1, n_cols)).to_dense()

        def scatter(Ablk, rows, X, Y, acc, s):               # Y = B^T X over the edge lists of the listed source rows
            calls.append('scatter')
            listed = rows[rows >= 0].long()
            assert listed.numel() == torch.unique(listed).numel()
            keep = torch.zeros(X.shape[0], dtype=torch.bool); keep[listed] = True
            assert float(X[~keep].abs().sum()) == 0.0        # the caller's claim
            Y.copy_(dense(Ablk, Y.shape[0]).t() @ X)
            if acc is not None:
                acc.add_(Y, alpha=s)

        def list_rows(Ablk, rows, X, Y, compact, acc, s):    # the listed rows of A X, nothing else
            calls.append('rows')
            listed = rows[rows >= 0].long()
            assert listed.numel() == torch.unique(listed).numel()
            part = dense(Ablk, X.shape[0])[listed] @ X
            if Y is not None:
                assert compact
                Y.zero_(); Y[(rows >= 0).nonzero().ravel()] = part
            if acc is not None:
                acc[listed] += s * part

        def scatter_add(G, idx, src, s):
            ok = idx >= 0
            G.index_add_(0, idx[ok].long(), s * src[ok])
        def gather(T, idx, out_):                            # rows of T at idx; zeros for the -1 padding entries
            calls.append('gather')
            out_.zero_(); ok = idx >= 0
            out_[ok] = T[idx[ok].long()]
        extra = dict(scatter=scatter, rows=list_rows, scatter_add=scatter_add, gather=gather) if row_lists else {}
        m = parallel.UserShardedLightGCN(
            A_ui, A_iu, torch.from_numpy(ego[lo:hi].copy()), torch.from_numpy(ego[U:].copy()), L, lr, reg, lo,
            spmm=spmm, grad=grad, adam=lambda var, mm, v, g, t: O.adam_tf1(var.numpy(), mm.numpy(), v.numpy(), g.numpy(), lr, t),
            scale=lambda dst, src, s: dst.copy_(src * s), axpy=lambda dst, src, s: dst.add_(src, alpha=s),
            item_side_blocks=blocks, **extra)
        Ur, Vr = ego[:U].copy(), ego[U:].copy()
        mU, vU, mV, vV = (np.zeros_like(x) for x in (Ur, Ur, Vr, Vr))
        for step in range(3):
            u = rng.integers(0, U, 7).astype(np.int32); i = rng.integers(0, I, 7).astype(np.int32)
            j = rng.integers(0, I, 7).astype(np.int32)
            ref_loss = O.lightgcn_step(A, Ur, Vr, mU, vU, mV, vV, u, i, j, L, lr, reg, step + 1)
            # the graph-replay API on tensors that are not on a GPU is the eager step (nothing to capture)
            loss = (m.train_step_graphed if step == 2 else m.train_step)(torch.from_numpy(u), torch.from_numpy(i), torch.from_numpy(j))
            assert m.graph_error is None and parallel.captured_graphs() == 0 and m.step == step + 1
            assert abs(float(loss) - ref_loss) < 1e-4 * abs(ref_loss) + 1e-6
            assert np.allclose(m.Eu.numpy(), Ur[lo:hi], rtol=1e-3, atol=1e-6), (rank, step)
            assert np.allclose(m.Ei.numpy(), Vr, rtol=1e-3, atol=1e-6), (rank, step)
        if row_lists:       # per step: last forward layer = 2 listed-row products, the item gradients exchanged as a gathered [rows, d] block, first backward layer = 2 scatters
            assert calls == (['rows', 'rows', 'gather', 'scatter', 'scatter']) * 3, calls
        out[rank] = 1
    finally:
        dist.destroy_process_group()


def _column_sharded_worker(rank, world, port, out):
    import numpy as np
    from oracle import bpr_oracle as O
    from qrec_b200 import engine as E
    from qrec_b200.base.graphRecommender import DeviceCSR
    from conftest import row_list_kernel_stand_ins
    import test_sgl_model_cpu as S
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        S._stub(_Setattr)                                       # spmm / axpby / adam restatements
        calls = row_list_kernel_stand_ins(_Setattr)

        def partial_scores(U_, V_, u, i, j, reg, y_part, loss):  # the contract of qrec_bpr_partial_scores_f32
            uu, ii, jj = (x.long() for x in (u, i, j))
            y_part.copy_((U_[uu] * (V_[ii] - V_[jj])).sum(1))
            loss += reg * 0.5 * float((U_[uu] ** 2).sum() + (V_[ii] ** 2).sum() + (V_[jj] ** 2).sum())

        def grad_from_scores(U_, V_, u, i, j, y_full, eps, reg, log_weight, gU, gV, loss):
            uu, ii, jj = (x.long() for x in (u, i, j))
            sg = torch.sigmoid(y_full.double())
            gy = (-sg * (1 - sg) / (sg + eps)).float()[:, None]
            gU.index_add_(0, uu, gy * (V_[ii] - V_[jj]) + reg * U_[uu])
            gV.index_add_(0, ii, gy * U_[uu] + reg * V_[ii])
            gV.index_add_(0, jj, -gy * U_[uu] + reg * V_[jj])
            loss += log_weight * float((-torch.log(sg + eps)).sum())
        E.bpr_partial_scores, E.bpr_grad_from_scores = partial_scores, grad_from_scores
        U, I, d, L, lr, reg = 9, 6, 8, 3, 0.01, 0.001
        A = _toy_graph(U, I, seed=3)
        adj = DeviceCSR(A, 'cpu')
        rng = np.random.default_rng(1)
        ego = (rng.standard_normal((U + I, d)) * 0.1).astype(np.float32)
        dw = d // world
        m = parallel.ColumnShardedLightGCN(adj, torch.from_numpy(ego[:, rank * dw:(rank + 1) * dw].copy()), U, L, lr, reg)
        Ur, Vr = ego[:U].copy(), ego[U:].copy()
        mU, vU, mV, vV = (np.zeros_like(x) for x in (Ur, Ur, Vr, Vr))
        for step in range(3):
            u = rng.integers(0, U, 7).astype(np.int32); i = rng.integers(0, I, 7).astype(np.int32)
            j = rng.integers(0, I, 7).astype(np.int32)
            ref_loss = O.lightgcn_step(A, Ur, Vr, mU, vU, mV, vV, u, i, j, L, lr, reg, step + 1)
            loss = m.train_step(torch.from_numpy(u), torch.from_numpy(i), torch.from_numpy(j))
            assert abs(float(loss) - ref_loss) < 1e-4 * abs(ref_loss) + 1e-6, (rank, step, float(loss), ref_loss)
            full = m.gather_columns().numpy()                   # every rank assembles the whole table
            assert np.allclose(full[:U], Ur, rtol=1e-3, atol=1e-6) and np.allclose(full[U:], Vr, rtol=1e-3, atol=1e-6), (rank, step)
        # the restricted layers ran: last forward on the row list, first backward as a scatter -- per step
        assert calls == ['rows', 'scatter_rows'] * 3, calls
        fu, fv, _ = O.lightgcn_forward(A, Ur, Vr, L)
        prop = m.gather_columns(m.propagated()).numpy()
        assert np.allclose(prop[:U], fu, rtol=1e-3, atol=1e-6) and np.allclose(prop[U:], fv, rtol=1e-3, atol=1e-6)
        out[rank] = 1
    finally:
        dist.destroy_process_group()


def test_column_sharded_lightgcn_matches_single_process_world2():
    """parallel.ColumnShardedLightGCN (feature parallel: every rank holds d/2 columns of every row, the whole
    adjacency, and exchanges only the [B] partial scores): same trajectory as the single-process oracle."""
    port = 36300 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_column_sharded_worker, args=(2, port, out), nprocs=2, join=True)
    assert dict(out) == {0: 1, 1: 1}


def _exit_decision_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        assert parallel.any_rank_captured_graphs() is False
        if rank == 1:
            parallel._CAPTURED_GRAPHS[0] = 2          # as if only this rank's capture had succeeded
        assert parallel.any_rank_captured_graphs() is True      # ... every rank must still take the same way out
        parallel._CAPTURED_GRAPHS[0] = 0
        out[rank] = 1
    finally:
        dist.destroy_process_group()


def test_exit_decision_after_graph_capture_is_collective_world2(monkeypatch):
    """bench.py / the tools end through parallel.finish_process() when ANY rank holds a captured NCCL graph: a rank
    deciding on its own would leave the others in the barrier."""
    port = 36300 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_exit_decision_worker, args=(2, port, out), nprocs=2, join=True)
    assert dict(out) == {0: 1, 1: 1}
    # no process group: this process's own count (pinned here: GPU tests earlier in the session may have captured graphs)
    monkeypatch.setattr(parallel, '_CAPTURED_GRAPHS', [0])
    assert parallel.any_rank_captured_graphs() is False
    monkeypatch.setattr(parallel, '_CAPTURED_GRAPHS', [2])
    assert parallel.any_rank_captured_graphs() is True


def test_user_sharded_lightgcn_row_restricted_layers_world2():
    """The row-restricted layers of the sharded step (last forward layer evaluated on the batch's rows only, with
    the ranks' [rows, d] partial blocks all-reduced instead of the whole item block; first backward layer
    scattered from the batch's rows): same trajectory as the single-process oracle, which propagates every row."""
    port = 35900 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_user_sharded_worker, args=(2, port, out, 1, True), nprocs=2, join=True)
    assert dict(out) == {0: 1, 1: 1}


def test_user_sharded_lightgcn_matches_single_process_world2():
    port = 35500 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_user_sharded_worker, args=(2, port, out), nprocs=2, join=True)
    assert dict(out) == {0: 1, 1: 1}


def test_user_sharded_lightgcn_with_column_blocked_item_side_world2():
    """item_side_blocks=2: the item-side product runs as two passes over column blocks of the local
    users (split_csr_columns + blocked_spmm); same training trajectory as the single-process oracle."""
    port = 37500 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_user_sharded_worker, args=(2, port, out, 2), nprocs=2, join=True)
    assert dict(out) == {0: 1, 1: 1}


class _CpuOverlappedSync(parallel.OverlappedTableSync):
    """The two local kernels of csrc/table_sync.cu restated with torch arithmetic (CPU stand-ins, as the
    other gloo tests do for the engine kernels); `late` is applied to the table BETWEEN delta and merge,
    i.e. it plays the K1 wave that keeps running while the exchange is in flight."""
    late = None

    def _delta(self):
        torch.sub(self.table.view(-1), self.base.view(-1), out=self.D)
        self.S.copy_(self.D)

    def _merge(self):
        if self.late is not None:
            self.late()
            self.late = None
        self.table.view(-1).add_(self.S - self.D)
        self.base.view(-1).add_(self.S)


def _overlap_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        torch.manual_seed(0)
        Q0 = torch.randn(50, 8)
        Q = Q0.clone()
        sync = _CpuOverlappedSync(Q)
        assert sync.backend == 'collective' and sync.world == world
        expect = Q0.clone()

        def updates(seed):
            gg = torch.Generator().manual_seed(seed)
            return torch.randint(0, 50, (30,), generator=gg), torch.randn(30, 8, generator=gg)
        for rnd in range(3):
            for r in range(world):                     # wave `rnd`: every rank scatter-adds its own updates
                rows, upd = updates(100 * rnd + r)
                expect.index_add_(0, rows, upd)
                if r == rank:
                    Q.index_add_(0, rows, upd)
            # ... and the NEXT wave is already running when the merge lands: its updates must survive the
            # merge untouched and be exchanged by the following wave_done
            rows_l, upd_l = updates(7000 + 100 * rnd + rank)
            sync.late = lambda rows_l=rows_l, upd_l=upd_l: Q.index_add_(0, rows_l, upd_l)
            sync.wave_done()
            mine = torch.zeros_like(Q0).index_add_(0, rows_l, upd_l)
            assert torch.allclose(Q, expect + mine, atol=1e-5), 'rank %d round %d: local late updates lost' % (rank, rnd)
            assert torch.allclose(sync.base, expect, atol=1e-5), 'base is the globally agreed table'
            for r in range(world):                     # the late updates of all ranks join the global table next time
                rows_r, upd_r = updates(7000 + 100 * rnd + r)
                expect.index_add_(0, rows_r, upd_r)
        sync.wave_done()
        sync.finalize()
        assert torch.allclose(Q, expect, atol=1e-5) and torch.equal(Q, sync.base)
        gathered = [torch.empty_like(Q) for _ in range(world)]
        dist.all_gather(gathered, Q)
        assert all(torch.equal(gathered[0], t) for t in gathered), 'ranks must end bit-identical'
        out[rank] = 1
    finally:
        dist.destroy_process_group()


def test_overlapped_table_sync_world2():
    """parallel.OverlappedTableSync: updates that land in Q while an exchange is in flight are neither lost
    nor double-counted (Q - base == not-yet-exchanged local updates, for any interleaving)."""
    world = 2
    port = 31500 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_overlap_worker, args=(world, port, out), nprocs=world, join=True)
    assert dict(out) == {0: 1, 1: 1}


def test_overlapped_sync_single_process_is_identity():
    Q = torch.ones(4, 4)
    s = parallel.OverlappedTableSync(Q)
    Q += 1
    assert s.wave_done() is Q and s.finalize() is Q and bool((Q == 2).all()) and s.world == 1


# ---------------------------------------------------------------------------------------------
# SimGCL over a row-sharded user table (BASELINE config 5's decomposition), gloo world 2, kernel stand-ins
# ---------------------------------------------------------------------------------------------
class _Setattr(object):
    """monkeypatch-like shim for the spawned worker processes."""
    @staticmethod
    def setattr(obj, name, value):
        setattr(obj, name, value)

    @staticmethod
    def chdir(path):
        os.chdir(path)


def _simgcl_worker(rank, world, port, out):
    import numpy as np
    from oracle import tf_models
    from qrec_b200 import engine as E
    import test_sgl_model_cpu as S
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        S._stub(_Setattr)                                       # numpy / torch restatements of the kernels' contracts
        U, I, d, L, lr, reg, cl_rate, eps, seed = 9, 6, 8, 2, 0.01, 0.001, 0.5, 0.1, 0x5151
        A = _toy_graph(U, I, seed=3)

        from conftest import row_list_kernel_stand_ins
        calls = row_list_kernel_stand_ins(_Setattr)             # incl. the noise, keyed by the GLOBAL row
        rp, co, va = (torch.from_numpy(x) for x in (A.indptr.astype(np.int64), A.indices.astype(np.int32), A.data))
        A_ui, A_iu, (lo, hi) = parallel.shard_bipartite_by_user(rp, co, va, U, I, rank, world)
        rng = np.random.default_rng(1)
        ego = (rng.standard_normal((U + I, d)) * 0.3).astype(np.float32)
        m = parallel.UserShardedSimGCL(A_ui, A_iu, torch.from_numpy(ego[lo:hi].copy()), torch.from_numpy(ego[U:].copy()), L, lr, reg,
                                       lo, U, cl_rate, eps, noise_seed=seed, d_valid=d)
        ego_ref = ego.astype(np.float64)
        for step in range(1, 3):
            u = rng.integers(0, U, 7).astype(np.int32); i = rng.integers(0, I, 7).astype(np.int32)
            j = rng.integers(0, I, 7).astype(np.int32)
            noise = [[tf_models.philox_uniform(U + I, d, seed, e * 16 + k, step) for k in range(L)] for e in (1, 2)]
            rrec, rcl, rgrad = tf_models.simgcl_loss_and_grad(A, ego_ref, U, u, i, j, L, eps, cl_rate, reg, noise)
            m.train_step(torch.from_numpy(u), torch.from_numpy(i), torch.from_numpy(j))
            _, rec, cl = m.losses()
            assert abs(rec - rrec) <= 1e-4 * abs(rrec) and abs(cl - rcl) <= 1e-4 * abs(rcl), (rank, step, rec, rrec, cl, rcl)
            assert np.abs(m.tot_u.numpy() - rgrad[lo:hi]).max() <= 1e-3 * np.abs(rgrad).max(), (rank, step)
            assert np.abs(m.tot_i.numpy() - rgrad[U:]).max() <= 1e-3 * np.abs(rgrad).max(), (rank, step)
            # follow the engine's tables for the next step (Adam's first steps amplify rounding; the gradient is the check)
            parts = [None] * world
            dist.all_gather_object(parts, (lo, hi, m.Eu.numpy().copy()))
            for a, b, blk in parts:
                ego_ref[a:b] = blk
            ego_ref[U:] = m.Ei.numpy()
            # the replicated item rows are identical on every rank
            others = [None] * world
            dist.all_gather_object(others, m.Ei.numpy().copy())
            assert all(np.array_equal(others[0], o) for o in others)
        # per step: three encoders whose last layer runs on the batch's rows (2 listed-row products each, + the noise on
        # both blocks for the two perturbed views), and a backward pass whose first layer is 2 scatters
        per_step = ['rows', 'rows'] + ['rows', 'rows', 'perturb_listed', 'perturb_listed'] * 2 + ['scatter_rows'] * 2
        assert calls == per_step * 2, calls
        out[rank] = 1
    finally:
        dist.destroy_process_group()


def test_user_sharded_simgcl_matches_autograd_world2():
    """parallel.UserShardedSimGCL: noise keyed by the global row, item-block all-reduces per layer, InfoNCE over the
    batch's users assembled from their owners, collapsed backward -- equal to the float64 autograd restatement of
    model/ranking/SimGCL.py on every rank."""
    port = 37500 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_simgcl_worker, args=(2, port, out), nprocs=2, join=True)
    assert dict(out) == {0: 1, 1: 1}


# ---------------------------------------------------------------------------------------------
# NeuMF data parallel (8e): user tables sharded, item tables + MLP replicated; gloo world 2, kernel stand-ins
# ---------------------------------------------------------------------------------------------
def _neumf_stand_ins():
    """torch restatements of the contracts of the kernels NeuMF.train_step composes (include/qrec.h)."""
    import numpy as np
    from oracle import bpr_oracle as O
    from qrec_b200 import engine as E

    def tc_gemm(A, B, C, b_is_nk=False, epilogue=0, bias=None, mask=None):
        out = A @ (B.t() if b_is_nk else B)
        if epilogue in (E.EPI_BIAS_RELU, E.EPI_BIAS):
            out = out + bias
        if epilogue == E.EPI_BIAS_RELU:
            out = torch.relu(out)
        if epilogue == E.EPI_RELU_MASK:
            out = out * (mask > 0)
        C.copy_(out)

    def head(mode, training, UG, IG, H3, h_mf, h_mlp, r, reg, loss, y, dz, GMF, dUG, dIG, dH3):
        wg, wm = (1.0, 0.0) if mode == 0 else ((0.0, 1.0) if mode == 1 else (0.5, 0.5))
        z = 0
        if mode != 1:
            z = z + wg * ((UG * IG) * h_mf).sum(1)
        if mode != 0:
            z = z + wm * (H3 * h_mlp).sum(1)
        yy = torch.sigmoid(z)
        y.copy_(yy)
        if not training:
            return
        e = 10e-10
        d_y = -r / (yy + e) + (1 - r) / (1 - yy + e)
        dzz = d_y * yy * (1 - yy)
        dz.copy_(dzz)
        l = -(r * torch.log(yy + e) + (1 - r) * torch.log(1 - yy + e)).sum()
        if mode != 1:
            l = l + 0.5 * reg * ((UG * UG).sum() + (IG * IG).sum())
            GMF.copy_(UG * IG)
            dUG.copy_(wg * dzz[:, None] * h_mf * IG + reg * UG)
            dIG.copy_(wg * dzz[:, None] * h_mf * UG + reg * IG)
        if mode != 0:
            dH3.copy_((H3 > 0) * (wm * dzz[:, None] * h_mlp))
        loss += float(l)

    def gemv_t(A, v, out, alpha=1.0, beta=0.0):
        res = alpha * (A.t() @ (v if v is not None else torch.ones(A.shape[0])))
        out.copy_(res if beta == 0.0 else out + res)

    def sgemm(A, B, C, trans_a=False, trans_b=False, alpha=1.0, beta=0.0):
        prod = alpha * ((A.t() if trans_a else A) @ (B.t() if trans_b else B))
        C.copy_(prod if beta == 0.0 else prod + beta * C)
    E.tc_gemm, E.neumf_head, E.gemv_t, E.sgemm = tc_gemm, head, gemv_t, sgemm
    E.gather_rows = lambda T, idx, out: out.copy_(T[idx.long()])
    E.scatter_add_rows = lambda G, idx, src, scale=1.0: G.index_add_(0, idx.long(), scale * src)
    E.axpby = lambda dst, a, b, alpha, beta: dst.copy_(alpha * a + beta * b)
    E.adam_dense_tf1 = lambda var, m, v, g, lr, t, beta1=0.9, beta2=0.999, eps=1e-8: O.adam_tf1(var.numpy(), m.numpy(), v.numpy(), g.numpy(), lr, t)


def _neumf_worker(rank, world, port, out):
    import numpy as np
    from oracle import tf_models
    from qrec_b200.base.deepRecommender import DeepRecommender
    from qrec_b200.model.ranking.NeuMF import NeuMF
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        _neumf_stand_ins()
        DeepRecommender.initModel = lambda self: None           # synthetic ids: no data plumbing
        U, I, d, reg = 12, 9, 8, 0.01
        Sharded = parallel.make_user_sharded_neumf(NeuMF)

        def build(cls, nu):
            class FakeData(object):
                user, item = range(nu), range(I)
            m = cls.__new__(cls)
            m.data, m.num_users, m.num_items, m.emb_size, m.batch_size = FakeData(), nu, I, d, 4
            m.lRate, m.regU, m.regI, m.engine_device, m.engine_seed, m.device = 0.01, reg, reg, 0, 0, torch.device('cpu')
            m.initModel()
            return m
        full = build(NeuMF, U)
        rng = np.random.default_rng(3)
        for k, v in full.params.items():
            v.copy_(torch.from_numpy(rng.standard_normal(tuple(v.shape)).astype(np.float32) * 0.4))
        lo, hi = parallel.user_range(rank, world, U)
        m = build(Sharded, hi - lo).shard(lo)
        for k, v in full.params.items():
            m.params[k].copy_(v[lo:hi] if k in ('PG', 'PM') else v)
        for mode in (0, 1, 2):
            before = {k: v.numpy().astype(np.float64).copy() for k, v in full.params.items()}
            u = rng.integers(0, U, 20).astype(np.int32); i = rng.integers(0, I, 20).astype(np.int32)
            r = (rng.random(20) < 0.3).astype(np.float32)
            if mode == 1:
                u[:] = rng.integers(0, parallel.user_range(0, world, U)[1], 20)      # rank 1 owns none of this minibatch
            ref_loss, ref_g, _ = tf_models.neumf_loss_and_grad(before, mode, u, i, r, reg)
            full.train_step(mode, torch.from_numpy(u), torch.from_numpy(i), torch.from_numpy(r))
            loss = m.train_step(mode, torch.from_numpy(u), torch.from_numpy(i), torch.from_numpy(r))
            # the sharded gradients (after the reduction, with the parameter-only regularisers) equal autograd of the
            # reference's loss on the WHOLE minibatch ...
            for k in m.opt_vars[mode]:
                want = ref_g[k][lo:hi] if k in ('PG', 'PM') else ref_g[k]
                assert np.abs(m.grads[k].numpy() - want).max() <= 1e-4 * max(1e-3, np.abs(ref_g[k]).max()), (rank, mode, k)
            # ... and the parameters follow the single-process class
            for k, v in full.params.items():
                mine = v[lo:hi] if k in ('PG', 'PM') else v
                assert torch.allclose(m.params[k], mine, rtol=1e-4, atol=1e-6), (rank, mode, k)
            # kernel loss = BCE + per-sample L2; the h-vector terms are added by loss_value()
            extra = 0.0 if mode == 1 else reg * 0.5 * float((before['h_mf'] ** 2).sum())
            extra += reg * 0.5 * 0.25 * float((before['h_mf'] ** 2).sum() + (before['h_mlp'] ** 2).sum()) if mode == 2 else 0.0
            assert abs(float(loss) + extra - ref_loss) <= 1e-4 * abs(ref_loss), (rank, mode, float(loss), ref_loss)
        out[rank] = 1
    finally:
        dist.destroy_process_group()


def test_user_sharded_neumf_matches_autograd_world2():
    """parallel.make_user_sharded_neumf: samples routed to their user's owner, replicated gradients summed between
    backward and Adam, head-vector regularisers applied once -- gradients equal float64 autograd of
    model/ranking/NeuMF.py's three losses on the whole minibatch, parameters follow the single-process class."""
    port = 39500 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_neumf_worker, args=(2, port, out), nprocs=2, join=True)
    assert dict(out) == {0: 1, 1: 1}


def test_sorted_unique_padded_is_a_fixed_length_unique():
    """parallel._sorted_unique_padded: the distinct values, sorted, repeats replaced by -1 -- same multiset of
    non-negative values as torch.unique, length independent of the data (no host synchronisation in the step)."""
    g = torch.Generator().manual_seed(0)
    for n, hi in ((1, 5), (50, 7), (4096, 100000), (300, 3)):
        x = torch.randint(-1, hi, (n,), generator=g, dtype=torch.int32)
        s = parallel._sorted_unique_padded(x)
        assert s.shape == x.shape and s.dtype == torch.int32
        kept = s[s >= 0]
        assert torch.equal(kept, torch.unique(x[x >= 0]).int())
