"""Multi-GPU parity (pytest -m gpu; a case is skipped when the box has fewer GPUs than it needs): the sharded
step of xflow_b200/csrc/comm.cu + mg_kernels.cu (tokens routed to the owners of their keys over peer memory,
owners run the Pull / Push handlers on their range shard of the device table), driven through the C ABI from
one process per GPU, against the oracle's single-table lock-step schedule: every worker pulls before any
push of the round, pushes land in rank order (one FTRL / SGD step per (worker, key))."""
import os

import numpy as np
import pytest

from common import assert_close, assert_close_noise_aware
from oracle import oracle as O
from xflow_b200 import api, datagen

pytestmark = pytest.mark.gpu

ROUNDS = 3
M64 = (1 << 64) - 1


def _edge_keys(world):
    """Keys at the range boundaries of postoffice.cc:134-143 (width = floor((2^64-1)/S)) and in the tail
    [S*width, 2^64-1) that the reference leaves unowned (kv_app.h:430 CHECK) and this build clamps to the
    last shard.  2^64-1 itself is the table's EMPTY marker and never a key."""
    width = M64 // world
    ks = [0, 1, width - 1, width, width + 1, (world - 1) * width - 1, (world - 1) * width, world * width - 1,
          min(world * width, M64 - 1), 0xFFFFFFFFFFFFFFF8, 0xFFFFFFFFFFFFFFFE]
    return np.array(sorted(set(k for k in ks if 0 <= k < M64)), np.uint64)


def _batch(case, world, rank, rnd):
    rp, keys, lab = datagen.make_csr_keys(500 + 10 * rnd + rank, case["B"], case["D"], case["space"], api.hash_decimal_ids,
                                          dist=case["dist"], zipf_s=1.1, ragged=case.get("ragged", False))
    if case.get("edges") and keys.size:
        e = _edge_keys(world)
        keys = keys.copy()
        n = min(e.size, keys.size)
        keys[:n] = e[:n]          # the first tokens of the batch carry the boundary keys
    return rp, keys, lab


def _imported(case, world):
    ks = np.unique(np.concatenate([_batch(case, world, r, 0)[1][:300] for r in range(world)]))
    rng = np.random.default_rng(77)
    return (ks, rng.normal(0, 0.3, ks.size).astype(np.float32), rng.uniform(0, 2, ks.size).astype(np.float32),
            rng.normal(0, 1, ks.size).astype(np.float32))


def _all_keys(case, world):
    return np.unique(np.concatenate([_batch(case, world, r, rnd)[1] for r in range(world) for rnd in range(ROUNDS)] +
                                    [np.zeros(1, np.uint64)]))


def _worker(rank, world, id_path, case, ret):
    from xflow_b200 import api as A
    if rank == 0:
        cid = A.Comm.new_id()
        np.save(id_path + ".tmp.npy", cid)
        os.replace(id_path + ".tmp.npy", id_path)
    else:
        import time
        while not os.path.exists(id_path):
            time.sleep(0.05)
        cid = np.load(id_path)
    model = A.MODEL_LR if case["model"] == "lr" else A.MODEL_FM
    opt = A.OPT_FTRL if case["opt"] == "ftrl" else A.OPT_SGD
    comm = A.Comm(cid, rank, world, rank)
    table = A.Table(latent_dim=case["K"], optimizer=opt, device=rank, v_init=A.VINIT_COUNTER, seed=9, shard_index=rank,
                    num_shards=world, capacity=1 << 16)
    max_nnz = max(_batch(case, world, r, rnd)[1].size for r in range(world) for rnd in range(ROUNDS)) + 8
    tr = A.Trainer(table, model=model, max_rows=case["B"], max_nnz=max_nnz, keep_loss=True, comm=comm)
    tr.init_push()
    if case.get("imported"):
        # rows whose weight is NOT f(z, n) (a model file loaded before training): the lazy table keeps such a
        # weight beside the state and the Push takes a fresh look at those rows instead of the stashed one
        ik, iw, inw, izw = _imported(case, world)
        mine = np.array([A.shard_of(int(k), world) == rank for k in ik])
        table.import_(ik[mine], w=iw[mine], nw=inw[mine], zw=izw[mine])
    comm.barrier()
    losses = []
    for rnd in range(ROUNDS):
        rp, keys, lab = _batch(case, world, rank, rnd)
        tr.step_host(rp, keys, lab)
        losses.append(tr.get_loss(case["B"]))
    # forward only through the sharded path (same collective schedule on every rank), on a batch whose keys
    # all exist already, so nothing changes in the table
    rp, keys, lab = _batch(case, world, rank, ROUNDS - 1)
    pctr = tr.predict_host(rp, keys)
    tr.sync()
    comm.barrier()
    allk = _all_keys(case, world)
    mine = np.array([A.shard_of(int(k), world) == rank for k in allk])
    ret[rank] = dict(keys=allk[mine], e=table.export(allk[mine]), losses=losses, size=table.size(),
                     uniq=tr.stats()["unique_keys"], pctr=pctr, launches=tr.launches())
    # foreign keys must be absent from this shard
    other = table.export(allk[~mine][:2000])
    assert not other["present"].any()
    comm.barrier()
    tr.close()
    table.close()
    comm.close()


CASES = {
    "lr_ftrl": dict(model="lr", opt="ftrl", K=0, B=4096, D=32, space=200000, dist="uniform"),
    "lr_ftrl_zipf_edges": dict(model="lr", opt="ftrl", K=0, B=4096, D=24, space=10 ** 9, dist="zipf", edges=True, ragged=True),
    "lr_ftrl_imported": dict(model="lr", opt="ftrl", K=0, B=2048, D=32, space=100000, dist="uniform", imported=True),
    "lr_sgd": dict(model="lr", opt="sgd", K=0, B=2048, D=16, space=50000, dist="uniform"),
    "fm_ftrl_k8": dict(model="fm", opt="ftrl", K=8, B=4096, D=32, space=200000, dist="uniform"),
    "fm_sgd_k4": dict(model="fm", opt="sgd", K=4, B=4096, D=32, space=200000, dist="uniform"),
    "fm_ftrl_k16_zipf": dict(model="fm", opt="ftrl", K=16, B=4096, D=32, space=10 ** 8, dist="zipf", edges=True),
    "fm_ftrl_k64": dict(model="fm", opt="ftrl", K=64, B=2048, D=32, space=100000, dist="uniform"),
    "fm_sgd_k33": dict(model="fm", opt="sgd", K=33, B=2048, D=32, space=100000, dist="uniform"),
}
RUNS = [(2, "lr_ftrl"), (2, "lr_ftrl_imported"), (2, "lr_ftrl_zipf_edges"), (2, "lr_sgd"), (2, "fm_ftrl_k8"), (2, "fm_sgd_k4"), (2, "fm_ftrl_k16_zipf"),
        (2, "fm_ftrl_k64"), (2, "fm_sgd_k33"), (4, "lr_ftrl_zipf_edges"), (4, "fm_ftrl_k16_zipf"), (8, "lr_ftrl_zipf_edges"), (8, "fm_ftrl_k16_zipf")]


def _lockstep_oracle(case, world, exact):
    oopt = O.OPT_FTRL if case["opt"] == "ftrl" else O.OPT_SGD
    K = case["K"]
    t = O.Table(K=K, opt=oopt, init_mode=O.INIT_COUNTER, seed=9)
    for _ in range(world):
        t.init_push()
    if case.get("imported"):
        ik, iw, inw, izw = _imported(case, world)
        t.import_(ik, w=iw, nw=inw, zw=izw)
    losses = {r: [] for r in range(world)}
    uniq = {r: 0 for r in range(world)}

    def run():
        for rnd in range(ROUNDS):
            pend = []
            for r in range(world):                       # every worker pulls + computes first ...
                rp, keys, lab = _batch(case, world, r, rnd)
                uk, gw, gv, loss = t.worker_compute(rp.astype(np.int64), keys, lab.astype(np.int32))
                pend.append((uk, gw, gv))
                losses[r].append(loss)
                uniq[r] += uk.size
            for uk, gw, gv in pend:                      # ... then the pushes land in rank order
                t.push(uk, gw, gv if K else None)
    if exact:
        with O.exact_sums():
            run()
    else:
        run()
    return t, losses, uniq


@pytest.mark.parametrize("world,name", RUNS, ids=["w%d-%s" % r for r in RUNS])
def test_sharded_step_matches_lockstep_oracle(world, name, tmp_path):
    if api.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    import torch.multiprocessing as mp
    case = CASES[name]
    K = case["K"]
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, str(tmp_path / "ncclid.npy"), case, ret), nprocs=world, join=True)
    t, ref_losses, uniq = _lockstep_oracle(case, world, exact=False)
    tx, ex_losses, _ = _lockstep_oracle(case, world, exact=True)   # noise yardstick for hot keys
    skew = case["dist"] == "zipf"
    total = 0
    for r in range(world):
        got = ret[r]
        assert got["uniq"] == uniq[r], "rank %d: unique keys counted by the owners" % r   # dedup is exact
        for a, b, c in zip(got["losses"], ref_losses[r], ex_losses[r]):
            if skew:
                # a hot key's reference noise shows in every row that holds the key (17 % of the rows at 8 ranks, also
                # for a float64 numpy model of the protocol): each row must be inside 8x that noise, their share is free
                assert_close_noise_aware(a, b, c, "loss rank %d" % r, abs_floor=1e-6, max_noisy_frac=1.0)
            else:
                assert_close(a, b, "loss rank %d" % r, abs_floor=1e-6)
        ref, refx = t.export(got["keys"]), tx.export(got["keys"])
        assert np.array_equal(got["e"]["present"], ref["present"])      # bucketing bit-exact, incl. clamped tail keys
        for k in ("w", "nw", "zw") + (("v", "nv", "zv") if K else ()):
            if skew:
                assert_close_noise_aware(got["e"][k], ref[k], refx[k], "rank %d %s" % (r, k), max_noisy_frac=0.02)
            else:
                assert_close(got["e"][k], ref[k], "rank %d %s" % (r, k))
        total += got["size"]
        assert got["launches"] > 0
    assert total == t.size()
    # every boundary key sits on the shard the rule names (and only there: checked in the workers)
    if case.get("edges"):
        for k in _edge_keys(world):
            owner = api.shard_of(int(k), world)
            assert owner == O.shard_of(int(k), world)
            assert k in ret[owner]["keys"]
    # predictions after training: the oracle's forward pass on the final table
    for r in range(world):
        rp, keys, lab = _batch(case, world, r, ROUNDS - 1)
        _, _, _, loss = t.worker_compute(rp.astype(np.int64), keys, lab.astype(np.int32))
        _, _, _, lossx = tx.worker_compute(rp.astype(np.int64), keys, lab.astype(np.int32))
        if skew:
            assert_close_noise_aware(ret[r]["pctr"], loss.astype(np.float64) + lab, lossx.astype(np.float64) + lab,
                                     "pctr rank %d" % r, abs_floor=1e-6, max_noisy_frac=1.0)
        else:
            assert_close(ret[r]["pctr"], loss.astype(np.float64) + lab, "pctr rank %d" % r, abs_floor=1e-6)
