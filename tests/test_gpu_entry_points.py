"""Every way of feeding a batch to a trainer (pytest -m gpu): host arrays, page-locked arrays, page-locked u32 ids
hashed on the device, device-resident CSR and the ingested text block.  The same batches through any of them leave
the same table, bit for bit; each entry point keeps its own rules for empty batches, for what it counts and for the
arguments it refuses."""
import ctypes as C

import numpy as np
import pytest

from xflow_b200 import api, datagen

pytestmark = pytest.mark.gpu

OK, ERR_ARG = 0, -1
# ids from a large space: a key occurs about once per batch, so the per-key sums of the FM steps have at most two
# terms and come out the same whatever order the atomics land in
SPACE = 1 << 30


def _torch():
    import torch
    return torch


def _bytes(a):
    """A numpy array's bytes as a torch uint8 tensor (host, shared memory)."""
    return _torch().from_numpy(np.ascontiguousarray(a).view(np.uint8))


def _ptrs(*tensors):
    return [C.c_void_p(t.data_ptr()) for t in tensors]


def _batches(seed, d):
    """4096 rows, 1500 ragged rows, and 8 rows: one thread block, so its loss sum is added up in a fixed order."""
    out = []
    for i, (rows, ragged) in enumerate(((4096, False), (1500, True), (8, False))):
        rp, ids, lab = datagen.make_ids(seed + i, rows, d, SPACE, ragged=ragged)
        vals = (datagen.uniform_u64(seed + i, ids.size, stream=5) % np.uint64(1000)).astype(np.float32) / 500.0 - 0.9
        out.append(dict(rp=rp, ids=ids.astype(np.uint32), keys=api.hash_decimal_ids(ids), lab=lab, vals=vals))
    return out


# ---- one step through each entry point; returns the mean |loss| the call reports (None: it reports none)
def _step_host(tr, b):
    return np.float32(tr.step_host(b["rp"], b["keys"], b["lab"]))


def _step_host_async(tr, b, ids=False):
    torch = _torch()
    bufs = [_bytes(a).pin_memory() for a in (b["rp"], b["ids"] if ids else b["keys"], b["lab"])]
    out = torch.full((1,), -1.0, dtype=torch.float32).pin_memory()
    fn = api.lib().xf_trainer_step_host_ids_async if ids else api.lib().xf_trainer_step_host_async
    assert fn(tr.h, *_ptrs(*bufs), b["lab"].size, b["keys"].size, C.c_void_p(out.data_ptr())) == OK
    tr.sync()
    return np.float32(out[0].item()) / np.float32(b["lab"].size)


def _step_host_ids_async(tr, b):
    return _step_host_async(tr, b, ids=True)


def _step_device(tr, b):
    torch = _torch()
    bufs = [_bytes(a).cuda() for a in (b["rp"], b["keys"], b["lab"])]
    torch.cuda.synchronize()
    tr.step_device(*[t.data_ptr() for t in bufs], b["lab"].size, b["keys"].size)
    tr.sync()
    return None


def _step_host_values(tr, b):
    return np.float32(tr.step_host_values(b["rp"], b["keys"], b["vals"], b["lab"]))


def _step_device_values(tr, b):
    torch = _torch()
    d_rp, d_keys, d_vals, d_lab = [_bytes(a).cuda() for a in (b["rp"], b["keys"], b["vals"], b["lab"])]
    torch.cuda.synchronize()
    assert api.lib().xf_trainer_step_device_values(tr.h, *_ptrs(d_rp, d_keys, d_vals, d_lab), b["lab"].size,
                                                   b["keys"].size) == OK, api.lib().xf_last_error()
    tr.sync()
    return None


GROUPS = {
    # name: (latent_dim, canonical, model, {entry point: (step, launches per call)})
    "lr_ftrl": (0, 0, api.MODEL_LR, {"step_host": (_step_host, 1), "step_host_async": (_step_host_async, 1),
                                     "step_host_ids_async": (_step_host_ids_async, 2), "step_device": (_step_device, 1)}),
    "fm_ftrl_k8": (8, 0, api.MODEL_FM, {"step_host": (_step_host, 2), "step_device": (_step_device, 2)}),
    "fm_canonical_k8": (8, 1, api.MODEL_FM_CANONICAL, {"step_host_values": (_step_host_values, 2),
                                                       "step_device_values": (_step_device_values, 2)}),
}


def _predict_three_ways(tr, b, tmp_path):
    """predict_host, predict_ingested and predict_ingested_metric on the first 512 rows of batch b."""
    lib = api.lib()
    n = 512
    rp, ids, lab = b["rp"][: n + 1], b["ids"][: b["rp"][n]], b["lab"][:n]
    p_host = tr.predict_host(rp, b["keys"][: b["rp"][n]])
    path = str(tmp_path / "predict.txt")
    datagen.write_text(path, rp, ids.astype(np.uint64), lab)
    assert tr.ingest_text(open(path, "rb").read()) == (n, int(rp[-1]))
    p_ing, lab_ing = tr.predict_ingested(0, n)
    assert np.array_equal(lab_ing, lab)
    m = C.c_void_p()
    assert lib.xf_metric_create(C.byref(m), 0) == OK
    p_met, lab_met = np.empty(n, np.float32), np.empty(n, np.uint8)
    assert lib.xf_trainer_predict_ingested_metric(tr.h, 0, n, m, api._p(p_met), api._p(lab_met)) == OK
    lib.xf_metric_destroy(m)
    assert np.array_equal(lab_met, lab)
    return p_host, p_ing, p_met


@pytest.mark.parametrize("group", sorted(GROUPS))
def test_every_entry_point_leaves_the_same_table(group, tmp_path):
    K, canon, model, paths = GROUPS[group]
    batches = _batches(40 + K + canon, 16 if K == 0 else 12)
    keys = np.unique(np.concatenate([b["keys"] for b in batches]))
    fields = ("w", "nw", "zw") + (("v", "nv", "zv") if K else ())
    runs = {}
    for name, (step, launches) in paths.items():
        t = api.Table(latent_dim=K, optimizer=api.OPT_FTRL, capacity=1 << 21, seed=3, canonical_fm=canon)
        tr = api.Trainer(t, model=model, max_rows=4096, max_nnz=4096 * 24, keep_loss=True)
        means, residuals = [], []
        for b in batches:
            l0 = tr.launches()
            means.append(step(tr, b))
            assert tr.launches() - l0 == launches, (name, tr.launches() - l0)
            residuals.append(tr.get_loss(b["lab"].size))
        st = tr.stats()
        assert (st["steps"], st["rows"], st["nnz"]) == (len(batches), sum(b["lab"].size for b in batches),
                                                        sum(b["keys"].size for b in batches)), (name, st)
        e = t.export(keys)
        assert e["present"].all()
        preds = _predict_three_ways(tr, batches[0], tmp_path) if not canon else None
        runs[name] = dict(means=means, residuals=residuals, stats=st, export=e, size=t.size(), preds=preds)
        tr.close()
        t.close()
    names = list(runs)
    a = runs[names[0]]
    if a["preds"] is not None:
        p_host, p_ing, p_met = a["preds"]
        assert np.array_equal(p_host.view(np.uint32), p_ing.view(np.uint32))
        assert np.array_equal(p_host.view(np.uint32), p_met.view(np.uint32))
    for other in names[1:]:
        o = runs[other]
        assert o["stats"] == a["stats"] and o["size"] == a["size"], (other, o["stats"], a["stats"])
        for f in fields:
            assert np.array_equal(o["export"][f].view(np.uint32), a["export"][f].view(np.uint32)), (other, f)
        for i, (ra, ro) in enumerate(zip(a["residuals"], o["residuals"])):
            assert np.array_equal(ra.view(np.uint32), ro.view(np.uint32)), (other, "residuals of batch", i)
        if o["preds"] is not None:
            for pa, po in zip(a["preds"], o["preds"]):
                assert np.array_equal(pa.view(np.uint32), po.view(np.uint32)), other
    # the mean |loss| wherever an entry point reports one: bit-equal on the one-block batch; on the larger ones the
    # thread blocks' partial sums are added in the order they finish, which moves the last bits
    reported = [n for n in names if runs[n]["means"][0] is not None]
    for other in reported[1:]:
        for i, b in enumerate(batches):
            x, y = runs[reported[0]]["means"][i], runs[other]["means"][i]
            if b["lab"].size <= 8:
                assert x.view(np.uint32) == y.view(np.uint32), (other, i, x, y)
            else:
                blocks = -(-b["lab"].size // 8)
                assert abs(float(x) - float(y)) <= 2 * blocks * 2.0 ** -24 * abs(float(x)), (other, i, x, y)


# ---- the rules of each entry point
def _lr(max_rows=64):
    t = api.Table(latent_dim=0, optimizer=api.OPT_FTRL, capacity=1 << 16, seed=3)
    return t, api.Trainer(t, model=api.MODEL_LR, max_rows=max_rows, max_nnz=max_rows * 8)


def _counts(tr):
    s = tr.stats()
    return s["steps"], s["rows"], s["nnz"]


def _small(seed, rows=40, d=4):
    rp, ids, lab = datagen.make_ids(seed, rows, d, SPACE)
    return rp, ids, api.hash_decimal_ids(ids), lab


def _ingest(tr, tmp_path, seed=7, rows=40):
    rp, ids, keys, lab = _small(seed, rows)
    path = str(tmp_path / ("block%d.txt" % seed))
    datagen.write_text(path, rp, ids, lab)
    assert tr.ingest_text(open(path, "rb").read()) == (rows, keys.size)
    return rows, keys.size


def test_empty_batches_and_what_each_entry_point_counts(tmp_path):
    torch = _torch()
    lib = api.lib()
    t, tr = _lr()
    rp, ids, keys, lab = _small(1)
    empty_rp = np.zeros(1, np.uint32)
    one = np.zeros(1, np.uint64)
    mean = C.c_float(7.0)

    # step_device: an empty batch is counted as a step (no rows, no tokens), nothing is launched
    d_rp, d_keys, d_lab = [_bytes(a).cuda() for a in (rp, keys, lab)]
    torch.cuda.synchronize()
    l0 = tr.launches()
    assert lib.xf_trainer_step_device(tr.h, *_ptrs(d_rp, d_keys, d_lab), 0, 0) == OK
    assert _counts(tr) == (1, 0, 0) and tr.launches() == l0
    # step_host: *mean = 0, not counted
    assert lib.xf_trainer_step_host(tr.h, api._p(empty_rp), api._p(one), api._p(lab), 0, 0, C.byref(mean)) == OK
    assert mean.value == 0.0 and _counts(tr) == (1, 0, 0)
    # the _async calls: not counted; the empty batch returns before the page-locked check
    for fn in (lib.xf_trainer_step_host_async, lib.xf_trainer_step_host_ids_async):
        assert fn(tr.h, api._p(empty_rp), api._p(one), api._p(lab), 0, 0, None) == OK
    assert _counts(tr) == (1, 0, 0)
    # predict_host: OK, never counted
    out = np.empty(1, np.float32)
    assert lib.xf_trainer_predict_host(tr.h, api._p(empty_rp), api._p(one), 0, 0, api._p(out)) == OK
    tr.predict_host(rp, keys)
    assert _counts(tr) == (1, 0, 0)
    # every step counts its rows and tokens ...
    tr.step_host(rp, keys, lab)
    assert _counts(tr) == (2, 40, keys.size)
    # ... except step_ingested, which counts rows but leaves the token count alone
    rows, _ = _ingest(tr, tmp_path)
    assert lib.xf_trainer_step_ingested(tr.h, 3, 3) == OK
    assert _counts(tr) == (2, 40, keys.size)
    tr.step_ingested(0, rows)
    tr.step_ingested(10, 25)
    assert _counts(tr) == (4, 40 + rows + 15, keys.size)
    # predict_ingested: an empty range returns before pctr_out is checked; a non-empty one needs it
    assert lib.xf_trainer_predict_ingested(tr.h, 2, 2, None, None) == OK
    assert lib.xf_trainer_predict_ingested(tr.h, 0, rows, None, None) == ERR_ARG
    tr.predict_ingested(0, rows)
    # predict_ingested_metric: OK on an empty range, asynchronous without result buffers, never counted
    m = C.c_void_p()
    assert lib.xf_metric_create(C.byref(m), 0) == OK
    assert lib.xf_trainer_predict_ingested_metric(tr.h, 5, 5, m, None, None) == OK
    assert lib.xf_trainer_predict_ingested_metric(tr.h, 0, rows, m, None, None) == OK
    tr.sync()
    res = (C.c_double * 6)()
    assert lib.xf_metric_finish(m, None, res) == OK and res[2] + res[3] == rows
    lib.xf_metric_destroy(m)
    assert _counts(tr) == (4, 40 + rows + 15, keys.size)
    tr.close()
    t.close()

    # the canonical FM's value entry points
    t = api.Table(latent_dim=8, optimizer=api.OPT_FTRL, capacity=1 << 16, seed=3, canonical_fm=1)
    tr = api.Trainer(t, model=api.MODEL_FM_CANONICAL, max_rows=64, max_nnz=512)
    mean.value = 7.0
    assert lib.xf_trainer_step_host_values(tr.h, api._p(empty_rp), api._p(one), None, api._p(lab), 0, 0,
                                           C.byref(mean)) == OK
    assert mean.value == 0.0 and _counts(tr) == (0, 0, 0)
    assert lib.xf_trainer_predict_host_values(tr.h, api._p(empty_rp), api._p(one), None, 0, 0, api._p(out)) == OK
    assert lib.xf_trainer_step_device_values(tr.h, *_ptrs(d_rp, d_keys), None, C.c_void_p(d_lab.data_ptr()), 0, 0) == OK
    assert _counts(tr) == (1, 0, 0)
    tr.step_host_values(rp, keys, None, lab)
    tr.predict_host_values(rp, keys, None)
    assert _counts(tr) == (2, 40, keys.size)
    tr.close()
    t.close()

    # the multi-view machine's field entry points
    t = api.Table(latent_dim=8, optimizer=api.OPT_FTRL, capacity=1 << 16, seed=3, canonical_fm=1)
    tr = api.Trainer(t, model=api.MODEL_MVM, max_rows=64, max_nnz=512)
    mean.value = 7.0
    f1 = np.zeros(1, np.uint8)
    assert lib.xf_trainer_step_host_fields(tr.h, api._p(empty_rp), api._p(one), api._p(f1), None, api._p(lab), 0, 0,
                                           C.byref(mean)) == OK
    assert mean.value == 0.0 and _counts(tr) == (0, 0, 0)
    assert lib.xf_trainer_predict_host_fields(tr.h, api._p(empty_rp), api._p(one), api._p(f1), None, 0, 0,
                                              api._p(out)) == OK
    fields = (np.arange(keys.size) % 5).astype(np.uint8)
    tr.step_host_fields(rp, keys, fields, None, lab)
    tr.predict_host_fields(rp, keys, fields, None)
    assert _counts(tr) == (1, 40, keys.size)
    tr.close()
    t.close()


def _refused(call, t, tr, valid_step):
    """call() returns XF_ERR_ARG, launches nothing and leaves the table as it was; the next valid step works."""
    n, launches = t.size(), tr.launches()
    assert call() == ERR_ARG, api.lib().xf_last_error()
    assert t.size() == n and tr.launches() == launches
    valid_step()


def test_refused_arguments(tmp_path):
    torch = _torch()
    lib = api.lib()
    P = api._p
    t, tr = _lr(max_rows=64)
    rp, ids, keys, lab = _small(2)
    big_rp, big_ids, big_keys, big_lab = _small(3, rows=65, d=1)
    ids32 = ids.astype(np.uint32)
    mean = C.c_float()
    out = np.empty(65, np.float32)
    seeds = iter(range(100, 1000))

    def step():
        r, _, k, y = _small(next(seeds))
        tr.step_host(r, k, y)

    d = [_bytes(a).cuda() for a in (rp, keys, lab)]
    d_big = [_bytes(a).cuda() for a in (big_rp, big_keys, big_lab)]
    pin = [_bytes(a).pin_memory() for a in (rp, keys, lab)]
    pin_ids = _bytes(ids32).pin_memory()
    pin_out = torch.zeros(1, dtype=torch.float32).pin_memory()
    torch.cuda.synchronize()
    n, z = lab.size, keys.size
    SH, SD = lib.xf_trainer_step_host, lib.xf_trainer_step_device
    SA, SI = lib.xf_trainer_step_host_async, lib.xf_trainer_step_host_ids_async
    cases = [
        # null arrays
        lambda: SH(tr.h, None, P(keys), P(lab), n, z, C.byref(mean)),
        lambda: SH(tr.h, P(rp), None, P(lab), n, z, C.byref(mean)),
        lambda: SH(tr.h, P(rp), P(keys), None, n, z, C.byref(mean)),
        lambda: SD(tr.h, None, *_ptrs(d[1], d[2]), n, z),
        lambda: SD(tr.h, C.c_void_p(d[0].data_ptr()), None, C.c_void_p(d[2].data_ptr()), n, z),
        lambda: SD(tr.h, *_ptrs(d[0], d[1]), None, n, z),
        lambda: SA(tr.h, *_ptrs(pin[0], pin[1]), None, n, z, None),
        lambda: SI(tr.h, C.c_void_p(pin[0].data_ptr()), None, C.c_void_p(pin[2].data_ptr()), n, z, None),
        lambda: lib.xf_trainer_predict_host(tr.h, P(rp), P(keys), n, z, None),
        lambda: lib.xf_trainer_predict_host(tr.h, P(rp), None, n, z, P(out)),
        # rows > max_rows
        lambda: SH(tr.h, P(big_rp), P(big_keys), P(big_lab), 65, big_keys.size, C.byref(mean)),
        lambda: SD(tr.h, *_ptrs(*d_big), 65, big_keys.size),
        lambda: lib.xf_trainer_predict_host(tr.h, P(big_rp), P(big_keys), 65, big_keys.size, P(out)),
        # pageable buffers for the page-locked entry points (each array, and the loss slot)
        lambda: SA(tr.h, P(rp), *_ptrs(pin[1], pin[2]), n, z, None),
        lambda: SA(tr.h, C.c_void_p(pin[0].data_ptr()), P(keys), C.c_void_p(pin[2].data_ptr()), n, z, None),
        lambda: SA(tr.h, *_ptrs(pin[0], pin[1]), P(lab), n, z, None),
        lambda: SA(tr.h, *_ptrs(*pin), n, z, P(out)),
        lambda: SI(tr.h, C.c_void_p(pin[0].data_ptr()), P(ids32), C.c_void_p(pin[2].data_ptr()), n, z, None),
        lambda: SI(tr.h, *_ptrs(pin[0], pin_ids, pin[2]), n, z, P(out)),
        # the value and field entry points on a trainer of another model
        lambda: lib.xf_trainer_step_host_values(tr.h, P(rp), P(keys), None, P(lab), n, z, C.byref(mean)),
        lambda: lib.xf_trainer_predict_host_values(tr.h, P(rp), P(keys), None, n, z, P(out)),
        lambda: lib.xf_trainer_step_device_values(tr.h, *_ptrs(d[0], d[1]), None, C.c_void_p(d[2].data_ptr()), n, z),
        lambda: lib.xf_trainer_step_host_fields(tr.h, P(rp), P(keys), P(np.zeros(z, np.uint8)), None, P(lab), n, z,
                                                C.byref(mean)),
        lambda: lib.xf_trainer_predict_host_fields(tr.h, P(rp), P(keys), P(np.zeros(z, np.uint8)), None, n, z, P(out)),
    ]
    for call in cases:
        _refused(call, t, tr, step)
    # the same arrays are accepted where they belong
    assert SA(tr.h, *_ptrs(*pin), n, z, C.c_void_p(pin_out.data_ptr())) == OK
    assert SI(tr.h, *_ptrs(pin[0], pin_ids, pin[2]), n, z, C.c_void_p(pin_out.data_ptr())) == OK
    tr.sync()

    # ingested row ranges: out of bounds or reversed
    rows, _ = _ingest(tr, tmp_path)
    m = C.c_void_p()
    assert lib.xf_metric_create(C.byref(m), 0) == OK
    p = np.empty(rows + 1, np.float32)
    for lo, hi in ((0, rows + 1), (rows + 1, rows + 1), (5, 3)):
        _refused(lambda: lib.xf_trainer_step_ingested(tr.h, lo, hi), t, tr, lambda: tr.step_ingested(0, rows))
        _refused(lambda: lib.xf_trainer_predict_ingested(tr.h, lo, hi, P(p), None), t, tr, step)
        _refused(lambda: lib.xf_trainer_predict_ingested_metric(tr.h, lo, hi, m, P(p), None), t, tr, step)
    _refused(lambda: lib.xf_trainer_predict_ingested_metric(tr.h, 0, rows, None, P(p), None), t, tr, step)
    lib.xf_metric_destroy(m)
    tr.close()
    t.close()

    # XF_MODEL_MVM: a field id of 32 is refused after the upload, before any kernel runs
    t = api.Table(latent_dim=8, optimizer=api.OPT_FTRL, capacity=1 << 16, seed=3, canonical_fm=1)
    tr = api.Trainer(t, model=api.MODEL_MVM, max_rows=64, max_nnz=512)
    fields = (np.arange(z) % 5).astype(np.uint8)
    bad = fields.copy()
    bad[z // 2] = 32

    def mvm_step():
        r, _, k, y = _small(next(seeds))
        tr.step_host_fields(r, k, (np.arange(k.size) % 7).astype(np.uint8), None, y)

    mvm_step()
    _refused(lambda: lib.xf_trainer_step_host_fields(tr.h, P(rp), P(keys), P(bad), None, P(lab), n, z, C.byref(mean)),
             t, tr, mvm_step)
    _refused(lambda: lib.xf_trainer_predict_host_fields(tr.h, P(rp), P(keys), P(bad), None, n, z, P(out)), t, tr, mvm_step)
    _refused(lambda: lib.xf_trainer_step_host_fields(tr.h, P(rp), P(keys), None, None, P(lab), n, z, C.byref(mean)),
             t, tr, mvm_step)
    tr.step_host_fields(rp, keys, fields, None, lab)
    assert tr.stats()["steps"] == 5
    tr.close()
    t.close()
