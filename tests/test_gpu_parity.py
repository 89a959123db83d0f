"""GPU parity tests (pytest -m gpu): the CUDA path, called through the C ABI, against
  (1) the golden vectors produced by the reference itself (tests/golden/*.npz),
  (2) the oracle on seeded random batches (per-step residuals, table state, predictions),
  (3) size-independent properties at BASELINE.json's full batch size.
Bit-exact where the work is integer (keys, bucketing, presence); within 1e-5 relative (abs floor
1e-7) for floats, the tolerance north_star states."""
import os

import numpy as np
import pytest

from cases import CASES
from common import (check_fm_first_step, assert_close, assert_close_noise_aware, data_prefixes, golden, oracle_case_run,
                    stored_rows)
from oracle import oracle as O
from xflow_b200 import api, datagen

pytestmark = pytest.mark.gpu


def _opt(name):
    return (api.OPT_FTRL, O.OPT_FTRL) if name == "ftrl" else (api.OPT_SGD, O.OPT_SGD)


def _gpu_train_predict(case, syn_data, capacity=0):
    c = CASES[case]
    g = golden(case)
    train, test = data_prefixes(case, syn_data)
    K = c["K"]
    gopt, _ = _opt(c["opt"])
    model = api.MODEL_LR if c["model"] == "lr" else api.MODEL_FM
    table = api.Table(latent_dim=K, optimizer=gopt, capacity=capacity,
                      v_init=api.VINIT_ZERO if c.get("preinit") else api.VINIT_DEFAULT)
    if c.get("preinit"):
        table.import_(g["keys"], w=g["init_w"], v=g["init_v"])
    tr = api.Trainer(table, model=model, max_rows=4096, max_nnz=4096 * 64)
    tr.init_push()
    block = c.get("block_mb", 2) << 20
    for _ in range(c["epochs"]):
        for rp, keys, lab in api.Loader(train + "-00000", block):
            tr.step_host(rp, keys, lab)
    labs, ps = [], []
    for rp, keys, lab in api.Loader(test + "-00000", (4 << 20) if c["model"] == "lr" else (2 << 20)):
        ps.append(tr.predict_host(rp, keys))
        labs.append(lab.astype(np.int32))
    e = table.export(g["keys"])
    return e, np.concatenate(labs), np.concatenate(ps), g, table, tr


@pytest.mark.parametrize("case", sorted(CASES))
def test_golden_case_matches_reference(case, syn_data):
    e, lab, p, g, table, tr = _gpu_train_predict(case, syn_data)
    assert np.array_equal(e["present"], g["present"])          # same key set (bit-exact hashing / insertion)
    if CASES[case]["data"] == "small":
        # few occurrences per key and batch: plain 1e-5 on every element
        for k in ("w", "nw", "zw", "v", "nv", "zv"):
            if k in g.files:
                assert_close(e[k], g[k], "%s.%s" % (case, k))
        # exact zeros of FTRL's L1 threshold must be zeros on both sides
        assert np.array_equal(e["w"] == 0.0, g["w"] == 0.0)
        assert_close(p, g["pred_pctr"], case + ".pctr", rel=2e-5, abs_floor=6e-7)  # reference prints 6 digits
    else:
        # Zipf ids: a few keys occur thousands of times per batch and the reference's own float32
        # summation order shows in its result; see assert_close_noise_aware
        x, _, xp = oracle_case_run(case, syn_data, exact=True)
        for k in ("w", "nw", "zw", "v", "nv", "zv"):
            if k in g.files:
                assert_close_noise_aware(stored_rows(e, g, k), g[k], stored_rows(x, g, k), "%s.%s" % (case, k),
                                         max_noisy_frac=0.02)
        # a single noisy hot key shows in every row that contains it: no bound on the noisy fraction
        assert_close_noise_aware(p, g["pred_pctr"], xp, case + ".pctr", rel=2e-5, abs_floor=6e-7,
                                 max_noisy_frac=1.0)
    assert np.array_equal(lab, g["pred_label"])
    m = api.auc_logloss(lab, p)
    noise_ll = noise_auc = 0.0
    if CASES[case]["data"] != "small":
        mx = O.auc_logloss(lab, xp)
        noise_ll = 8 * abs(mx["logloss"] - float(g["logloss"]))
        noise_auc = 8 * abs(mx["auc"] - float(g["auc"]))
    assert abs(m["logloss"] - float(g["logloss"])) <= 1e-5 * abs(float(g["logloss"])) + 6e-7 + noise_ll
    assert abs(m["auc"] - float(g["auc"])) <= 2e-5 + noise_auc


def test_golden_case_with_table_growth(syn_data):
    """Same result when the table starts tiny and has to rehash several times."""
    case = "syn_fm_ftrl_k8_e1"
    e, lab, p, g, table, tr = _gpu_train_predict(case, syn_data, capacity=1024)
    assert table.capacity() >= 2 * g["keys"].size
    x, _, _ = oracle_case_run(case, syn_data, exact=True)
    for k in ("w", "nw", "zw", "v", "nv", "zv"):
        assert_close_noise_aware(stored_rows(e, g, k), g[k], stored_rows(x, g, k), "growth.%s" % k, max_noisy_frac=0.02)


@pytest.mark.parametrize("model,opt,K", [("lr", "ftrl", 0), ("lr", "sgd", 0), ("fm", "sgd", 8), ("fm", "ftrl", 16),
                                         ("fm", "ftrl", 10), ("fm", "sgd", 3)])
@pytest.mark.parametrize("dist", ["uniform", "zipf"])
def test_random_batches_match_oracle(model, opt, K, dist):
    """Several steps on seeded batches: per-row residuals and the whole table after every step."""
    gopt, oopt = _opt(opt)
    B, d, space = 2048, 24, 30000
    gt = api.Table(latent_dim=K, optimizer=gopt, v_init=api.VINIT_COUNTER, seed=11)
    ot = O.Table(K=K, opt=oopt, init_mode=O.INIT_COUNTER, seed=11)
    xt = O.Table(K=K, opt=oopt, init_mode=O.INIT_COUNTER, seed=11)  # double-accumulating yardstick
    tr = api.Trainer(gt, model=api.MODEL_LR if model == "lr" else api.MODEL_FM, max_rows=B, max_nnz=B * d * 2,
                     keep_loss=True)
    tr.init_push()
    ot.init_push()
    xt.init_push()
    all_keys = [np.zeros(1, np.uint64)]
    for step in range(4):
        rp, keys, lab = datagen.make_csr_keys(100 + step, B, d, space, api.hash_decimal_ids, dist=dist,
                                              zipf_s=1.3, ragged=(step == 2))
        mean_abs = tr.step_host(rp, keys, lab)
        gl = tr.get_loss(B)
        U, ol = ot.step(rp.astype(np.int64), keys, lab.astype(np.int32))
        with O.exact_sums():
            xt.step(rp.astype(np.int64), keys, lab.astype(np.int32))
        all_keys.append(keys)
        uk = np.unique(np.concatenate(all_keys))
        ge, oe, xe = gt.export(uk), ot.export(uk), xt.export(uk)
        assert np.array_equal(ge["present"], oe["present"])
        if dist == "uniform":
            assert_close(gl, ol, "loss step %d" % step, abs_floor=1e-6)
            assert abs(mean_abs - np.abs(ol).mean()) < 1e-5
            for k in ("w", "nw", "zw") + (("v", "nv", "zv") if K else ()):
                assert_close(ge[k], oe[k], "%s step %d" % (k, step))
        else:
            for k in ("w", "nw", "zw") + (("v", "nv", "zv") if K else ()):
                # every accumulator (G, and the factorised latent-gradient sums L, Aq) is f64: what is left
                # is the reference's own float32 summation-order noise on hot keys
                assert_close_noise_aware(ge[k], oe[k], xe[k], "%s step %d" % (k, step), rel=1e-5, max_noisy_frac=0.02)
        assert tr.stats()["unique_keys"] >= U
    st = tr.stats()
    assert st["steps"] == 4 and st["rows"] == 4 * B
    # forward-only path on a fresh batch
    rp, keys, lab = datagen.make_csr_keys(999, B, d, space, api.hash_decimal_ids, dist=dist)
    if dist == "uniform":
        assert_close(tr.predict_host(rp, keys), ot.predict(rp.astype(np.int64), keys), "pctr", abs_floor=1e-6)
    else:
        assert_close_noise_aware(tr.predict_host(rp, keys), ot.predict(rp.astype(np.int64), keys),
                                 xt.predict(rp.astype(np.int64), keys), "pctr", abs_floor=1e-6, max_noisy_frac=0.2)
    assert gt.size() == ot.size()


def test_unique_key_count_is_exact():
    B, d = 4096, 32
    gt = api.Table()
    tr = api.Trainer(gt, max_rows=B, max_nnz=B * d)
    total = 0
    for s in range(3):
        rp, keys, lab = datagen.make_csr_keys(s, B, d, 5000, api.hash_decimal_ids, dist="zipf", zipf_s=1.1)
        tr.step_host(rp, keys, lab)
        total += np.unique(keys).size
    assert tr.stats()["unique_keys"] == total


@pytest.mark.parametrize("opt,K", [("ftrl", 0), ("sgd", 0), ("ftrl", 8), ("sgd", 10)])
def test_pull_push_api_matches_oracle(opt, K):
    """The KVWorker::Pull/Push-shaped entry points against the FTRL/SGD handles of the oracle."""
    gopt, oopt = _opt(opt)
    gt = api.Table(latent_dim=K, optimizer=gopt, v_init=api.VINIT_COUNTER, seed=3, capacity=1024)
    ot = O.Table(K=K, opt=oopt, init_mode=O.INIT_COUNTER, seed=3)
    rng = np.random.default_rng(0)
    universe = rng.integers(0, 2 ** 64, 20000, dtype=np.uint64)
    for it in range(5):
        keys = np.unique(rng.choice(universe, 3000))
        gw, gv = gt.pull(keys)
        ow, ov = ot.pull(keys)
        assert np.array_equal(gw.view(np.uint32), ow.view(np.uint32)) if it == 0 else True
        assert_close(gw, ow, "pull w")
        if K:
            assert_close(gv, ov, "pull v")
        g1 = (rng.standard_normal(keys.size) * 0.1).astype(np.float32)
        g2 = (rng.standard_normal((keys.size, K)) * 0.1).astype(np.float32) if K else None
        g1[::7] = 0.0
        gt.push(keys, g1, g2)
        ot.push(keys, g1, g2)
    e, o = gt.export(universe), ot.export(universe)
    assert np.array_equal(e["present"], o["present"])
    for k in ("w", "nw", "zw") + (("v", "nv", "zv") if K else ()):
        # same inputs, same op order: the optimizer arithmetic itself is bit-exact
        assert np.array_equal(e[k].view(np.uint32), o[k].view(np.uint32)), k
    assert gt.size() == ot.size() == int(o["present"].sum())


def test_counter_init_bit_exact_and_insert_on_pull():
    gt = api.Table(latent_dim=16, optimizer=api.OPT_FTRL, seed=42)
    ot = O.Table(K=16, opt=O.OPT_FTRL, seed=42)
    keys = np.arange(1, 5001, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    gw, gv = gt.pull(keys)
    ow, ov = ot.pull(keys)
    assert np.array_equal(gv.view(np.uint32), ov.view(np.uint32))
    assert not gw.any() and gt.size() == 5000
    e = gt.export(keys[:10])
    assert e["present"].all()
    assert not gt.export(np.array([12345], np.uint64))["present"].any()  # export never inserts
    assert gt.size() == 5000


def test_save_load_roundtrip(tmp_path):
    gt = api.Table(latent_dim=8, optimizer=api.OPT_FTRL, seed=1)
    tr = api.Trainer(gt, model=api.MODEL_FM, max_rows=1024, max_nnz=1024 * 16)
    for s in range(3):
        tr.step_host(*datagen.make_csr_keys(s, 1024, 16, 4000, api.hash_decimal_ids))
    keys = np.sort(gt.list_keys())
    assert keys.size == gt.size()
    a = gt.export(keys)
    path = str(tmp_path / "ckpt.bin")
    gt.save(path)
    g2 = api.Table(latent_dim=8, optimizer=api.OPT_FTRL, seed=99, v_init=api.VINIT_ZERO)
    g2.load(path)
    b = g2.export(keys)
    for k in ("w", "nw", "zw", "v", "nv", "zv", "present"):
        assert np.array_equal(a[k], b[k]), k
    assert g2.size() == gt.size()


def test_empty_and_degenerate_batches():
    gt = api.Table()
    ot = O.Table()
    tr = api.Trainer(gt, max_rows=64, max_nnz=4096, keep_loss=True)
    # rows without tokens, a row with one key repeated, a long row (> 128 tokens)
    lens = [0, 3, 0, 200, 1, 40]
    rp = np.zeros(len(lens) + 1, np.uint32)
    rp[1:] = np.cumsum(lens)
    ids = np.concatenate([np.array([7, 7, 7], np.uint64), np.arange(200, dtype=np.uint64) % 50,
                          np.array([7], np.uint64), np.arange(40, dtype=np.uint64)])
    keys = api.hash_decimal_ids(ids)
    lab = np.array([1, 0, 0, 1, 1, 0], np.uint8)
    for _ in range(3):
        tr.step_host(rp, keys, lab)
        gl = tr.get_loss(len(lens))
        _, ol = ot.step(rp.astype(np.int64), keys, lab.astype(np.int32))
        assert_close(gl, ol, "loss", abs_floor=1e-6)
    uk = np.unique(keys)
    ge, oe = gt.export(uk), ot.export(uk)
    for k in ("w", "nw", "zw"):
        assert_close(ge[k], oe[k], k)
    assert tr.step_host(np.zeros(1, np.uint32), np.zeros(0, np.uint64), np.zeros(0, np.uint8)) == 0.0


def test_full_size_batch_properties():
    """BASELINE configs[1] shape (B = 65536, 64 nnz/row, 1e7 ids): properties that need no oracle run."""
    B, d, space = 65536, 64, 10 ** 7
    gt = api.Table(capacity=1 << 24)
    tr = api.Trainer(gt, max_rows=B, max_nnz=B * d, keep_loss=True)
    rp, keys, lab = datagen.make_csr_keys(1, B, d, space, api.hash_decimal_ids)
    tr.step_host(rp, keys, lab)
    loss = tr.get_loss(B)
    # first step from an all-zero table: pctr = sigmoid(0) = 0.5 exactly
    assert np.array_equal(loss, np.float32(0.5) - lab.astype(np.float32))
    uk, cnt = np.unique(keys, return_counts=True)
    assert tr.stats()["unique_keys"] == uk.size == gt.size()
    # closed form of the first FTRL step: g = sum(residual over occurrences)/B, n = g^2, z = g
    occ_row = np.repeat(np.arange(B), d)
    g_sum = np.zeros(uk.size, np.float64)
    np.add.at(g_sum, np.searchsorted(uk, keys), loss[occ_row].astype(np.float64))
    e = gt.export(uk)
    g32 = (g_sum / B).astype(np.float32)
    assert_close(e["zw"], g32, "z after step 1", rel=2e-6)
    assert_close(e["nw"], g32.astype(np.float64) ** 2, "n after step 1", rel=4e-6, abs_floor=1e-12)
    # idempotence of pulls and sortedness-independence: permuting tokens inside rows changes nothing
    gt2 = api.Table(capacity=1 << 24)
    tr2 = api.Trainer(gt2, max_rows=B, max_nnz=B * d)
    perm = np.arange(keys.size).reshape(B, d)[:, ::-1].reshape(-1)
    tr2.step_host(rp, keys[perm], lab)
    e2 = gt2.export(uk)
    assert_close(e2["w"], e["w"], "w under token permutation", rel=2e-6)
    # a second, identical batch: every key already present -> size unchanged, unique count doubles
    tr.step_host(rp, keys, lab)
    assert gt.size() == uk.size and tr.stats()["unique_keys"] == 2 * uk.size


def test_full_size_fm_batch_properties():
    """cfg5 shape (B = 65536, 64 nnz/row, Zipf(1.05) ids in 1e8, K = 16, FTRL): the first step in closed form
    (common.check_fm_first_step, float64 numpy; the CPU suite pins the same checker to the oracle).
    Exercises the hot-key path (one key holds ~8 % of the tokens) and the factorised latent gradient
    gv = Aq - v L at full size."""
    B, d, space, K = 65536, 64, 10 ** 8, 16
    gt = api.Table(latent_dim=K, capacity=1 << 23, v_init=api.VINIT_COUNTER, seed=3)
    tr = api.Trainer(gt, model=api.MODEL_FM, max_rows=B, max_nnz=B * d, keep_loss=True)
    rp, keys, lab = datagen.make_csr_keys(2, B, d, space, api.hash_decimal_ids, dist="zipf")
    uk, cnt = np.unique(keys, return_counts=True)
    assert cnt.max() > 0.03 * keys.size          # there is a genuinely hot key
    w0, v0 = gt.pull(uk)                         # insert-on-pull; v = counter-based initial values
    assert not w0.any() and gt.size() == uk.size
    tr.step_host(rp, keys, lab)
    loss = tr.get_loss(B)
    assert tr.stats()["unique_keys"] == uk.size == gt.size()
    _, e = check_fm_first_step(rp, keys, lab, K, lambda k: v0, loss, gt.export)
    # token order inside rows changes nothing (beyond the float32 rounding of the row sums)
    gt2 = api.Table(latent_dim=K, capacity=1 << 23, v_init=api.VINIT_COUNTER, seed=3)
    tr2 = api.Trainer(gt2, model=api.MODEL_FM, max_rows=B, max_nnz=B * d, keep_loss=True)
    perm = np.arange(keys.size).reshape(B, d)[:, ::-1].reshape(-1)
    tr2.step_host(rp, keys[perm], lab)
    check_fm_first_step(rp, keys[perm], lab, K, lambda k: v0, tr2.get_loss(B), gt2.export)


def test_device_id_hashing_is_bit_exact_and_ids_path_trains_identically():
    """ingest.cu: keys made on the device from u32 ids == std::hash of the decimal strings; the ids entry
    point leaves the same table as the keys entry point."""
    import torch
    rng = np.random.default_rng(7)
    ids = rng.integers(0, 2 ** 32, 200000, dtype=np.uint64).astype(np.uint32)
    ids[:6] = [0, 9, 10, 99, 100, 4294967295]
    d_ids = torch.from_numpy(ids.view(np.int32)).cuda()
    d_keys = torch.empty(ids.size, dtype=torch.int64, device="cuda")
    assert api.lib().xf_hash_decimal_ids_device(d_ids.data_ptr(), ids.size, d_keys.data_ptr(), None) == 0
    torch.cuda.synchronize()
    got = d_keys.cpu().numpy().view(np.uint64)
    assert np.array_equal(got, O.hash_decimal_ids(ids.astype(np.uint64)))
    assert int(got[5]) == O.std_hash(b"4294967295")

    B, d = 4096, 32
    rp, idv, lab = datagen.make_ids(3, B, d, 50000)
    keys = api.hash_decimal_ids(idv)
    ta, tb = api.Table(), api.Table()
    tra, trb = api.Trainer(ta, max_rows=B, max_nnz=B * d), api.Trainer(tb, max_rows=B, max_nnz=B * d)
    pin = [torch.from_numpy(a.view(np.uint8)).pin_memory() for a in (rp, idv.astype(np.uint32), lab)]
    for _ in range(3):
        tra.step_host(rp, keys, lab)
        trb.step_host_ids_async(pin[0].data_ptr(), pin[1].data_ptr(), pin[2].data_ptr(), B, B * d)
    trb.sync()
    uk = np.unique(keys)
    a, b = ta.export(uk), tb.export(uk)
    for k in ("w", "nw", "zw", "present"):
        assert np.array_equal(a[k], b[k]), k


FULL = {
    # BASELINE.json configs[1], configs[2] and the shape of configs[4], at the full batch size
    "cfg2": dict(model="lr", opt="ftrl", K=0, space=10 ** 7, d=64, dist="uniform", steps=3),
    "cfg3": dict(model="fm", opt="sgd", K=8, space=10 ** 7, d=64, dist="uniform", steps=2),
    "cfg5": dict(model="fm", opt="ftrl", K=16, space=10 ** 8, d=100, dist="zipf", steps=2),
}


@pytest.mark.parametrize("name", sorted(FULL))
def test_full_batch_multi_step_matches_oracle(name):
    """Several steps at B = 65 536 against the ORACLE itself (not closed forms): every row's residual at
    every step and the whole optimizer state of every touched key at the end."""
    c = FULL[name]
    B, d, K = 65536, c["d"], c["K"]
    gopt, oopt = _opt(c["opt"])
    gt = api.Table(latent_dim=K, optimizer=gopt, v_init=api.VINIT_COUNTER, seed=21, capacity=1 << 23)
    ot = O.Table(K=K, opt=oopt, init_mode=O.INIT_COUNTER, seed=21)
    skew = c["dist"] == "zipf"
    xt = O.Table(K=K, opt=oopt, init_mode=O.INIT_COUNTER, seed=21) if skew else None
    tr = api.Trainer(gt, model=api.MODEL_LR if c["model"] == "lr" else api.MODEL_FM, max_rows=B, max_nnz=B * d,
                     keep_loss=True)
    tr.init_push(); ot.init_push()
    if xt:
        xt.init_push()
    seen = [np.zeros(1, np.uint64)]
    for step in range(c["steps"]):
        rp, keys, lab = datagen.make_csr_keys(40 + step, B, d, c["space"], api.hash_decimal_ids, dist=c["dist"])
        tr.step_host(rp, keys, lab)
        gl = tr.get_loss(B)
        _, ol = ot.step(rp.astype(np.int64), keys, lab.astype(np.int32))
        if xt:
            with O.exact_sums():
                _, xl = xt.step(rp.astype(np.int64), keys, lab.astype(np.int32))
            assert_close_noise_aware(gl, ol, xl, "%s loss step %d" % (name, step), abs_floor=1e-6, max_noisy_frac=1.0)
        else:
            assert_close(gl, ol, "%s loss step %d" % (name, step), abs_floor=1e-6)
        seen.append(keys)
    uk = np.unique(np.concatenate(seen))
    ge, oe = gt.export(uk), ot.export(uk)
    assert np.array_equal(ge["present"], oe["present"]) and gt.size() == ot.size()
    xe = xt.export(uk) if xt else None
    for k in ("w", "nw", "zw") + (("v", "nv", "zv") if K else ()):
        if xt:
            assert_close_noise_aware(ge[k], oe[k], xe[k], "%s %s" % (name, k), max_noisy_frac=0.02)
        else:
            assert_close(ge[k], oe[k], "%s %s" % (name, k))


def test_lazy_sequence_ring_restarts(monkeypatch):
    """Lazy LR tables number their batches in a fixed ring (rows_by_seq); when it is used up one sweep folds
    every pending step in and the numbering restarts.  With a 5-entry ring, 14 steps cross that point 3 times."""
    monkeypatch.setenv("XFLOW_SEQ_RING", "5")
    B, d = 1024, 16
    gt = api.Table(optimizer=api.OPT_FTRL)
    ot = O.Table(K=0, opt=O.OPT_FTRL)
    tr = api.Trainer(gt, max_rows=B, max_nnz=B * d * 2, keep_loss=True)
    seen = []
    for step in range(14):
        rows = B if step % 3 else B // 2          # the divisor of a pending step is ITS batch's row count
        rp, keys, lab = datagen.make_csr_keys(300 + step, rows, d, 6000, api.hash_decimal_ids, ragged=(step % 4 == 1))
        tr.step_host(rp, keys, lab)
        _, ol = ot.step(rp.astype(np.int64), keys, lab.astype(np.int32))
        assert_close(tr.get_loss(rows), ol, "loss step %d" % step, abs_floor=1e-6)
        seen.append(keys)
        if step in (4, 9, 13):
            uk = np.unique(np.concatenate(seen))
            ge, oe = gt.export(uk), ot.export(uk)
            for k in ("w", "nw", "zw"):
                assert_close(ge[k], oe[k], "%s after step %d" % (k, step))


def test_lazy_protocol_under_contention_equals_eager(monkeypatch):
    """The one-kernel LR step (claim with a CAS on the tag, publish with one 256-bit store, readers poll the tag)
    under heavy contention — 48 distinct keys, 260 000 tokens per batch, every row holds duplicates — against the
    two-kernel path that has no such protocol (XFLOW_EAGER=1) and against the oracle run with exact sums."""
    B, d = 8192, 32
    lazy = api.Table(optimizer=api.OPT_FTRL)
    monkeypatch.setenv("XFLOW_EAGER", "1")
    eager = api.Table(optimizer=api.OPT_FTRL)
    monkeypatch.delenv("XFLOW_EAGER")
    xt = O.Table(K=0, opt=O.OPT_FTRL)
    tl = api.Trainer(lazy, max_rows=B, max_nnz=B * d, keep_loss=True)
    te = api.Trainer(eager, max_rows=B, max_nnz=B * d, keep_loss=True)
    for step in range(6):
        rp, keys, lab = datagen.make_csr_keys(900 + step, B, d, 48, api.hash_decimal_ids)
        tl.step_host(rp, keys, lab)
        te.step_host(rp, keys, lab)
        with O.exact_sums():
            _, xl = xt.step(rp.astype(np.int64), keys, lab.astype(np.int32))
        a, b = tl.get_loss(B), te.get_loss(B)
        # both sum a key's ~5400 residuals exactly (64-bit fixed point / double): they agree to the last bits
        assert_close(a, b, "lazy vs eager residuals, step %d" % step, rel=2e-6, abs_floor=2e-7)
        assert_close(a, xl, "residual vs exact-sum oracle, step %d" % step, rel=2e-5, abs_floor=2e-6)
    uk = np.unique(api.hash_decimal_ids(np.arange(48, dtype=np.uint64)))
    la, ea = lazy.export(uk), eager.export(uk)
    for k in ("w", "nw", "zw"):
        assert_close(la[k], ea[k], k, rel=2e-6, abs_floor=1e-9)
    # and the lazy path is bit-reproducible: integer sums do not depend on the order the atomics land in
    lazy2 = api.Table(optimizer=api.OPT_FTRL)
    t2 = api.Trainer(lazy2, max_rows=B, max_nnz=B * d)
    for step in range(6):
        t2.step_host(*datagen.make_csr_keys(900 + step, B, d, 48, api.hash_decimal_ids))
    lb = lazy2.export(uk)
    for k in ("w", "nw", "zw"):
        assert np.array_equal(la[k].view(np.uint32), lb[k].view(np.uint32)), k


def test_checkpoint_rejects_corrupt_files(tmp_path):
    gt = api.Table(latent_dim=4, optimizer=api.OPT_FTRL, seed=1)
    tr = api.Trainer(gt, model=api.MODEL_FM, max_rows=256, max_nnz=256 * 8)
    tr.step_host(*datagen.make_csr_keys(1, 256, 8, 900, api.hash_decimal_ids))
    path = str(tmp_path / "ckpt.bin")
    gt.save(path)
    assert not os.path.exists(path + ".tmp")
    blob = open(path, "rb").read()
    g2 = api.Table(latent_dim=4, optimizer=api.OPT_FTRL)
    for bad in (blob[: len(blob) // 2], blob[:12] + (2 ** 60).to_bytes(8, "little")[:4] + blob[16:], blob + b"xx"):
        open(path, "wb").write(bad)
        with pytest.raises(api.XflowError):
            g2.load(path)
    with pytest.raises(api.XflowError):
        gt.save(str(tmp_path / "no_such_dir" / "x.bin"))


def test_device_metric_matches_host_metric():
    """metric.cu: sort + rank sums on the device against the host implementations of Base::calculate_auc
    (base.h:84-110, float quirks) and of the exact metric; many ties, both classes, and a one-class case."""
    import ctypes as C
    import torch
    rng = np.random.default_rng(5)
    n = 50000
    p = np.round(rng.random(n), 3).astype(np.float32).clip(1e-4, 1 - 1e-4)   # 1000 distinct values: heavy ties
    y = (rng.random(n) < p).astype(np.uint8)
    lib = api.lib()
    m = C.c_void_p()
    assert lib.xf_metric_create(C.byref(m), 0) == 0
    d_p, d_y = torch.from_numpy(p).cuda(), torch.from_numpy(y).cuda()
    torch.cuda.synchronize()
    for lo, hi in ((0, 17000), (17000, 17001), (17001, n)):                   # appended block by block
        assert lib.xf_metric_add_device(m, C.c_void_p(d_p.data_ptr() + 4 * lo), C.c_void_p(d_y.data_ptr() + lo), hi - lo, None) == 0
    out = (C.c_double * 6)()
    assert lib.xf_metric_finish(m, None, out) == 0, lib.xf_last_error()
    ex = api.auc_logloss_exact(y.astype(np.int32), p)
    assert out[2] == ex["positives"] and out[3] == ex["negatives"]
    assert abs(out[4] - ex["logloss"]) <= 1e-9 * abs(ex["logloss"])
    assert abs(out[5] - ex["auc"]) <= 1e-12
    # the reference-style numbers: same definitions, float accumulators on the host; ties make the reference's AUC
    # depend on its sort's tie order, so compare on data without ties across classes
    q = (np.arange(n, dtype=np.float32) + 1) / (n + 1)
    rng.shuffle(q)
    d_q = torch.from_numpy(q).cuda()
    torch.cuda.synchronize()
    assert lib.xf_metric_reset(m) == 0
    assert lib.xf_metric_add_device(m, C.c_void_p(d_q.data_ptr()), C.c_void_p(d_y.data_ptr()), n, None) == 0
    assert lib.xf_metric_finish(m, None, out) == 0
    ref = api.auc_logloss(y.astype(np.int32), q)
    assert abs(out[0] - ref["logloss"]) <= 2e-5 * abs(ref["logloss"])      # the host accumulates in a float
    assert abs(out[1] - ref["auc"]) <= 2e-5
    # one class only: no AUC
    assert lib.xf_metric_reset(m) == 0
    d_z = torch.zeros(n, dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    assert lib.xf_metric_add_device(m, C.c_void_p(d_q.data_ptr()), C.c_void_p(d_z.data_ptr()), n, None) == 0
    assert lib.xf_metric_finish(m, None, out) == 0
    assert out[2] == 0 and np.isnan(out[1]) and np.isnan(out[5])
    lib.xf_metric_destroy(m)


def _ftrl64(g, w, n, z, alpha=0.05, beta=1.0, l1=5e-5, l2=10.0):
    n2 = n + g * g
    z2 = z + g - (np.sqrt(n2) - np.sqrt(n)) / alpha * w
    w2 = np.where(np.abs(z2) <= l1, 0.0, (z2 - np.sign(z2) * l1) / -((beta + np.sqrt(n2)) / alpha + l2))
    return w2, n2, z2


@pytest.mark.parametrize("K,opt", [(8, "ftrl"), (16, "sgd"), (4, "ftrl")])
def test_canonical_fm_with_values_matches_float64_model(K, opt):
    """XF_MODEL_FM_CANONICAL (step_fmc.cu; SURVEY 8f-4, NOT the reference's model): the textbook FM with feature
    values, y = sum w x + 1/2 sum_k[(sum v_k x)^2 - sum (v_k x)^2], against a float64 numpy model of the same
    definition (forward, gradients / rows, FTRL or SGD step per touched key) over three steps."""
    gopt, _ = _opt(opt)
    B, d, space = 512, 12, 3000
    t = api.Table(latent_dim=K, optimizer=gopt, v_init=api.VINIT_COUNTER, seed=4, canonical_fm=1)
    tr = api.Trainer(t, model=api.MODEL_FM_CANONICAL, max_rows=B, max_nnz=B * d * 2, keep_loss=True)
    rng = np.random.default_rng(K)
    state = {}

    def rows_of(uk):
        for k in uk:
            if int(k) not in state:
                state[int(k)] = None
        new = np.array([k for k in uk if state[int(k)] is None], np.uint64)
        if new.size:
            w0, v0 = t.pull(new)                       # insert-on-pull: default w, counter-based v
            for k, a, b in zip(new, w0, v0):
                state[int(k)] = [float(a), 0.0, 0.0, b.astype(np.float64), np.zeros(K), np.zeros(K)]

    for step in range(3):
        rp, keys, lab = datagen.make_csr_keys(70 + step, B, d, space, api.hash_decimal_ids, ragged=(step == 1))
        x = (rng.random(keys.size) * 1.5 + 0.25).astype(np.float32)
        x[::7] *= -1.0
        uk, inv = np.unique(keys, return_inverse=True)
        rows_of(uk)
        W = np.array([state[int(k)][0] for k in uk]); V = np.stack([state[int(k)][3] for k in uk])
        row_of = np.repeat(np.arange(B), np.diff(rp).astype(np.int64))
        x64 = x.astype(np.float64)
        wx = np.zeros(B); np.add.at(wx, row_of, W[inv] * x64)
        S = np.zeros((B, K)); np.add.at(S, row_of, V[inv] * x64[:, None])
        Q = np.zeros(B); np.add.at(Q, row_of, ((V[inv] * x64[:, None]) ** 2).sum(1))
        y = wx + 0.5 * ((S ** 2).sum(1) - Q)
        p = np.where(y < -30, 1e-6, np.where(y > 30, 1.0, np.power(2.718281828, y) / (1 + np.power(2.718281828, y))))
        loss = p - lab
        tr.step_host_values(rp, keys, x, lab)
        assert_close(tr.get_loss(B), loss, "canonical FM residuals, step %d" % step, rel=2e-5, abs_floor=2e-6)
        r = loss[row_of] * x64
        gw = np.zeros(uk.size); np.add.at(gw, inv, r)
        A = np.zeros((uk.size, K)); np.add.at(A, inv, r[:, None] * S[row_of])
        L2 = np.zeros(uk.size); np.add.at(L2, inv, r * x64)
        gv = (A - V * L2[:, None]) / B
        gw = gw / B
        for i, k in enumerate(uk):
            s = state[int(k)]
            if opt == "ftrl":
                s[0], s[1], s[2] = _ftrl64(gw[i], s[0], s[1], s[2])
                s[3], s[4], s[5] = _ftrl64(gv[i], s[3], s[4], s[5])
            else:
                s[0] -= 1e-3 * gw[i]
                s[3] = s[3] - 1e-3 * gv[i]
    allk = np.array(sorted(state), np.uint64)
    e = t.export(allk)
    ref = {k: np.array([np.atleast_1d(state[int(q)][j]) for q in allk]).reshape(allk.size, -1)
           for j, k in enumerate(("w", "nw", "zw", "v", "nv", "zv"))}
    for k in ("w", "v") + (("nw", "zw", "nv", "zv") if opt == "ftrl" else ()):
        assert_close(e[k].reshape(allk.size, -1), ref[k], "canonical FM %s" % k, rel=2e-4, abs_floor=2e-7)
    # forward only, with values
    rp, keys, lab = datagen.make_csr_keys(99, B, d, space, api.hash_decimal_ids)
    x = (rng.random(keys.size) + 0.5).astype(np.float32)
    got = tr.predict_host_values(rp, keys, x)
    assert np.isfinite(got).all() and got.min() >= 0 and got.max() <= 1
    # a canonical table refuses the reference-shaped models and vice versa
    with pytest.raises(api.XflowError):
        api.Trainer(t, model=api.MODEL_FM, max_rows=B, max_nnz=B * d)


@pytest.mark.parametrize("K,opt,with_vals", [(8, "sgd", True), (16, "ftrl", True), (4, "ftrl", False), (32, "sgd", False)])
def test_defined_mvm_matches_float64_model(K, opt, with_vals):
    """XF_MODEL_MVM (step_mvm.cu; SURVEY 8f-4): y = sum_k prod_{fields present} (sum_{tokens of the field} v_k x),
    gradient of a token = residual * x * product of the OTHER fields' sums, one FTRL / SGD step per touched key on v —
    against a float64 numpy model of that definition over three steps (the reference's MVMWorker reads past its
    buffers and has no defined output to compare with, DESIGN.md section 8)."""
    gopt, _ = _opt(opt)
    B, d, space, F = 384, 9, 2500, 5
    lr = 20.0                                                  # SGD: large enough for the steps to show in float32
    t = api.Table(latent_dim=K, optimizer=gopt, v_init=api.VINIT_COUNTER, seed=4, canonical_fm=1, learning_rate=lr)
    tr = api.Trainer(t, model=api.MODEL_MVM, max_rows=B, max_nnz=B * d * 2, keep_loss=True)
    rng = np.random.default_rng(100 + K)
    batches = []
    for step in range(3):
        rp, keys, lab = datagen.make_csr_keys(170 + step, B, d, space, api.hash_decimal_ids, ragged=(step == 1))
        fields = rng.integers(0, F, keys.size).astype(np.uint8)
        if step == 2:
            fields[: keys.size // 3] = 31                     # the largest admissible field id
        x = (rng.random(keys.size) * 1.5 + 0.25).astype(np.float32) if with_vals else None
        if x is not None:
            x[::5] *= -1.0
        batches.append((rp, keys, fields, x, lab))
    allk = np.unique(np.concatenate([b[1] for b in batches]))
    V0 = rng.normal(0.0, 0.6, (allk.size, K)).astype(np.float32)
    t.import_(allk, v=V0)
    V = V0.astype(np.float64); NV = np.zeros_like(V); ZV = np.zeros_like(V)
    for step, (rp, keys, fields, x, lab) in enumerate(batches):
        idx = np.searchsorted(allk, keys)
        row_of = np.repeat(np.arange(B), np.diff(rp).astype(np.int64))
        x64 = np.ones(keys.size) if x is None else x.astype(np.float64)
        S = np.zeros((B, 32, K)); np.add.at(S, (row_of, fields.astype(np.int64)), V[idx] * x64[:, None])
        present = np.zeros((B, 32), bool); present[row_of, fields.astype(np.int64)] = True
        Sp = np.where(present[:, :, None], S, 1.0)
        y = np.where(present.any(1), Sp.prod(1).sum(1), 0.0)
        p = np.where(y < -30, 1e-6, np.where(y > 30, 1.0, np.power(2.718281828, y) / (1 + np.power(2.718281828, y))))
        loss = p - lab
        tr.step_host_fields(rp, keys, fields, x, lab)
        assert_close(tr.get_loss(B), loss, "MVM residuals, step %d" % step, rel=5e-5, abs_floor=5e-6)
        # product over the other fields of the row, per token
        excl = np.ones((keys.size, K))
        for f in range(32):
            other = present[row_of, f] & (fields != f)
            excl[other] *= S[row_of[other], f]
        gtok = loss[row_of, None] * x64[:, None] * excl
        A = np.zeros_like(V); np.add.at(A, idx, gtok)
        touched = np.zeros(allk.size, bool); touched[idx] = True
        g = A / B
        for i in np.nonzero(touched)[0]:
            if opt == "ftrl":
                V[i], NV[i], ZV[i] = _ftrl64(g[i], V[i], NV[i], ZV[i])
            else:
                V[i] = V[i] - lr * g[i]
    e = t.export(allk)
    assert e["present"].all()
    if opt == "ftrl":
        for name, ref in (("v", V), ("nv", NV), ("zv", ZV)):
            assert_close(e[name].reshape(allk.size, -1), ref, "MVM %s" % name, rel=5e-4, abs_floor=5e-7)
    else:
        # what the steps moved, not the (much larger) starting values
        moved = np.abs(V - V0).max()
        assert moved > 1e-3
        assert_close(e["v"].reshape(allk.size, -1) - V0, V - V0, "MVM v - v0", rel=2e-3, abs_floor=2e-6 + 1e-4 * moved)
    assert not e["w"].any()                                    # no linear term: w is never moved
    # forward only
    rp, keys, fields, x, lab = batches[0]
    got = tr.predict_host_fields(rp, keys, fields, x)
    assert np.isfinite(got).all() and got.min() >= 0 and got.max() <= 1
    # field ids the kernel has no room for are refused, and the model needs its field ids
    bad = fields.copy(); bad[0] = 32
    with pytest.raises(api.XflowError):
        tr.step_host_fields(rp, keys, bad, x, lab)
    with pytest.raises(api.XflowError):
        tr.step_host(rp, keys, lab)


def test_push_refuses_repeated_keys():
    """KVWorker::Push takes unique keys; a repeated key would be two unordered updates of one row.  The host
    entry point refuses it (sorted or not) before anything is applied."""
    t = api.Table(latent_dim=0, optimizer=api.OPT_FTRL, capacity=1 << 12)
    keys = np.array([5, 9, 11], np.uint64)
    t.push(keys, gw=np.ones(3, np.float32))
    before = t.export(keys)
    for bad in (np.array([5, 9, 9, 11], np.uint64), np.array([11, 5, 9, 5], np.uint64)):
        rc = api.lib().xf_table_push(t.h, bad.ctypes.data_as(api.C.c_void_p), bad.size,
                                     np.ones(bad.size, np.float32).ctypes.data_as(api.C.c_void_p), None)
        assert rc != 0 and b"more than once" in api.lib().xf_last_error()
    after = t.export(keys)
    for k in ("w", "nw", "zw"):
        assert np.array_equal(before[k], after[k])
    t.push(np.array([11, 5, 9], np.uint64), gw=np.ones(3, np.float32))      # unsorted but unique: fine
    t.close()
