"""One-GPU parity at the shapes and switches the step and update kernels branch on (pytest -m gpu):

  A  reference-shaped FM at every latent-width branch of step.cu / kernels.cu (VEC 1/2/4, the 256-bit loads,
     more than 32 latent chunks per row, K up to 1024), on rows of 0 to 600 tokens, and the Pull / Push API
  B  LR, lazy and eager, FTRL and SGD, with every probing-bucket size, on a table that grows while rows hold
     pending steps and imported weights
  C  checkpoints of lazy LR tables with pending steps: a loaded table continues bit for bit
  D  the canonical FM and the multi-view machine at every accepted width, their predictions value by value
  E  the kernel switches read once per process (XFLOW_UPDATE_WIDE, XFLOW_FM_CACHE_LOG2), in child processes
  F  the sharded step on a one-rank communicator, and table pre-population from decimal ids

The yardsticks are the oracle (oracle.Table, the CPU restatement of the reference) and float64 models of the
canonical FM and the MVM (tests/common.py).  Tolerances are those of tests/common.py: 1e-5 relative with an
absolute floor of 1e-7 on table state, 1e-6 on residuals; FTRL's exact zeros agree exactly."""
import os
import subprocess
import sys

import numpy as np
import pytest

from common import (CanonicalFM64, assert_close, assert_close_noise_aware, bits_equal,
                    canonical_fm_forward64, mvm_forward64)
from oracle import oracle as O
from xflow_b200 import api

pytestmark = pytest.mark.gpu

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
M64 = (1 << 64) - 1

# row lengths around every boundary of the step kernels: a 32-token lane group, a 64-token chunk, the two chunks
# whose slots stay in registers (128 tokens), and rows that probe again in phase B
LENS = (0, 1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 200, 300, 600)
# one key at these positions of a 300-token row: four times in the first 32-token group of chunk 0, twice in one
# group of chunk 2, once in chunk 4
HOT_POS = (0, 3, 9, 17, 130, 150, 299)


def _opt(name):
    return (api.OPT_FTRL, O.OPT_FTRL) if name == "ftrl" else (api.OPT_SGD, O.OPT_SGD)


def _csr(rows, rng):
    """Rows (lists of id arrays) in a shuffled order -> (row_ptr u32, keys u64, labels u8)."""
    rows = [rows[i] for i in rng.permutation(len(rows))]
    rp = np.zeros(len(rows) + 1, np.uint32)
    rp[1:] = np.cumsum([r.size for r in rows])
    ids = np.concatenate(rows).astype(np.uint64) if rows else np.zeros(0, np.uint64)
    lab = rng.integers(0, 2, len(rows)).astype(np.uint8)
    return rp, api.hash_decimal_ids(ids), lab


def long_batch(seed, id_hi, extra_rows=0, extra_lo=0):
    """One row of every length in LENS plus a 300-token row that holds one key at HOT_POS, uniform ids in
    [0, id_hi); optionally `extra_rows` 64-token rows of ids never used elsewhere (from extra_lo on)."""
    rng = np.random.default_rng(seed)
    rows = [rng.integers(0, id_hi, n) for n in LENS]
    hot = rng.integers(0, id_hi, 300)
    hot[list(HOT_POS)] = rng.integers(0, id_hi)
    rows.append(hot)
    rows += [np.arange(64) + extra_lo + 64 * i for i in range(extra_rows)]
    return _csr(rows, rng)


def _steps_of(s):
    """Step s of a run: ids in a range that grows by 1500 per step, so that step 0 sees only fresh keys and every
    later step mixes keys with materialised rows and keys never seen."""
    return long_batch(10 + s, 2500 + 1500 * s)


def _keywise(ref, exact):
    """The exact-sum yardstick of a latent field with each key's noise taken as the largest of its coordinates': the
    K coordinates of a key share its row sums (Aq, L), and where a coordinate's float and exact runs happen to round
    alike the per-coordinate measure reads zero."""
    if ref.ndim != 2:
        return exact
    return ref + np.abs(np.asarray(ref, np.float64) - exact).max(1, keepdims=True)


def _compare_tables(ge, oe, fields, what, ftrl):
    assert np.array_equal(ge["present"], oe["present"]), what + ": key sets differ"
    for k in fields:
        assert_close(ge[k], oe[k], "%s %s" % (what, k))
    if ftrl:
        # the L1 threshold's exact zeros of w are zeros on both sides
        assert np.array_equal(ge["w"] == 0.0, oe["w"] == 0.0), "%s: exact zeros of w differ" % what


# -------------------------------------------------------------------------------------------------------------
# A. reference-shaped FM across latent widths
# -------------------------------------------------------------------------------------------------------------
def fm_run_vs_oracle(K, opt, steps=3):
    """`steps` steps of XF_MODEL_FM on long_batch rows against the oracle: per-row residuals and every seen key's
    w, n, z, v, nv, zv after each step; then predictions on a fresh batch, the unique-key count and the size.
    The reference sums a row's S = sum_tokens sum_k v in one float32 running sum, k outer (fm_worker.cc:178-192): at
    K >= 33 on rows of hundreds of tokens its rounding alone moves residuals by up to ~1e-4.  The oracle run with
    every sum in double (exact_sums(rows=True)) measures that noise element by element (assert_close_noise_aware)."""
    gopt, oopt = _opt(opt)
    gt = api.Table(latent_dim=K, optimizer=gopt, v_init=api.VINIT_COUNTER, seed=5, capacity=1 << 14)
    ot = O.Table(K=K, opt=oopt, init_mode=O.INIT_COUNTER, seed=5)
    xt = O.Table(K=K, opt=oopt, init_mode=O.INIT_COUNTER, seed=5)
    tr = api.Trainer(gt, model=api.MODEL_FM, max_rows=64, max_nnz=8192, keep_loss=True)
    tr.init_push()
    ot.init_push()
    xt.init_push()
    seen, uniq = [], 0
    for s in range(steps):
        rp, keys, lab = _steps_of(s)
        tr.step_host(rp, keys, lab)
        gl = tr.get_loss(lab.size)
        U, ol = ot.step(rp.astype(np.int64), keys, lab.astype(np.int32))
        with O.exact_sums(rows=True):
            _, xl = xt.step(rp.astype(np.int64), keys, lab.astype(np.int32))
        uniq += U
        what = "K=%d %s step %d" % (K, opt, s)
        # a row's rounding noise shows in its residual whatever the row: no bound on the noisy fraction
        assert_close_noise_aware(gl, ol, xl, what + " residuals", abs_floor=1e-6, max_noisy_frac=1.0)
        seen.append(keys)
        uk = np.unique(np.concatenate(seen))
        ge, oe, xe = gt.export(uk), ot.export(uk), xt.export(uk)
        assert np.array_equal(ge["present"], oe["present"]), what + ": key sets differ"
        # a long row's rounding reaches every key of the row (measured: 10 % of the elements at K = 24, up to 60 %
        # at K = 1024 of the oracle itself differ from its exact-sum run by more than 1e-5): each element must stay
        # within 8x its own measured noise, their share is free
        for k in ("w", "nw", "zw", "v", "nv", "zv"):
            assert_close_noise_aware(ge[k], oe[k], _keywise(oe[k], xe[k]), "%s %s" % (what, k), max_noisy_frac=1.0)
        if opt == "ftrl":
            # the L1 threshold's exact zeros are zeros on both sides wherever both oracle runs agree on them
            for k in ("w", "v"):
                decided = (oe[k] == 0.0) == (xe[k] == 0.0)
                assert np.array_equal((ge[k] == 0.0)[decided], (oe[k] == 0.0)[decided]), what + ": zeros of " + k
    rp, keys, _ = long_batch(99, 8000)
    with O.exact_sums(rows=True):
        xp = xt.predict(rp.astype(np.int64), keys)
    assert_close_noise_aware(tr.predict_host(rp, keys), ot.predict(rp.astype(np.int64), keys), xp,
                             "K=%d %s pctr" % (K, opt), abs_floor=1e-6, max_noisy_frac=1.0)
    assert tr.stats()["unique_keys"] == uniq
    assert gt.size() == ot.size()
    tr.close()
    gt.close()


def pull_push_vs_oracle(K, opt):
    """The Pull / Push entry points (xf_k_update with pushed gradients) against the oracle, bit for bit; the first
    Pull returns the counter-based initial v of every coordinate k < K."""
    gopt, oopt = _opt(opt)
    gt = api.Table(latent_dim=K, optimizer=gopt, v_init=api.VINIT_COUNTER, seed=3, capacity=1 << 13)
    ot = O.Table(K=K, opt=oopt, init_mode=O.INIT_COUNTER, seed=3)
    rng = np.random.default_rng(K)
    universe = rng.integers(0, 2 ** 64 - 1, 3000, dtype=np.uint64)
    for it in range(4):
        keys = np.unique(rng.choice(universe, 800))
        gw, gv = gt.pull(keys)
        ow, ov = ot.pull(keys)
        if it == 0:
            assert bits_equal(gw, ow) and bits_equal(gv, ov), "K=%d: initial values" % K
        assert_close(gw, ow, "pull w")
        assert_close(gv, ov, "pull v")
        g1 = (rng.standard_normal(keys.size) * 0.1).astype(np.float32)
        g2 = (rng.standard_normal((keys.size, K)) * 0.1).astype(np.float32)
        g1[::7] = 0.0
        g2[::5] = 0.0
        gt.push(keys, g1, g2)
        ot.push(keys, g1, g2)
    e, o = gt.export(universe), ot.export(universe)
    assert np.array_equal(e["present"], o["present"])
    for k in ("w", "nw", "zw", "v", "nv", "zv"):
        # same inputs, same operation order: the optimizer arithmetic itself is bit-exact
        assert bits_equal(e[k], o[k]), "K=%d %s: %s" % (K, opt, k)
    assert gt.size() == ot.size() == int(o["present"].sum())
    gt.close()


# K: VEC 1/2 with one lane per key (1, 2), VEC 1 with idle lanes (7), VEC 4 without the 256-bit loads (12, 20),
# the 256-bit loop (24, 32), 33 latent chunks for VEC 1/2/4 (33, 66, 132), two and eight chunks per lane (256, 1024)
FM_CASES = ([(K, "ftrl") for K in (1, 2, 7, 12, 20, 24, 32, 33, 66, 132, 256, 1024)] +
            [(K, "sgd") for K in (33, 132, 256)])


@pytest.mark.parametrize("K,opt", FM_CASES)
def test_fm_latent_widths_match_oracle(K, opt):
    fm_run_vs_oracle(K, opt)


@pytest.mark.parametrize("K,opt", FM_CASES)
def test_pull_push_latent_widths_bit_exact(K, opt):
    pull_push_vs_oracle(K, opt)


# -------------------------------------------------------------------------------------------------------------
# B. LR, lazy and eager, on a growing table
# -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bucket_log2", ["0", "2", "4"])
@pytest.mark.parametrize("eager", [False, True], ids=["lazy", "eager"])
@pytest.mark.parametrize("opt", ["ftrl", "sgd"])
def test_lr_long_rows_and_growth_match_oracle(opt, eager, bucket_log2, monkeypatch):
    """LR on long_batch rows plus 60 rows of fresh ids per step, from a 1024-slot table: the table grows several
    times while rows hold pending steps (lazy) and rows hold imported weights that are not f(z, n)."""
    monkeypatch.setenv("XFLOW_BUCKET_LOG2", bucket_log2)   # read whenever the table is allocated
    if eager:
        monkeypatch.setenv("XFLOW_EAGER", "1")              # read when the table is created
    gopt, oopt = _opt(opt)
    gt = api.Table(optimizer=gopt, capacity=1024)
    ot = O.Table(K=0, opt=oopt)
    tr = api.Trainer(gt, max_rows=128, max_nnz=8192, keep_loss=True)
    monkeypatch.delenv("XFLOW_EAGER", raising=False)
    seen, uniq, caps = [], 0, []
    rng = np.random.default_rng(7)
    for s in range(6):
        rp, keys, lab = long_batch(40 + s, 2000 + 1000 * s, extra_rows=60, extra_lo=10 ** 6 + 4000 * s)
        tr.step_host(rp, keys, lab)
        U, ol = ot.step(rp.astype(np.int64), keys, lab.astype(np.int32))
        uniq += U
        assert_close(tr.get_loss(lab.size), ol, "residuals step %d" % s, abs_floor=1e-6)
        seen.append(keys)
        caps.append(gt.capacity())
        if s == 1:
            # imported rows: some of them are touched again later, some never; w is not f(z, n)
            ik = np.unique(np.concatenate([keys[:200], api.hash_decimal_ids(np.arange(5 * 10 ** 6, 5 * 10 ** 6 + 100))]))
            iw = rng.normal(0, 0.3, ik.size).astype(np.float32)
            inw = rng.uniform(0, 2, ik.size).astype(np.float32) if opt == "ftrl" else None   # SGD keeps w only
            izw = rng.normal(0, 1, ik.size).astype(np.float32) if opt == "ftrl" else None
            gt.import_(ik, w=iw, nw=inw, zw=izw)
            ot.import_(ik, w=iw, nw=inw, zw=izw)
            seen.append(ik)
        uk = np.unique(np.concatenate(seen))
        _compare_tables(gt.export(uk), ot.export(uk), ("w", "nw", "zw"), "step %d" % s, opt == "ftrl")
    assert caps[-1] >= 4 * caps[0], "the table must grow at least twice after the first step: %s" % caps
    rp, keys, _ = long_batch(98, 12000)
    assert_close(tr.predict_host(rp, keys), ot.predict(rp.astype(np.int64), keys), "pctr", abs_floor=1e-6)
    assert tr.stats()["unique_keys"] == uniq
    assert gt.size() == ot.size()


# -------------------------------------------------------------------------------------------------------------
# C. checkpoints of lazy tables
# -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("opt", ["ftrl", "sgd"])
def test_lazy_checkpoint_continues_bit_equal(opt, tmp_path):
    """A lazy LR table with pending steps and imported weights, saved and loaded into a fresh table: both tables
    then take the same three steps and must end bit-equal (residual sums are integers, folding is pure)."""
    gopt, _ = _opt(opt)
    ta = api.Table(optimizer=gopt, capacity=1 << 14)
    tra = api.Trainer(ta, max_rows=128, max_nnz=8192)
    for s in range(2):
        tra.step_host(*long_batch(60 + s, 3000))
    rng = np.random.default_rng(3)
    ik = np.unique(api.hash_decimal_ids(np.concatenate([np.arange(0, 3000, 7), np.arange(10 ** 7, 10 ** 7 + 50)])))
    ta.import_(ik, w=rng.normal(0, 0.3, ik.size).astype(np.float32), nw=rng.uniform(0, 2, ik.size).astype(np.float32),
               zw=rng.normal(0, 1, ik.size).astype(np.float32))
    tra.step_host(*long_batch(62, 3000))                  # the rows of this step stay pending
    path = str(tmp_path / "lazy.bin")
    ta.save(path)
    tb = api.Table(optimizer=gopt, capacity=1 << 10)
    tb.load(path)
    trb = api.Trainer(tb, max_rows=128, max_nnz=8192)
    for s in range(3):
        batch = long_batch(70 + s, 4000)
        tra.step_host(*batch)
        trb.step_host(*batch)
    keys = np.sort(ta.list_keys())
    assert keys.size == ta.size() == tb.size()
    assert np.array_equal(keys, np.sort(tb.list_keys()))
    a, b = ta.export(keys), tb.export(keys)
    for k in ("w", "nw", "zw"):
        assert bits_equal(a[k], b[k]), k


# -------------------------------------------------------------------------------------------------------------
# D. canonical FM and MVM at every accepted width, and their predictions
# -------------------------------------------------------------------------------------------------------------
CANON_LENS = (0, 1, 5, 31, 32, 33, 40, 64, 65, 100)


def _canon_batch(seed, id_hi, rows=96):
    """Rows of the CANON_LENS lengths (empty ones included), uniform ids, values in +-[0.25, 1.75] with exact
    zeros and negatives."""
    rng = np.random.default_rng(seed)
    rp, keys, lab = _csr([rng.integers(0, id_hi, CANON_LENS[i % len(CANON_LENS)]) for i in range(rows)], rng)
    x = (rng.random(keys.size) * 1.5 + 0.25).astype(np.float32)
    x[::7] *= -1.0
    x[3::11] = 0.0
    return rp, keys, x, lab


@pytest.mark.parametrize("opt", ["ftrl", "sgd"])
@pytest.mark.parametrize("K", [4, 8, 16, 32, 64, 128])
def test_canonical_fm_widths_match_float64_model(K, opt):
    gopt, _ = _opt(opt)
    t = api.Table(latent_dim=K, optimizer=gopt, v_init=api.VINIT_COUNTER, seed=4, canonical_fm=1, capacity=1 << 14)
    tr = api.Trainer(t, model=api.MODEL_FM_CANONICAL, max_rows=128, max_nnz=8192, keep_loss=True)
    model = CanonicalFM64(K, opt == "ftrl", t.pull)
    uniq = 0
    for step in range(3):
        rp, keys, x, lab = _canon_batch(80 + step, 1500 + 1000 * step)
        loss = model.step(rp, keys, x, lab)
        tr.step_host_values(rp, keys, x, lab)
        uniq += np.unique(keys).size
        assert_close(tr.get_loss(lab.size), loss, "K=%d residuals, step %d" % (K, step), rel=2e-5, abs_floor=2e-6)
    allk = np.array(sorted(model.state), np.uint64)
    e, ref = t.export(allk), model.export(allk)
    for k in ("w", "v") + (("nw", "zw", "nv", "zv") if opt == "ftrl" else ()):
        assert_close(e[k].reshape(allk.size, -1), ref[k], "canonical FM K=%d %s" % (K, k), rel=2e-4, abs_floor=2e-7)
    assert tr.stats()["unique_keys"] == uniq
    # predictions, value by value, against the float64 forward pass on the table's own rows (a Pull inserts the
    # keys the batch has not seen, with the same defaults the forward pass uses)
    rp, keys, x, _ = _canon_batch(99, 4000)
    got = tr.predict_host_values(rp, keys, x)
    w, v = t.pull(keys)
    want = canonical_fm_forward64(rp, w, v, x)[0]
    assert_close(got, want, "canonical FM K=%d pctr" % K, rel=2e-5, abs_floor=2e-6)


@pytest.mark.parametrize("K", [4, 8, 16, 32])
def test_mvm_predictions_match_float64_forward(K):
    t = api.Table(latent_dim=K, optimizer=api.OPT_FTRL, v_init=api.VINIT_COUNTER, seed=4, canonical_fm=1,
                  capacity=1 << 13)
    tr = api.Trainer(t, model=api.MODEL_MVM, max_rows=128, max_nnz=8192, keep_loss=True)
    rng = np.random.default_rng(200 + K)
    rp, keys, x, lab = _canon_batch(120 + K, 1200)
    fields = rng.integers(0, 5, keys.size).astype(np.uint8)
    fields[::13] = 31
    uk = np.unique(keys)
    t.import_(uk, v=rng.normal(0.0, 0.6, (uk.size, K)).astype(np.float32))
    tr.step_host_fields(rp, keys, fields, x, lab)          # move the rows away from what was imported
    for with_vals in (True, False):
        xv = x if with_vals else None
        got = tr.predict_host_fields(rp, keys, fields, xv)
        _, v = t.pull(keys)
        want = mvm_forward64(rp, v, fields, xv)[0]
        assert_close(got, want, "MVM K=%d pctr (values: %s)" % (K, with_vals), rel=5e-5, abs_floor=5e-6)


# -------------------------------------------------------------------------------------------------------------
# E. kernel switches read once per process: checked in child processes
# -------------------------------------------------------------------------------------------------------------
def _child(fn, env, timeout=900):
    """Run `fn` of this module in a fresh interpreter with `env` added to the environment; its output is shown
    when it fails.  subprocess.run waits for the child and kills it on timeout."""
    code = "import sys; sys.path[:0] = %r; import test_gpu_kernel_shapes as m; m.%s()" % (
        [ROOT, TESTS, os.path.join(TESTS, "golden")], fn)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    r = subprocess.run(cmd, env=dict(os.environ, **env), cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, "%s with %s failed (exit %d):\n%s\n%s" % (fn, env, r.returncode, r.stdout[-4000:],
                                                                         r.stderr[-12000:])


# every shape xf_k_update_wide accepts: not canonical, K % 4 == 0, row <= 512 bytes
WIDE_CASES = [(K, "ftrl") for K in (4, 8, 16, 32, 36)] + [(K, "sgd") for K in (64, 116)]


def wide_child():
    for K, opt in WIDE_CASES:
        fm_run_vs_oracle(K, opt)
        pull_push_vs_oracle(K, opt)


def test_wide_update_kernel_matches_oracle():
    _child("wide_child", {"XFLOW_UPDATE_WIDE": "1"})


def zipf_batch(seed, rows=112):
    """CANON-like long rows (LENS, repeated) over Zipf(1.1) ids: the hottest key holds a large share of the
    tokens, and it occurs many times within single rows."""
    rng = np.random.default_rng(seed)
    lens = [LENS[i % len(LENS)] for i in range(rows)]
    ids = np.minimum(rng.zipf(1.1, sum(lens)), 10 ** 6) - 1
    rp = np.zeros(rows + 1, np.uint32)
    rp[1:] = np.cumsum(lens)
    return rp, api.hash_decimal_ids(ids.astype(np.uint64)), rng.integers(0, 2, rows).astype(np.uint8)


def cache_child():
    """XF_MODEL_FM with the hot-key cache size the environment sets, on Zipf batches, against the oracle; where
    the reference's own float32 summation order shows (hot keys), within its measured noise."""
    for K in (8, 33):
        gt = api.Table(latent_dim=K, optimizer=api.OPT_FTRL, v_init=api.VINIT_COUNTER, seed=6, capacity=1 << 15)
        ot = O.Table(K=K, opt=O.OPT_FTRL, init_mode=O.INIT_COUNTER, seed=6)
        xt = O.Table(K=K, opt=O.OPT_FTRL, init_mode=O.INIT_COUNTER, seed=6)
        tr = api.Trainer(gt, model=api.MODEL_FM, max_rows=128, max_nnz=1 << 15, keep_loss=True)
        tr.init_push(); ot.init_push(); xt.init_push()
        seen, uniq = [], 0
        for s in range(3):
            rp, keys, lab = zipf_batch(300 + s)
            _, cnt = np.unique(keys, return_counts=True)
            assert cnt.max() > 0.05 * keys.size
            tr.step_host(rp, keys, lab)
            U, ol = ot.step(rp.astype(np.int64), keys, lab.astype(np.int32))
            with O.exact_sums(rows=True):
                _, xl = xt.step(rp.astype(np.int64), keys, lab.astype(np.int32))
            uniq += U
            assert_close_noise_aware(tr.get_loss(lab.size), ol, xl, "K=%d residuals step %d" % (K, s), abs_floor=1e-6,
                                     max_noisy_frac=1.0)
            seen.append(keys)
            uk = np.unique(np.concatenate(seen))
            ge, oe, xe = gt.export(uk), ot.export(uk), xt.export(uk)
            assert np.array_equal(ge["present"], oe["present"])
            # a hot key's noise reaches every row that holds it, and every key of those rows
            for k in ("w", "nw", "zw", "v", "nv", "zv"):
                assert_close_noise_aware(ge[k], oe[k], _keywise(oe[k], xe[k]), "K=%d %s step %d" % (K, k, s),
                                         max_noisy_frac=1.0)
        assert tr.stats()["unique_keys"] == uniq
        assert gt.size() == ot.size()
        tr.close()
        gt.close()


@pytest.mark.parametrize("log2", ["0", "10"])
def test_hot_key_cache_sizes_match_oracle(log2):
    _child("cache_child", {"XFLOW_FM_CACHE_LOG2": log2})


# -------------------------------------------------------------------------------------------------------------
# F. the sharded step on one GPU, and pre-population
# -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model,opt,K,stash", [("lr", "ftrl", 0, None), ("lr", "ftrl", 0, "0"), ("fm", "ftrl", 8, None),
                                               ("fm", "sgd", 33, None), ("fm", "ftrl", 64, None)])
def test_sharded_step_on_one_rank_matches_oracle(model, opt, K, stash, monkeypatch):
    """XFLOW_MG_FORCE=1 runs the routed step (route, owner Pull / Push handlers, reply) with a one-rank
    communicator; with one worker the lock-step schedule is the plain sequence of steps."""
    monkeypatch.setenv("XFLOW_MG_FORCE", "1")
    if stash is not None:
        monkeypatch.setenv("XFLOW_MG_STASH", stash)
    gopt, oopt = _opt(opt)
    comm = api.Comm(api.Comm.new_id(), 0, 1, 0)
    gt = api.Table(latent_dim=K, optimizer=gopt, v_init=api.VINIT_COUNTER, seed=9, shard_index=0, num_shards=1,
                   capacity=1 << 16)
    ot = O.Table(K=K, opt=oopt, init_mode=O.INIT_COUNTER, seed=9)
    xt = O.Table(K=K, opt=oopt, init_mode=O.INIT_COUNTER, seed=9)     # every sum in double: the noise yardstick
    B = 2048
    tr = api.Trainer(gt, model=api.MODEL_LR if model == "lr" else api.MODEL_FM, max_rows=B, max_nnz=B * 64,
                     keep_loss=True, comm=comm)
    tr.init_push()
    ot.init_push()
    xt.init_push()
    fields = ("w", "nw", "zw") + (("v", "nv", "zv") if K else ())
    # FM rows of up to 63 tokens: the reference's float32 row sums show (see fm_run_vs_oracle)
    frac = 1.0 if K else 0.0
    seen, uniq = [], 0
    for s in range(3):
        rp, keys, lab = _mg_batch(s, B)
        tr.step_host(rp, keys, lab)
        U, ol = ot.step(rp.astype(np.int64), keys, lab.astype(np.int32))
        with O.exact_sums(rows=True):
            _, xl = xt.step(rp.astype(np.int64), keys, lab.astype(np.int32))
        uniq += U
        assert_close_noise_aware(tr.get_loss(B), ol, xl, "residuals step %d" % s, abs_floor=1e-6, max_noisy_frac=frac)
        seen.append(keys)
        uk = np.unique(np.concatenate(seen))
        ge, oe, xe = gt.export(uk), ot.export(uk), xt.export(uk)
        assert np.array_equal(ge["present"], oe["present"])
        for k in fields:
            assert_close_noise_aware(ge[k], oe[k], _keywise(oe[k], xe[k]), "%s step %d" % (k, s), max_noisy_frac=frac)
        if opt == "ftrl":
            assert np.array_equal(ge["w"] == 0.0, oe["w"] == 0.0), "exact zeros of w, step %d" % s
    rp, keys, _ = _mg_batch(2, B)
    with O.exact_sums(rows=True):
        xp = xt.predict(rp.astype(np.int64), keys)
    assert_close_noise_aware(tr.predict_host(rp, keys), ot.predict(rp.astype(np.int64), keys), xp, "pctr",
                             abs_floor=1e-6, max_noisy_frac=frac)
    tr.sync()
    assert tr.stats()["unique_keys"] == uniq
    assert gt.size() == ot.size()
    tr.close()
    gt.close()
    comm.close()


def _mg_batch(s, B):
    from xflow_b200 import datagen
    return datagen.make_csr_keys(600 + s, B, 32, 60000, api.hash_decimal_ids, ragged=True)


def _check_touched(t, first, count, shard=None, S=1):
    ids = np.arange(count, dtype=np.uint64) + np.uint64(first)
    want = O.hash_decimal_ids(ids)
    if shard is not None:
        want = want[np.array([O.shard_of(int(k), S) == shard for k in want], bool)]
    want = np.unique(want)
    got = np.sort(t.list_keys())
    assert got.size == t.size() == want.size, (first, count, got.size, want.size)
    assert np.array_equal(got, want), (first, count)
    e = t.export(want)
    assert e["present"].all()
    for k in ("w", "nw", "zw"):
        assert not e[k].any(), k                              # default contents


@pytest.mark.parametrize("first,count", [(0, 121), ((1 << 32) - 60, 120), (10 ** 10 - 50, 101), (M64 - 63, 64)],
                         ids=["0-120", "2^32", "1e10", "2^64"])
def test_touch_decimal_ids_inserts_the_hashed_range(first, count):
    t = api.Table(capacity=1024)
    t.touch_decimal_ids(first, count)
    _check_touched(t, first, count)
    t.touch_decimal_ids(first, count)                         # touching again inserts nothing
    assert t.size() == count


def test_touch_decimal_ids_beyond_one_host_chunk():
    """2^24 + 1000 ids (the host launches 2^24 at a time), across the change from 9 to 10 digits."""
    first, count = 10 ** 9 - (1 << 23), (1 << 24) + 1000
    t = api.Table(capacity=1 << 20)
    t.touch_decimal_ids(first, count)
    _check_touched(t, first, count)
    t.close()


def test_touch_decimal_ids_keeps_its_shard():
    """A table holding shard 3 of 4 (the last one, which also owns the tail [4 * width, 2^64 - 1)) keeps exactly
    the keys postoffice.cc's ranges give it."""
    t = api.Table(capacity=1024, num_shards=4, shard_index=3)
    want = []
    for first, count in ((0, 121), (10 ** 6, 20000), (M64 - 63, 64)):
        t.touch_decimal_ids(first, count)
        ids = np.arange(count, dtype=np.uint64) + np.uint64(first)
        keys = O.hash_decimal_ids(ids)
        want.append(keys[np.array([O.shard_of(int(k), 4) == 3 for k in keys], bool)])
    want = np.unique(np.concatenate(want))
    assert 0 < want.size
    got = np.sort(t.list_keys())
    assert got.size == t.size() and np.array_equal(got, want)
    e = t.export(want)
    assert e["present"].all() and not (e["w"].any() or e["nw"].any() or e["zw"].any())
