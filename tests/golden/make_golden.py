"""Regenerates tests/golden/*.npz by RUNNING THE REFERENCE ITSELF (oracle/_ref/xflow_ref = the
reference's src/ compiled unmodified against the in-process ps shim, core_num = 1).

    python tests/golden/make_golden.py        # needs /root/reference (this container only)

Each golden file holds, for one (data, model, optimizer, epochs) case: the sorted key list, the
reference's final table (w and, for FTRL, n and z; v rows for FM), the initial table when the case
replays a pre-initialised latent table, the reference's predictions (as printed to pred_0_0.txt,
6 significant digits) and its logloss / auc line.  The synthetic text inputs are regenerated from a
seed by xflow_b200.datagen (bit-reproducible), the bundled 200-row shards are copied as data fixtures.
Each REF_RUNS entry is stored as the reference's final table on a sample of its keys.
"""
import os
import shutil
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from oracle import oracle as O  # noqa: E402
from xflow_b200 import datagen  # noqa: E402

REF_DATA = "/root/reference/data"

from cases import CASES, REF_RUNS, SYN, SYN_TEST, ref_run_name  # noqa: E402


def sample_rows(n, size):
    """A fixed, seeded choice of `size` of `n` rows, sorted."""
    return np.sort(np.random.default_rng(0).choice(n, size, replace=False))


def ref_run_keys(keys, train_prefix, size=512, hot=32):
    """Of a reference run's sorted `keys`, the ones stored: the `hot` most frequent keys of the training shard
    (the keys whose many occurrences per batch the reference sums in float32) and a seeded sample of the rest,
    `size` in all.  Returns a boolean mask over `keys`."""
    seen = np.concatenate([k for _, k, _ in O.load_blocks(train_prefix + "-00000", 1 << 20)])
    uk, cnt = np.unique(seen, return_counts=True)
    mask = np.isin(keys, uk[np.argsort(-cnt, kind="stable")[:hot]])
    rest = np.flatnonzero(~mask)
    mask[rest[sample_rows(rest.size, size - int(mask.sum()))]] = True
    return mask


def materialise_data(kind, tmp):
    """Returns (train_prefix, test_prefix) with '<prefix>-00000' files present."""
    if kind == "small":
        d = os.path.join(HERE, "data")
        return os.path.join(d, "small_train"), os.path.join(d, "small_test")
    tr, te = os.path.join(tmp, "syn_train"), os.path.join(tmp, "syn_test")
    if not os.path.exists(tr + "-00000"):
        datagen.write_text(tr + "-00000", *datagen.make_ids(**SYN))
        datagen.write_text(te + "-00000", *datagen.make_ids(**SYN_TEST))
    return tr, te


def main():
    if not O.have_ref():
        O.build()
    assert O.have_ref(), "reference binary could not be built (is /root/reference present?)"
    os.makedirs(os.path.join(HERE, "data"), exist_ok=True)
    for name in ("small_train-00000", "small_test-00000"):
        dst = os.path.join(HERE, "data", name)
        if not os.path.exists(dst):
            shutil.copyfile(os.path.join(REF_DATA, name), dst)
            os.chmod(dst, 0o644)
    tmp = tempfile.mkdtemp()
    for name, c in CASES.items():
        train, test = materialise_data(c["data"], tmp)
        run = tempfile.mkdtemp()
        pre = os.path.join(run, "pre.bin") if c.get("preinit") else None
        r = O.run_ref(c["model"], c["opt"], train, test, c["epochs"], run, core=1, block_mb=c.get("block_mb", 2),
                      vdim=c["K"] or 10, dump=os.path.join(run, "final.bin"), preinit_dump=pre, fix_time=1.5e9)
        d = O.read_dump(os.path.join(run, "final.bin"))
        out = dict(keys=d["keys"], w=d["w"], present=d["present"], logloss=np.float64(r["logloss"]),
                   auc=np.float64(r.get("auc", np.nan)))
        for k in ("nw", "zw", "v", "nv", "zv"):
            if k in d:
                out[k] = d[k]
        if pre:
            p = O.read_dump(pre)
            assert np.array_equal(p["keys"], d["keys"])
            out["init_w"] = p["w"]
            out["init_v"] = p["v"]
        if c.get("latent_rows"):
            out["latent_rows"] = sample_rows(d["keys"].size, c["latent_rows"])
            for k in ("v", "nv", "zv"):
                out[k] = out[k][out["latent_rows"]]
        pred = np.loadtxt(r["pred_path"], ndmin=2)
        out["pred_pctr"] = pred[:, 0].astype(np.float64)
        out["pred_label"] = pred[:, 2].astype(np.int32)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        print("%-24s keys=%d logloss=%s auc=%s" % (name, d["keys"].size, r["logloss"], r.get("auc")))
    for model, opt, K, epochs in REF_RUNS:
        train, test = materialise_data("syn", tmp)
        run = tempfile.mkdtemp()
        O.run_ref(model, opt, train, test, epochs, run, core=1, block_mb=1, vdim=K or 10,
                  dump=os.path.join(run, "final.bin"), fix_time=1.5e9)
        d = O.read_dump(os.path.join(run, "final.bin"))
        keep = ref_run_keys(d["keys"], train)
        name = ref_run_name(model, opt, K, epochs)
        np.savez_compressed(os.path.join(HERE, name + ".npz"),
                            **{k: d[k][keep] for k in ("keys", "w", "nw", "zw", "v", "nv", "zv") if k in d})
        print("%-24s keys=%d of %d" % (name, int(keep.sum()), d["keys"].size))
    # known-answer vectors of std::hash<std::string> (libstdc++), via the real std::hash
    strs = [b"0", b"1163", b"8672", b"185", b"7755", b"", b"1520", b"2738", b"123456789",
            b"feature_with_a_long_name_0123456789"]
    np.savez(os.path.join(HERE, "std_hash.npz"), strings=np.array(strs, dtype="S64"),
             hashes=np.array([O.std_hash(s) for s in strs], np.uint64))
    shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
