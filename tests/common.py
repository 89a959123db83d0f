"""Helpers shared by the test modules."""
import os

import numpy as np

from cases import CASES, SYN, SYN_TEST  # tests/golden/cases.py
from xflow_b200 import datagen

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")

REL_TOL = 1e-5   # north_star: "within 1e-5 relative on float logloss and learned weights"
ABS_FLOOR = 1e-7  # SURVEY §8d: abs floor near 0 (FTRL produces exact zeros)


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def stored_rows(e, g, k):
    """e[k] (an export on g["keys"]) on the rows golden g holds field k for: a case with latent_rows stores
    v, nv and zv for that sample of its keys only."""
    if k in ("v", "nv", "zv") and "latent_rows" in g.files:
        return e[k][g["latent_rows"]]
    return e[k]


def materialise_syn(tmp):
    tr, te = os.path.join(tmp, "syn_train"), os.path.join(tmp, "syn_test")
    datagen.write_text(tr + "-00000", *datagen.make_ids(**SYN))
    datagen.write_text(te + "-00000", *datagen.make_ids(**SYN_TEST))
    return tr, te


def data_prefixes(case, syn_data):
    if CASES[case]["data"] == "small":
        d = os.path.join(GOLDEN, "data")
        return os.path.join(d, "small_train"), os.path.join(d, "small_test")
    return syn_data


def close(a, b, rel=REL_TOL, abs_floor=ABS_FLOOR):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return np.abs(a - b) <= rel * np.abs(b) + abs_floor


def assert_close(a, b, what, rel=REL_TOL, abs_floor=ABS_FLOOR, max_bad_frac=0.0):
    """All (or all but max_bad_frac) elements within rel*|b| + abs_floor."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    ok = close(a, b, rel, abs_floor)
    bad = int((~ok).sum())
    if bad > max_bad_frac * max(ok.size, 1):
        idx = np.argwhere(~ok)[:5]
        detail = ", ".join("%s: got %.9g want %.9g" % (tuple(i), a[tuple(i)], b[tuple(i)]) for i in idx)
        raise AssertionError("%s: %d/%d outside tolerance (%s)" % (what, bad, ok.size, detail))


def bits_equal(a, b):
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def assert_close_noise_aware(got, ref, exact, what, rel=REL_TOL, abs_floor=ABS_FLOOR, max_noisy_frac=2e-3,
                             noise_factor=8.0):
    """Parity against the reference where the reference's own float32 summation order is part of its
    result.  A key that occurs thousands of times in one batch gets its gradient summed sequentially
    in float by the reference (lr_worker.cc:108-113), in the order its unstable std::sort left the
    occurrences; that sum carries rounding noise far above 1e-5 that no other summation order can
    reproduce.  `exact` is the same algorithm with the per-key sums accumulated in double
    (oracle.exact_sums), so |ref - exact| measures that noise element by element.  Required:
      * every element within rel*|ref| + abs_floor of the reference, OR within noise_factor times
        the reference's own measured noise;
      * the second clause is needed by at most max_noisy_frac of the elements."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    exact = np.asarray(exact, np.float64)
    assert got.shape == ref.shape == exact.shape, what
    strict = close(got, ref, rel, abs_floor)
    noise = np.abs(ref - exact)
    loose = np.abs(got - ref) <= noise_factor * noise + rel * np.abs(ref) + abs_floor
    bad = ~(strict | loose)
    if bad.any():
        idx = np.argwhere(bad)[:5]
        detail = ", ".join("%s: got %.9g ref %.9g exact %.9g" % (tuple(i), got[tuple(i)], ref[tuple(i)],
                                                                exact[tuple(i)]) for i in idx)
        raise AssertionError("%s: %d/%d outside tolerance AND outside the reference's own noise (%s)"
                             % (what, int(bad.sum()), bad.size, detail))
    noisy = int((~strict).sum())
    assert noisy <= max_noisy_frac * strict.size, "%s: %d/%d elements needed the noise clause" % (
        what, noisy, strict.size)
    return noisy


def oracle_case_run(case, syn_data, exact=False):
    """Run a golden case through the CPU restatement.  exact=True accumulates gradient sums in double
    (noise yardstick, see assert_close_noise_aware).  Returns (export dict on the golden keys, labels, pctr)."""
    from oracle import oracle as O
    c = CASES[case]
    g = golden(case)
    train, test = data_prefixes(case, syn_data)
    opt = O.OPT_FTRL if c["opt"] == "ftrl" else O.OPT_SGD
    if c.get("preinit"):
        t = O.Table(K=c["K"], opt=opt, init_mode=O.INIT_ZERO)
        t.import_(g["keys"], w=g["init_w"], v=g["init_v"])
    else:
        t = O.Table(K=c["K"], opt=opt)
    block = c.get("block_mb", 2) << 20
    if exact:
        with O.exact_sums():
            O.train_file(t, train + "-00000", block, c["epochs"])
    else:
        O.train_file(t, train + "-00000", block, c["epochs"])
    lab, p = O.predict_file(t, test + "-00000", (4 << 20) if c["model"] == "lr" else (2 << 20))
    return t.export(g["keys"]), lab, p


def check_fm_first_step(rp, keys, lab, K, v0_of, loss, export_of, alpha=0.05, beta=1.0, l1=5e-5, l2=10.0):
    """Closed form of the FIRST FM + FTRL step on a fresh table (w = 0, n = z = 0, v = v0) in float64,
    compared with an implementation's residuals and exported state.  Tolerances are noise-aware: a sum
    over a key's occurrences is accepted within a few float32 ulps of the sum of the |terms| (both the
    reference's sequential float sums and any other association of the same terms stay inside that).

      v0_of(unique_keys) -> v0[U, K] float32      export_of(unique_keys) -> dict(zw, nw, v, nv, zv)
      loss: the implementation's per-row residuals (float32, used as the exact input of the gradient)
    Follows fm_worker.cc:126-202 (S, Q, residual, gw = K sum loss, gv = sum loss (S - v), / rows) and
    ftrl.h:59-74.
    """
    B = lab.size
    d = keys.size // B
    assert keys.size == B * d and np.array_equal(np.diff(rp), np.full(B, d))
    uk, inv = np.unique(keys, return_inverse=True)
    v64 = v0_of(uk).astype(np.float64)
    S = v64.sum(1)[inv].reshape(B, d).sum(1)
    Q = (v64 ** 2).sum(1)[inv].reshape(B, d).sum(1)
    ex = np.power(2.718281828, S * S - Q)  # Base::sigmoid; arguments stay far inside the clamps
    loss = np.asarray(loss, np.float64)
    assert_close(loss, ex / (1.0 + ex) - lab, "FM residual, step 1", rel=1e-5, abs_floor=1e-6)
    occ_row = np.repeat(np.arange(B), d)
    eps = 2.0 ** -23

    def per_key(x):
        out = np.zeros(uk.size)
        np.add.at(out, inv, x[occ_row])
        return out

    L, Aq = per_key(loss), per_key(loss * S)
    # noise scales: S itself is a float32 sum of d*K terms, so its error is relative to sum |v| of the row
    Sabs = np.abs(v64).sum(1)[inv].reshape(B, d).sum(1)
    magL, magA = per_key(np.abs(loss)), per_key(np.abs(loss) * Sabs)
    e = export_of(uk)

    def within(got, ref, tol, what):
        bad = np.abs(np.asarray(got, np.float64) - ref) > tol
        assert not bad.any(), "%s: %d/%d outside tolerance, worst %g vs tol %g" % (
            what, int(bad.sum()), bad.size, float(np.abs(got - ref)[bad].max()), float(tol[bad].min()))

    # w: g = K * L / B ; from the zero state n = g^2, z = g
    gw = K * L / B
    tol_gw = 1e-5 * np.abs(gw) + 8 * eps * K * magL / B + 1e-30
    within(e["zw"], gw, tol_gw, "zw after step 1")
    within(e["nw"], gw ** 2, 2 * np.abs(gw) * tol_gw + tol_gw ** 2 + 1e-5 * gw ** 2, "nw after step 1")
    # v: g = (Aq - v L) / B ; n = g^2 ; z = g - |g| / alpha * v ; v' from (z, n)
    g = (Aq[:, None] - v64 * L[:, None]) / B
    tol_g = 1e-5 * np.abs(g) + 8 * eps * (magA[:, None] + np.abs(v64) * magL[:, None]) / B + 1e-30
    z = g - np.abs(g) / alpha * v64
    tol_z = tol_g * (1 + np.abs(v64) / alpha) + 1e-5 * np.abs(z)
    within(e["nv"], g ** 2, 2 * np.abs(g) * tol_g + tol_g ** 2 + 1e-5 * g ** 2, "nv after step 1")
    within(e["zv"], z, tol_z, "zv after step 1")
    denom = (beta + np.abs(g)) / alpha + l2
    vn = np.where(np.abs(z) <= l1, 0.0, (z - np.sign(z) * l1) / -denom)
    decided = np.abs(np.abs(z) - l1) > 2 * tol_z  # at the L1 threshold the last bit decides
    tol_v = tol_z / denom + 1e-5 * np.abs(vn) + 1e-30
    got_v = np.asarray(e["v"], np.float64)
    bad = decided & (np.abs(got_v - vn) > tol_v)
    assert not bad.any(), "v after step 1: %d/%d outside tolerance" % (int(bad.sum()), bad.size)
    return uk, e


def build_and_run_ps_compat(tmp_dir):
    """Compile tests/cxx/ps_compat_check.cc against the shipped headers + library and run it."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(str(tmp_dir), "ps_compat_check")
    libdir = os.path.join(root, "xflow_b200", "lib")
    r = subprocess.run(["g++", "-std=c++14", "-Wall", "-Wextra", "-I", os.path.join(root, "include"),
                        os.path.join(root, "tests", "cxx", "ps_compat_check.cc"), "-o", exe, "-L", libdir,
                        "-lxflow_b200", "-Wl,-rpath," + libdir, "-lpthread"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "warning" not in r.stderr, r.stderr
    return subprocess.run([exe], capture_output=True, text=True, timeout=120)
