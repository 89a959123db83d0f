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


def ftrl64(g, w, n, z, alpha=0.05, beta=1.0, l1=5e-5, l2=10.0):
    """One FTRL-proximal step (ftrl.h:59-74) in float64."""
    n2 = n + g * g
    z2 = z + g - (np.sqrt(n2) - np.sqrt(n)) / alpha * w
    w2 = np.where(np.abs(z2) <= l1, 0.0, (z2 - np.sign(z2) * l1) / -((beta + np.sqrt(n2)) / alpha + l2))
    return w2, n2, z2


def sigmoid64(y):
    """Base::sigmoid (base.h:54-63) in float64: the clamps, then pow(2.718281828, y)."""
    y = np.asarray(y, np.float64)
    e = np.power(2.718281828, np.clip(y, -30.0, 30.0))
    return np.where(y < -30, 1e-6, np.where(y > 30, 1.0, e / (1 + e)))


def canonical_fm_forward64(rp, w, v, x):
    """XF_MODEL_FM_CANONICAL's forward pass in float64, y = sum w x + 1/2 sum_k[(sum v_k x)^2 - sum (v_k x)^2],
    on the per-token rows w[nnz], v[nnz, K] and values x[nnz].  Returns (pctr, S[B, K], row index of each token)."""
    B = rp.size - 1
    row_of = np.repeat(np.arange(B), np.diff(rp).astype(np.int64))
    x64 = np.asarray(x, np.float64)
    vx = np.asarray(v, np.float64) * x64[:, None]
    wx = np.zeros(B); np.add.at(wx, row_of, np.asarray(w, np.float64) * x64)
    S = np.zeros((B, vx.shape[1])); np.add.at(S, row_of, vx)
    Q = np.zeros(B); np.add.at(Q, row_of, (vx ** 2).sum(1))
    return sigmoid64(wx + 0.5 * ((S ** 2).sum(1) - Q)), S, row_of


class CanonicalFM64:
    """Float64 model of a canonical FM table trained by XF_MODEL_FM_CANONICAL (step_fmc.cu): per touched key one
    FTRL or SGD step on w with gw = sum r x / B and on v with gv_k = (sum r x S_k - v_k sum r x^2) / B.  New keys
    take their starting values from `pull(keys) -> (w, v)` (the table's insert-on-pull defaults)."""

    FIELDS = ("w", "nw", "zw", "v", "nv", "zv")

    def __init__(self, K, ftrl, pull, lr=1e-3):
        self.K, self.ftrl, self.pull, self.lr = K, ftrl, pull, lr
        self.state = {}

    def _rows(self, keys):
        uk, inv = np.unique(keys, return_inverse=True)
        new = np.array([k for k in uk if int(k) not in self.state], np.uint64)
        if new.size:
            w0, v0 = self.pull(new)
            for k, a, b in zip(new, w0, v0):
                self.state[int(k)] = [float(a), 0.0, 0.0, b.astype(np.float64), np.zeros(self.K), np.zeros(self.K)]
        W = np.array([self.state[int(k)][0] for k in uk])
        V = np.stack([self.state[int(k)][3] for k in uk]) if uk.size else np.zeros((0, self.K))
        return uk, inv, W, V

    def forward(self, rp, keys, x):
        uk, inv, W, V = self._rows(keys)
        return canonical_fm_forward64(rp, W[inv], V[inv], x)[0]

    def step(self, rp, keys, x, lab):
        uk, inv, W, V = self._rows(keys)
        B = rp.size - 1
        p, S, row_of = canonical_fm_forward64(rp, W[inv], V[inv], x)
        loss = p - lab
        x64 = np.asarray(x, np.float64)
        r = loss[row_of] * x64
        gw = np.zeros(uk.size); np.add.at(gw, inv, r)
        A = np.zeros((uk.size, self.K)); np.add.at(A, inv, r[:, None] * S[row_of])
        L2 = np.zeros(uk.size); np.add.at(L2, inv, r * x64)
        gv = (A - V * L2[:, None]) / B
        gw = gw / B
        for i, k in enumerate(uk):
            s = self.state[int(k)]
            if self.ftrl:
                s[0], s[1], s[2] = (float(a) for a in ftrl64(gw[i], s[0], s[1], s[2]))
                s[3], s[4], s[5] = ftrl64(gv[i], s[3], s[4], s[5])
            else:
                s[0] -= self.lr * gw[i]
                s[3] = s[3] - self.lr * gv[i]
        return loss

    def export(self, keys):
        return {f: np.array([np.atleast_1d(self.state[int(q)][j]) for q in keys]).reshape(len(keys), -1)
                for j, f in enumerate(self.FIELDS)}


def mvm_forward64(rp, v, fields, x):
    """XF_MODEL_MVM's forward pass in float64, y = sum_k prod_{fields present} (sum_{tokens of the field} v_k x), on
    the per-token rows v[nnz, K]; a row without tokens has y = 0.  Returns (pctr, S[B, 32, K], present[B, 32], row of
    each token)."""
    B = rp.size - 1
    K = v.shape[1]
    row_of = np.repeat(np.arange(B), np.diff(rp).astype(np.int64))
    x64 = np.ones(row_of.size) if x is None else np.asarray(x, np.float64)
    f = np.asarray(fields, np.int64)
    S = np.zeros((B, 32, K)); np.add.at(S, (row_of, f), np.asarray(v, np.float64) * x64[:, None])
    present = np.zeros((B, 32), bool); present[row_of, f] = True
    y = np.where(present.any(1), np.where(present[:, :, None], S, 1.0).prod(1).sum(1), 0.0)
    return sigmoid64(y), S, present, row_of


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
