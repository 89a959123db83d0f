"""ctypes binding of oracle/liboracle.so (the CPU restatement) and a runner for oracle/_ref/xflow_ref.

TEST INFRASTRUCTURE ONLY.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
``--impl reference`` leg may import this module; the product (xflow_b200/) never does.
"""
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liboracle.so")
REF_BIN = os.path.join(HERE, "_ref", "xflow_ref")

OPT_FTRL, OPT_SGD = 0, 1
INIT_DEFAULT, INIT_COUNTER, INIT_REFRNG, INIT_ZERO = 0, 1, 2, 3

_lib = None


def build(force=False):
    """Compile liboracle.so (always possible) and _ref/xflow_ref (only where /root/reference exists)."""
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(
            os.path.join(HERE, "xflow_oracle.cc")):
        subprocess.check_call(["make", "-C", HERE, "oracle"], stdout=subprocess.DEVNULL)
    ref_root = os.environ.get("XFLOW_REFERENCE", "/root/reference")
    if os.path.isdir(os.path.join(ref_root, "src", "model")):
        subprocess.check_call(["make", "-C", HERE, "ref", "REF=" + ref_root], stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        build()
    L = C.CDLL(LIB_PATH)
    u64, i64, f32, vp = C.c_uint64, C.c_int64, C.c_float, C.c_void_p
    L.xo_hash_bytes.restype = u64
    L.xo_hash_bytes.argtypes = [C.c_char_p, u64]
    L.xo_std_hash.restype = u64
    L.xo_std_hash.argtypes = [C.c_char_p, u64]
    L.xo_hash_decimal_ids.argtypes = [vp, u64, vp]
    L.xo_shard_of.restype = C.c_int
    L.xo_shard_of.argtypes = [u64, C.c_int]
    L.xo_sigmoid.restype = f32
    L.xo_sigmoid.argtypes = [f32]
    L.xo_counter_normal.restype = f32
    L.xo_counter_normal.argtypes = [u64, C.c_uint32, u64]
    L.xo_loader_open.restype = vp
    L.xo_loader_open.argtypes = [C.c_char_p, u64]
    L.xo_loader_close.argtypes = [vp]
    L.xo_loader_next.restype = i64
    L.xo_loader_next.argtypes = [vp]
    L.xo_loader_nnz.restype = i64
    L.xo_loader_nnz.argtypes = [vp]
    L.xo_loader_get.argtypes = [vp, vp, vp, vp]
    L.xo_table_create.restype = vp
    L.xo_table_create.argtypes = [C.c_int, C.c_int, f32, f32, f32, f32, f32, C.c_int, u64]
    L.xo_table_destroy.argtypes = [vp]
    L.xo_table_size.restype = u64
    L.xo_table_size.argtypes = [vp]
    L.xo_table_pull.argtypes = [vp, vp, u64, vp, vp]
    L.xo_table_push.argtypes = [vp, vp, u64, vp, vp]
    L.xo_table_import.argtypes = [vp, vp, u64, vp, vp, vp, vp, vp, vp]
    L.xo_table_export.argtypes = [vp, vp, u64, vp, vp, vp, vp, vp, vp, vp]
    L.xo_worker_compute.restype = i64
    L.xo_worker_compute.argtypes = [vp, vp, vp, vp, i64]
    L.xo_worker_get.argtypes = [vp, vp, vp, vp]
    L.xo_step.restype = i64
    L.xo_step.argtypes = [vp, vp, vp, vp, i64, vp]
    L.xo_init_push.argtypes = [vp]
    L.xo_predict.argtypes = [vp, vp, vp, i64, vp]
    L.xo_auc_logloss.argtypes = [vp, vp, i64, vp]
    L.xo_set_exact_sums.argtypes = [C.c_int]
    L.xo_worker_compute_given.restype = i64
    L.xo_worker_compute_given.argtypes = [C.c_int, vp, vp, vp, i64, vp, vp]
    _lib = L
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def hash_str(s: bytes) -> int:
    return lib().xo_hash_bytes(s, len(s))


def std_hash(s: bytes) -> int:
    return lib().xo_std_hash(s, len(s))


def hash_decimal_ids(ids):
    ids = np.ascontiguousarray(ids, dtype=np.uint64)
    out = np.empty_like(ids)
    lib().xo_hash_decimal_ids(_p(ids), ids.size, _p(out))
    return out


def shard_of(key: int, S: int) -> int:
    return lib().xo_shard_of(key, S)


def sigmoid(x: float) -> float:
    return lib().xo_sigmoid(x)


def load_blocks(path, block_bytes):
    """Yield (row_ptr int64[B+1], keys uint64[nnz], labels int32[B]) per reference block."""
    L = lib()
    h = L.xo_loader_open(path.encode(), block_bytes)
    if not h:
        raise FileNotFoundError(path)
    try:
        while True:
            B = L.xo_loader_next(h)
            if B <= 0:
                break
            nnz = L.xo_loader_nnz(h)
            rp = np.empty(B + 1, np.int64)
            keys = np.empty(nnz, np.uint64)
            lab = np.empty(B, np.int32)
            L.xo_loader_get(h, _p(rp), _p(keys), _p(lab))
            yield rp, keys, lab
    finally:
        L.xo_loader_close(h)


class Table:
    """Restated parameter store (KV apps 0 and 1) + FTRL/SGD."""

    def __init__(self, K=0, opt=OPT_FTRL, alpha=5e-2, beta=1.0, l1=5e-5, l2=10.0, lr=1e-3,
                 init_mode=INIT_DEFAULT, seed=0):
        self.K, self.opt = K, opt
        self.h = lib().xo_table_create(K, opt, alpha, beta, l1, l2, lr, init_mode, seed)

    def __del__(self):
        if getattr(self, "h", None):
            lib().xo_table_destroy(self.h)
            self.h = None

    def size(self):
        return lib().xo_table_size(self.h)

    def pull(self, keys, want_w=True, want_v=True):
        keys = np.ascontiguousarray(keys, np.uint64)
        w = np.empty(keys.size, np.float32) if want_w else None
        v = np.empty((keys.size, self.K), np.float32) if (want_v and self.K) else None
        lib().xo_table_pull(self.h, _p(keys), keys.size, _p(w), _p(v))
        return w, v

    def push(self, keys, gw=None, gv=None):
        keys = np.ascontiguousarray(keys, np.uint64)
        gw = None if gw is None else np.ascontiguousarray(gw, np.float32)
        gv = None if gv is None else np.ascontiguousarray(gv, np.float32)
        lib().xo_table_push(self.h, _p(keys), keys.size, _p(gw), _p(gv))

    def import_(self, keys, w=None, nw=None, zw=None, v=None, nv=None, zv=None):
        keys = np.ascontiguousarray(keys, np.uint64)
        arrs = [None if a is None else np.ascontiguousarray(a, np.float32) for a in (w, nw, zw, v, nv, zv)]
        lib().xo_table_import(self.h, _p(keys), keys.size, *[_p(a) for a in arrs])

    def export(self, keys):
        keys = np.ascontiguousarray(keys, np.uint64)
        n, K = keys.size, self.K
        out = dict(keys=keys, w=np.zeros(n, np.float32), nw=np.zeros(n, np.float32), zw=np.zeros(n, np.float32),
                   v=np.zeros((n, K), np.float32), nv=np.zeros((n, K), np.float32),
                   zv=np.zeros((n, K), np.float32), present=np.zeros(n, np.uint8))
        lib().xo_table_export(self.h, _p(keys), n, _p(out["w"]), _p(out["nw"]), _p(out["zw"]),
                              _p(out["v"]) if K else None, _p(out["nv"]) if K else None,
                              _p(out["zv"]) if K else None, _p(out["present"]))
        return out

    def init_push(self):
        lib().xo_init_push(self.h)

    def step(self, row_ptr, keys, labels):
        """One update() on a slice; returns (U, loss[B])."""
        row_ptr = np.ascontiguousarray(row_ptr, np.int64)
        keys = np.ascontiguousarray(keys, np.uint64)
        labels = np.ascontiguousarray(labels, np.int32)
        B = labels.size
        loss = np.empty(B, np.float32)
        U = lib().xo_step(self.h, _p(row_ptr), _p(keys), _p(labels), B, _p(loss))
        return U, loss

    def worker_compute(self, row_ptr, keys, labels):
        """Pull + forward + gradient, no push: returns (unique_keys, gw, gv, loss)."""
        row_ptr = np.ascontiguousarray(row_ptr, np.int64)
        keys = np.ascontiguousarray(keys, np.uint64)
        labels = np.ascontiguousarray(labels, np.int32)
        B = labels.size
        U = lib().xo_worker_compute(self.h, _p(row_ptr), _p(keys), _p(labels), B)
        uk = np.empty(U, np.uint64)
        gw = np.empty(U, np.float32)
        gv = np.empty((U, self.K), np.float32)
        loss = np.empty(B, np.float32)
        lib().xo_worker_get(_p(uk), _p(gw), _p(gv) if self.K else None, _p(loss))
        return uk, gw, gv, loss

    def predict(self, row_ptr, keys):
        row_ptr = np.ascontiguousarray(row_ptr, np.int64)
        keys = np.ascontiguousarray(keys, np.uint64)
        B = row_ptr.size - 1
        p = np.empty(B, np.float32)
        lib().xo_predict(self.h, _p(row_ptr), _p(keys), B, _p(p))
        return p


class exact_sums:
    """Context manager: accumulate the per-key gradient sums in double, and with rows=True also the per-row
    forward sums (w x, sum v, sum v^2) (analysis aid that measures the float32 summation-order noise of the
    reference itself; NOT the reference's arithmetic)."""

    def __init__(self, rows=False):
        self.mode = 3 if rows else 1

    def __enter__(self):
        lib().xo_set_exact_sums(self.mode)

    def __exit__(self, *a):
        lib().xo_set_exact_sums(0)


def worker_compute_given(K, row_ptr, keys, labels, w, v=None):
    """calculate_loss + calculate_gradient with externally pulled values for the SORTED unique keys.
    Returns (gw[U], gv[U,K], loss[B])."""
    row_ptr = np.ascontiguousarray(row_ptr, np.int64)
    keys = np.ascontiguousarray(keys, np.uint64)
    labels = np.ascontiguousarray(labels, np.int32)
    w = np.ascontiguousarray(w, np.float32)
    v = None if v is None else np.ascontiguousarray(v, np.float32)
    B = labels.size
    U = lib().xo_worker_compute_given(K, _p(row_ptr), _p(keys), _p(labels), B, _p(w), _p(v))
    gw = np.empty(U, np.float32)
    gv = np.empty((U, K), np.float32)
    loss = np.empty(B, np.float32)
    lib().xo_worker_get(None, _p(gw), _p(gv) if K else None, _p(loss))
    return gw, gv, loss


def auc_logloss(labels, pctr):
    """Base::calculate_auc: returns dict(logloss, auc, tp, fp) in the reference's definitions."""
    labels = np.ascontiguousarray(labels, np.int32)
    pctr = np.ascontiguousarray(pctr, np.float32)
    out = np.zeros(4, np.float64)
    lib().xo_auc_logloss(_p(labels), _p(pctr), labels.size, _p(out))
    return dict(logloss=float(out[0]), auc=float(out[1]), tp=int(out[2]), fp=int(out[3]))


def train_file(table, path, block_bytes, epochs, slices=1, init_push=True):
    """LRWorker/FMWorker::batch_training (lr_worker.cc:179-205) with core_num = `slices`
    processed sequentially: each block is cut in `slices` equal row ranges, remainder rows dropped."""
    if init_push:
        table.init_push()
    rows = 0
    for _ in range(epochs):
        for rp, keys, lab in load_blocks(path, block_bytes):
            B = lab.size
            ts = B // slices
            for i in range(slices):
                s, e = i * ts, (i + 1) * ts
                if e <= s:
                    continue
                sub_rp = rp[s:e + 1] - rp[s]
                table.step(sub_rp, keys[rp[s]:rp[e]], lab[s:e])
                rows += e - s
    return rows


def predict_file(table, path, block_bytes, slices=1):
    """predict(): lr_worker.cc:73-98.  Returns (labels, pctr) in output order."""
    labs, ps = [], []
    for rp, keys, lab in load_blocks(path, block_bytes):
        B = lab.size
        ts = B // slices
        for i in range(slices):
            s, e = i * ts, (i + 1) * ts
            if e <= s:
                continue
            sub_rp = rp[s:e + 1] - rp[s]
            ps.append(table.predict(sub_rp, keys[rp[s]:rp[e]]))
            labs.append(lab[s:e])
    if not ps:
        return np.zeros(0, np.int32), np.zeros(0, np.float32)
    return np.concatenate(labs), np.concatenate(ps)


# ------------------------------------------------------------------------------------------------
# the real reference (oracle/_ref/xflow_ref)
# ------------------------------------------------------------------------------------------------
def have_ref():
    return os.path.exists(REF_BIN)


def read_dump(path):
    """Parse a table dump written by ref_harness.cc."""
    with open(path, "rb") as f:
        raw = f.read()
    assert raw[:4] == b"XFTB"
    n = int(np.frombuffer(raw, np.uint64, 1, 4)[0])
    K, has_nz = [int(x) for x in np.frombuffer(raw, np.uint32, 2, 12)]
    off = 20
    out = {"K": K, "has_nz": has_nz}

    def take(dtype, count, shape=None):
        nonlocal off
        a = np.frombuffer(raw, dtype, count, off).copy()
        off += a.nbytes
        return a if shape is None else a.reshape(shape)

    out["keys"] = take(np.uint64, n)
    out["w"] = take(np.float32, n)
    if has_nz:
        out["nw"] = take(np.float32, n)
        out["zw"] = take(np.float32, n)
    if K:
        out["v"] = take(np.float32, n * K, (n, K))
        if has_nz:
            out["nv"] = take(np.float32, n * K, (n, K))
            out["zv"] = take(np.float32, n * K, (n, K))
    out["present"] = take(np.uint8, n)
    assert off == len(raw), (off, len(raw))
    return out


def run_ref(model, opt, train_prefix, test_prefix, epochs, cwd, core=1, block_mb=2, vdim=10,
            dump=None, preinit_dump=None, no_predict=False, fix_time=None, extra=(), servers=1, warm_epochs=0):
    """Run the compiled reference; returns dict(stdout, train_seconds, logloss, auc, pred_path).
    servers / warm_epochs are benchmark-only (ref_harness.cc): key-range server shards in the shim, and
    extra epochs timed on the warm table (-> warm_seconds)."""
    cmd = [REF_BIN, "--model", model, "--opt", opt, "--train", train_prefix, "--test", test_prefix,
           "--epochs", str(epochs), "--core", str(core), "--block-mb", str(block_mb), "--vdim", str(vdim)]
    if dump:
        cmd += ["--dump", dump]
    if preinit_dump:
        cmd += ["--preinit-dump", preinit_dump]
    if no_predict:
        cmd += ["--no-predict"]
    if fix_time is not None:
        cmd += ["--fix-time", repr(float(fix_time))]
    if servers > 1:
        cmd += ["--servers", str(servers)]
    if warm_epochs > 0:
        cmd += ["--warm-epochs", str(warm_epochs)]
    cmd += list(extra)
    res = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True, check=True)
    out = {"stdout": res.stdout, "pred_path": os.path.join(cwd, "pred_0_0.txt")}
    for line in res.stdout.splitlines():
        if line.startswith("XFREF train_seconds"):
            out["train_seconds"] = float(line.split()[-1])
        if line.startswith("XFREF warm_seconds"):
            out["warm_seconds"] = float(line.split()[-1])
        if line.startswith("logloss:"):
            toks = line.replace("=", " ").split()
            out["logloss"] = float(toks[1])
            if "auc" in toks:
                out["auc"] = float(toks[toks.index("auc") + 1])
    return out
