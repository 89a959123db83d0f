#!/usr/bin/env python
"""bench.py — training examples/sec of the xflow hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workloads a,b,...] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch per GPU: LRWorker::update / FMWorker::update (pull,
forward, gradient, push) plus the server-side FTRL step it triggers.  The line's own numbers are the
metric's configuration: LR + FTRL on synthetic libffm rows, ids uniform in a 1e8-feature space, 100 nnz per
row, 65 536 rows per GPU and step (keys = std::hash of the decimal id string, as the reference's loader
makes them), the table pre-populated with all 1e8 ids.  `extra` carries the same measurement for
FM k=16 + FTRL on the same data (the metric's other half) and for the other BASELINE configs that fit the
GPUs at hand (cfg2 / cfg3 at N = 1; cfg4 (1e9 ids) and cfg5 (FM k=16, Zipf ids) at N > 1).  For N > 1
(torchrun, one rank per GPU) every rank trains its own batch against the table range-sharded over the N
GPUs (weak scaling: 65 536 rows per GPU, the id space stays what the config says).

  value     whole-job examples/s, batches already resident in HBM (device-timed, max over ranks)
  e2e       same metric from a TEXT shard in host memory through the C ABI (block formation on the host,
            H2D of the raw text, parse + hash + step on the device) — what the reference arm does from its
            text shard; e2e.binary_ids is the same with a pre-parsed CSR of u32 ids in page-locked memory
  roofline  dominant kernel: SURVEY §8d algorithmic bytes / its CUDA-event time, vs the measured HBM peak
  cpu_baseline  the reference's own CPU implementation (oracle/_ref, compiled from the reference's
            sources) on the box's host cores, on a bounded sample of the same workload

--impl reference times only that CPU implementation (same rows per step, warm table, all host cores,
key-range server shards in the in-process ps shim) and prints the same line with "impl": "reference".
"""
import argparse
import ctypes as C
import json
import os
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_ROWS = 65536
WORKLOADS = {
    # BASELINE.json metric: "LR & FM-k16 FTRL, 1e8-feat libsvm ~100nnz"
    "headline_lr": dict(model="lr", opt="ftrl", K=0, id_space=10 ** 8, nnz=100, dist="uniform",
                        name="LR+FTRL, synthetic libffm ids uniform in 1e8-feature space, 100 nnz/row, batch 65536 per GPU"),
    "headline_fm": dict(model="fm", opt="ftrl", K=16, id_space=10 ** 8, nnz=100, dist="uniform",
                        name="FM k=16+FTRL, synthetic libffm ids uniform in 1e8-feature space, 100 nnz/row, batch 65536 per GPU"),
    # BASELINE.json configs[1..4]
    "cfg2": dict(model="lr", opt="ftrl", K=0, id_space=10 ** 7, nnz=64, dist="uniform",
                 name="cfg2: LR+FTRL, ids uniform in 1e7-feature space, 64 nnz/row, batch 65536"),
    "cfg3": dict(model="fm", opt="sgd", K=8, id_space=10 ** 7, nnz=64, dist="uniform",
                 name="cfg3: FM k=8+SGD, ids uniform in 1e7-feature space, 64 nnz/row, batch 65536"),
    "cfg4": dict(model="lr", opt="ftrl", K=0, id_space=10 ** 9, nnz=100, dist="uniform",
                 name="cfg4: LR+FTRL, ids uniform in 1e9-feature hash space, 100 nnz/row, batch 65536 per GPU"),
    "cfg5": dict(model="fm", opt="ftrl", K=16, id_space=10 ** 8, nnz=100, dist="zipf",
                 name="cfg5: FM k=16+FTRL, Zipf(1.05)-skewed ids in 1e8-feature space, 100 nnz/row, batch 65536 per GPU"),
}
MAIN = "headline_lr"
RING = 8  # distinct batches cycled through (8 x 52 MB of keys > 126 MB L2; the tables are GBs)
DUMP_KEYS = 1 << 16  # keys per workload written by --dump-outputs: all six workloads stay under 32 MB


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def config_of(wl, world):
    """The workload description both arms print (identical dict in the reference arm's line)."""
    return {"workload": wl["name"], "model": wl["model"], "optimizer": wl["opt"], "latent_dim": wl["K"],
            "batch_per_gpu": B_ROWS, "nnz_per_row": wl["nnz"], "id_space": wl["id_space"], "id_distribution": wl["dist"],
            "parallelism": "dp%d, table range-sharded over %d GPU(s)" % (world, world)}


def algorithmic_bytes(wl, B, nnz, U):
    """SURVEY.md §8d: keys + row_ptr + labels + pull + optimizer state read + write, per batch."""
    D = 1 + wl["K"]
    R = 3 if wl["opt"] == "ftrl" else 1
    step = nnz * 8 + (B + 1) * 4 + B * 4 + U * D * 4          # CSR in, w/v rows pulled
    update = U * D * 4 * R * 2                                 # optimizer state read + written
    return step, update


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the benchmark runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max_mhz = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                self.samples.append((time.monotonic(), mhz, reasons))
            except Exception:
                pass
            time.sleep(0.004)

    def summary(self, windows):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        nv = self.nv
        win = [s for s in self.samples if any(t0 <= s[0] <= t1 for t0, t1 in windows)] or self.samples[-3:]
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        seen = set()
        for _, _, r in win:
            for bit, name in names.items():
                if r & bit:
                    seen.add(name)
        mhz = sorted(s[1] for s in win)
        return {"sm_mhz": float(mhz[len(mhz) // 2]) if mhz else None, "sm_max_mhz": float(self.max_mhz),
                "reasons": sorted(seen), "samples": len(win)}


def make_ids(wl, seed, rows=B_ROWS):
    from xflow_b200 import datagen
    return datagen.make_ids(seed=seed, rows=rows, nnz_per_row=wl["nnz"], id_space=wl["id_space"], dist=wl["dist"],
                            zipf_s=1.05)


# --------------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# --------------------------------------------------------------------------------------------------
def cpu_reference(wl, rows, warm_epochs, cores, servers):
    """The reference's CPU implementation (oracle/_ref = its own sources + in-process ps shim) on a text shard
    of `rows` rows of the workload: one cold epoch (empty table: the std::unordered_map grows) and
    `warm_epochs` more on the warm table.  Returns dict(cold, warm examples/s, seconds, kind, how)."""
    from oracle import oracle as O
    from xflow_b200 import datagen
    tmp = tempfile.mkdtemp(prefix="xfbench_")
    rp, ids, lab = make_ids(wl, 4242, rows)
    train = os.path.join(tmp, "train")
    datagen.write_text(train + "-00000", rp, ids, lab)
    open(os.path.join(tmp, "empty-00000"), "w").close()
    size_mb = os.path.getsize(train + "-00000") // (1 << 20) + 2
    out = {"rows": rows}
    if O.have_ref():
        r = O.run_ref(wl["model"], wl["opt"], train, os.path.join(tmp, "empty"), 1, tmp, core=cores, block_mb=size_mb,
                      vdim=wl["K"] or 10, no_predict=True, servers=servers, warm_epochs=warm_epochs)
        out.update(kind="reference", cores=cores, cold=rows / r["train_seconds"], cold_seconds=r["train_seconds"],
                   warm=(warm_epochs * rows / r["warm_seconds"]) if warm_epochs else None,
                   warm_seconds=r.get("warm_seconds"),
                   how="oracle/_ref/xflow_ref = the reference's src/ compiled unmodified (-O2) + in-process ps shim "
                       "(zero transport cost), core_num=%d worker threads, %d key-range server shard(s)" % (cores, servers))
    else:
        t = O.Table(K=wl["K"], opt=O.OPT_FTRL if wl["opt"] == "ftrl" else O.OPT_SGD)
        t0 = time.perf_counter()
        O.train_file(t, train + "-00000", size_mb << 20, 1)
        t1 = time.perf_counter()
        if warm_epochs:
            O.train_file(t, train + "-00000", size_mb << 20, warm_epochs, init_push=False)
        t2 = time.perf_counter()
        out.update(kind="port", cores=1, cold=rows / (t1 - t0), cold_seconds=t1 - t0,
                   warm=(warm_epochs * rows / (t2 - t1)) if warm_epochs else None, warm_seconds=t2 - t1,
                   how="oracle/xflow_oracle.cc (scalar port), 1 thread")
    try:
        os.remove(train + "-00000")
    except OSError:
        pass
    return out


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    servers = max(1, min(32, cores))
    r = cpu_reference(wl, B_ROWS, args.steps, cores, servers)   # the cold epoch is the warm-up
    value = r["warm"]
    line = {
        "impl": "reference", "metric": "training examples/sec", "value": value, "unit": "examples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["warm_seconds"] / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(wl, args.gpus),
        "cpu_baseline": {"value": value, "unit": "examples/s", "cores": r["cores"], "kind": r["kind"],
                         "cold_table_value": r["cold"],
                         "sample": "every step = one epoch over a text shard of %d rows x %d nnz of the workload (the GPU arm's "
                                   "rows per GPU and step): text parse + update(); `value` = %d epochs on the WARM table (all "
                                   "keys present, like the GPU arm's steady state), cold_table_value = the first epoch on an "
                                   "empty table (unordered_map growth), which serves as the warm-up; %s. The host has one set "
                                   "of cores whatever N is: the same run stands for every --gpus N."
                                   % (B_ROWS, wl["nnz"], args.steps, r["how"])},
        "e2e": {"value": value, "unit": "examples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
class Ring:
    """RING distinct batches of one workload: device-resident CSR with keys hashed on the device, and
    page-locked host CSR of u32 ids for the binary end-to-end leg."""

    def __init__(self, wl, rank, api, torch, stream):
        self.dev, self.pin = [], []
        self.nnz = B_ROWS * wl["nnz"]
        lib = api.lib()
        for i in range(RING):
            rp, ids, lab = make_ids(wl, 1 + 1000 * rank + i)
            ids32 = ids.astype(np.uint32)
            d_rp = torch.from_numpy(rp.view(np.uint8)).cuda()
            d_ids = torch.from_numpy(ids32.view(np.uint8)).cuda()
            d_lab = torch.from_numpy(lab.view(np.uint8)).cuda()
            d_keys = torch.empty(ids32.size * 8, dtype=torch.uint8, device="cuda")
            torch.cuda.current_stream().synchronize()
            assert lib.xf_hash_decimal_ids_device(C.c_void_p(d_ids.data_ptr()), ids32.size, C.c_void_p(d_keys.data_ptr()),
                                                  C.c_void_p(stream.cuda_stream)) == 0
            stream.synchronize()   # d_ids goes back to the allocator only after the hash kernel has read it
            self.dev.append((d_rp, d_keys, d_lab))
            self.pin.append(tuple(torch.from_numpy(a.view(np.uint8)).pin_memory() for a in (rp, ids32, lab)))
            del d_ids


def text_leg(api, tr, wl, rank, steps, warm, barrier):
    """Text -> model: one batch as a text shard in the reference's format; every step = H2D of the raw text +
    device parse/hash + one training step, pipelined through the two-phase ingest of the C ABI (block i+1 is
    copied and parsed while block i trains).  Two variants: text blocks already in page-locked host memory
    (the contract's end-to-end: host buffers in, copies inside the timed region), and from the FILE through
    xf_loader_next_raw (block formation from the page cache, what the reference's fread does).  Host wall clock
    around synced runs."""
    from xflow_b200 import datagen
    tmp = tempfile.mkdtemp(prefix="xftext_")
    path = os.path.join(tmp, "shard-%05d" % rank)
    rp, ids, lab = make_ids(wl, 777 + rank)
    datagen.write_text(path, rp, ids, lab)
    size = os.path.getsize(path)
    lib = api.lib()
    text, ln, r, z = C.c_void_p(), C.c_uint64(), C.c_uint32(), C.c_uint32()
    ld = api.Loader(path, size + (1 << 20))

    def check(rc):
        assert rc == 0, lib.xf_last_error()

    # ---- (a) from the file: loader forms the block (two alternating page-locked buffers), rewound per epoch
    def next_block():
        check(lib.xf_loader_rewind(ld.h))   # the same shard again
        check(lib.xf_loader_next_raw(ld.h, C.byref(text), C.byref(ln)))
        check(lib.xf_trainer_ingest_begin(tr.h, text, ln.value))

    # Both variants keep TWO blocks in flight behind the one being trained on (include/xflow_b200.h,
    # xf_trainer_ingest_begin): H2D of block i+2, parse of block i+1 and the step of block i run at the same time.
    def run_file(n):
        for i in range(min(n, 2)):
            next_block()
        for i in range(n):
            check(lib.xf_trainer_ingest_end(tr.h, C.byref(r), C.byref(z)))
            assert r.value == B_ROWS
            check(lib.xf_trainer_step_ingested(tr.h, 0, r.value))
            if i + 2 < n:   # the loader's buffer of block i is free again: its copy finished before _end(i) returned
                next_block()
    # ---- (b) text already in page-locked host memory (two copies, alternated like a reader would)
    bufs = []
    for _ in range(2):
        p = C.c_void_p()
        check(lib.xf_host_alloc(C.byref(p), size + 16))
        C.memmove(p, open(path, "rb").read(), size)
        bufs.append(p)

    def run_pinned(n):
        for i in range(min(n, 2)):
            check(lib.xf_trainer_ingest_begin(tr.h, bufs[i & 1], size))
        for i in range(n):
            check(lib.xf_trainer_ingest_end(tr.h, C.byref(r), C.byref(z)))
            assert r.value == B_ROWS
            check(lib.xf_trainer_step_ingested(tr.h, 0, r.value))
            if i + 2 < n:
                check(lib.xf_trainer_ingest_begin(tr.h, bufs[i & 1], size))
    out = {"text_bytes_per_step": size}
    for name, fn in (("file", run_file), ("pinned", run_pinned)):
        fn(warm)
        tr.sync()
        barrier()
        t0 = time.perf_counter()
        fn(steps)
        tr.sync()
        barrier()
        out[name] = (time.perf_counter() - t0) / steps
    ld.close()
    for p in bufs:
        lib.xf_host_free(p)
    os.remove(path)
    return out


def dump_outputs(out_dir, name, wl, table, d_keys):
    """What the device-resident timed path computed in its last step: the table rows of that batch's keys as the
    step left them (what a pull or export returns), on a fixed, seeded sample of DUMP_KEYS of its unique keys in
    key order.  One float32 file per field, <out_dir>/<workload>.<field>.npy (FM k=16 + FTRL: 13 MB)."""
    keys = np.unique(d_keys.cpu().numpy().view(np.uint64))
    keys = keys[np.sort(np.random.default_rng(0).choice(keys.size, min(DUMP_KEYS, keys.size), replace=False))]
    e = table.export(keys)
    assert e["present"].all()
    fields = ["w", "nw", "zw"] if wl["opt"] == "ftrl" else ["w"]
    if wl["K"]:
        fields += ["v", "nv", "zv"] if wl["opt"] == "ftrl" else ["v"]
    for f in fields:
        np.save(os.path.join(out_dir, "%s.%s.npy" % (name, f)), e[f].astype(np.float32))


def run_workload(name, wl, args, rank, world, local, comm, api, torch, stream, sampler, barrier, allmax):
    B, nnz = B_ROWS, B_ROWS * wl["nnz"]
    model = api.MODEL_LR if wl["model"] == "lr" else api.MODEL_FM
    ids_per_shard = wl["id_space"] // world
    cap = 1 << 20
    while cap < 2.0 * ids_per_shard + 2.0 * nnz:   # load <= 0.5 with every id of the space present
        cap <<= 1
    cap <<= int(os.environ.get("XF_BENCH_CAP_SHIFT", "0"))   # A/B: lower load factors
    table = api.Table(latent_dim=wl["K"], optimizer=api.OPT_FTRL if wl["opt"] == "ftrl" else api.OPT_SGD, device=local,
                      capacity=cap, seed=1, shard_index=rank, num_shards=world)
    table.set_stream(stream.cuda_stream)
    tr = api.Trainer(table, model=model, max_rows=B, max_nnz=nnz + 1024, comm=comm)
    ring = Ring(wl, rank, api, torch, stream)
    results = torch.zeros(max(args.steps, 1), dtype=torch.float32).pin_memory()
    out = {}
    with torch.cuda.stream(stream):
        table.touch_decimal_ids(0, wl["id_space"])   # every id of the feature space exists (this shard: its range)
        tr.init_push()

        def run_device(k0, k):
            for i in range(k0, k0 + k):
                d = ring.dev[i % RING]
                tr.step_device(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), B, nnz)
        run_device(0, RING)              # every ring key has been updated once (FM: latent rows materialised)
        run_device(0, args.warmup)       # warm-up steps (untimed)
        tr.sync()
        # ---------------- device-resident timed region
        st0 = tr.stats()
        l0 = tr.launches()
        tr.set_profile(True)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_w0 = time.monotonic()
        e0.record(stream)
        run_device(args.warmup, args.steps)
        e1.record(stream)
        barrier()
        t_w1 = time.monotonic()
        ms = e0.elapsed_time(e1)
        prof = tr.profile()
        tr.set_profile(False)
        st1 = tr.stats()
        launches = tr.launches() - l0
        sampler_windows = [(t_w0, t_w1)]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, name, wl, table, ring.dev[(args.warmup + args.steps - 1) % RING][1])
        # ---------------- end-to-end, binary: page-locked host CSR of u32 ids, hashed on the device
        def one(i, addr):
            p = ring.pin[i % RING]
            tr.step_host_ids_async(p[0].data_ptr(), p[1].data_ptr(), p[2].data_ptr(), B, nnz, addr)
        for i in range(args.warmup):
            one(i, results.data_ptr())
        tr.sync()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for i in range(args.steps):
            one(i, results.data_ptr() + 4 * i)
        f1.record(stream)
        tr.sync()
        barrier()
        ms_bin = f0.elapsed_time(f1)
        assert np.isfinite(results[: args.steps].numpy()).all()
        # ---------------- end-to-end, text (the headline e2e): what the reference arm does from its shard
        text = None
        if not args.no_text_e2e:
            text = text_leg(api, tr, wl, rank, args.steps, 2, barrier)
    ms, ms_bin = allmax(ms), allmax(ms_bin)
    steps = args.steps
    U = (st1["unique_keys"] - st0["unique_keys"]) / max(steps, 1)
    peak, peak_src = load_peaks()
    b_step, b_update = algorithmic_bytes(wl, B, nnz, U)
    t_a = prof["step_ms"] / max(prof["steps"], 1) * 1e-3
    t_b = prof["update_ms"] / max(prof["steps"], 1) * 1e-3
    if world > 1:
        kern = [("owner Pull over routed tokens: xf_k_pull_tokens", b_step, t_a),
                ("owner Push, S sources: %s" % ("xf_k_push_tokens_lr" if wl["K"] == 0 else "xf_k_acc_tokens + xf_k_update"), b_update, t_b)]
    elif t_b > 0.05 * t_a:
        kern = [("xf_k_step (fused pull+forward+gradient)", b_step, t_a), ("xf_k_update (optimizer over touched rows)", b_update, t_b)]
    else:
        kern = [("xf_k_step_lr_lazy (pull+forward+gradient+optimizer in one kernel)", b_step + b_update, t_a)]
    dom = max(kern, key=lambda k: k[2])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            import re
            kname = re.search(r"xf_k_\w+", dom[0]).group(0)
            traffic = json.load(open(tpath)).get(name, {}).get(kname)
        except Exception:
            traffic = None
    out["roofline"] = {
        "bound": "hbm", "kernel": dom[0], "achieved": dom[1] / dom[2] / 1e9 if dom[2] else None, "peak": peak, "unit": "GB/s",
        "frac": dom[1] / dom[2] / 1e9 / peak if dom[2] else None, "traffic": traffic,
        "traffic_source": (("ncu --set full capture of this workload (profiles/traffic.json)" if world == 1 else
                            "ncu --set full of the owner kernel with this workload's per-GPU token count on one GPU acting as "
                            "its own peer (profiles/traffic.json, profiles/r02_multigpu.md); S launches together")
                           if traffic else None),
        "peak_source": peak_src, "algorithmic_bytes_per_launch": dom[1], "avg_launch_ms": dom[2] * 1e3,
        "kernels": [{"kernel": n, "algorithmic_bytes": b, "avg_ms": t * 1e3, "gbs": b / t / 1e9 if t else None} for n, b, t in kern],
        "step_algorithmic_bytes": b_step + b_update, "step_gbs": (b_step + b_update) / (ms * 1e-3 / steps) / 1e9,
        "step_frac": (b_step + b_update) / (ms * 1e-3 / steps) / 1e9 / peak, "unique_keys_per_batch_per_gpu": U,
    }
    out.update({
        "value": world * B * steps / (ms * 1e-3), "unit": "examples/s", "ms_per_step": ms / steps,
        "gpu_launches": int(launches), "config": config_of(wl, world),
        "gpu": {"table_slots_per_gpu": table.capacity(), "table_row_bytes": table.row_bytes(), "table_keys_per_gpu": table.size(),
                "ring_batches": RING,
                "l2": "inputs larger than L2: %d distinct batches (%.0f MB of keys) cycled, table %.1f GB per GPU"
                      % (RING, RING * nnz * 8 / 1e6, table.capacity() * table.row_bytes() / 1e9)},
    })
    e2e_bin = {"value": world * B * steps / (ms_bin * 1e-3), "unit": "examples/s", "ms_per_step": ms_bin / steps,
               "h2d_bytes_per_step": (B + 1) * 4 + nnz * 4 + B, "d2h_bytes_per_step": 4,
               "api": "xf_trainer_step_host_ids_async (C ABI): page-locked host CSR of u32 feature ids, hashed to keys on the device"}
    if text:
        t, tf = allmax(text["pinned"]), allmax(text["file"])
        out["e2e"] = {"value": world * B / t, "unit": "examples/s", "ms_per_step": t * 1e3,
                      "h2d_bytes_per_step": text["text_bytes_per_step"], "d2h_bytes_per_step": 12,
                      "text_gbs_per_gpu": text["text_bytes_per_step"] / t / 1e9,
                      "api": "xf_trainer_ingest_begin / _end + xf_trainer_step_ingested (C ABI): the batch as TEXT in the "
                             "reference's format in page-locked host memory -> H2D of the raw text -> parse + hash + step on "
                             "the device; block i+2 is copied and block i+1 parsed while block i trains",
                      "from_file": {"value": world * B / tf, "unit": "examples/s", "ms_per_step": tf * 1e3,
                                    "api": "the same with xf_loader_next_raw forming each block from the text shard in the page "
                                           "cache (what the reference's fread + parser do per epoch)"},
                      "binary_ids": e2e_bin}
    else:
        out["e2e"] = e2e_bin
    out["_clock_windows"] = sampler_windows
    tr.close()
    table.close()
    del ring
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workloads", default="", help="comma list; default = the metric's LR config + extras")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-text-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps of each workload, write what its last step computed to DIR (one GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference_arm(args, WORKLOADS[MAIN])
        return

    import torch
    from xflow_b200 import api

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    if args.dump_outputs:
        if world > 1:
            raise SystemExit("--dump-outputs needs a single process: each rank's table holds only its key range")
        os.makedirs(args.dump_outputs, exist_ok=True)
    if api.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    comm = None
    dist = None
    if world == 1 and os.environ.get("XFLOW_MG_FORCE") == "1":
        comm = api.Comm(api.Comm.new_id(), 0, 1, local)   # profiling: the sharded step on one GPU (all keys local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        cid = torch.from_numpy(api.Comm.new_id() if rank == 0 else np.zeros(api.COMM_ID_BYTES, np.uint8)).cuda()
        dist.broadcast(cid, 0)
        comm = api.Comm(cid.cpu().numpy(), rank, world, local)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    if args.workloads:
        names = [w for w in args.workloads.split(",") if w]
    elif args.no_extras:
        names = [MAIN]
    elif world == 1:
        names = [MAIN, "headline_fm", "cfg2", "cfg3"]
    else:
        names = [MAIN, "headline_fm", "cfg4", "cfg5"]
    stream = torch.cuda.Stream()
    sampler = ClockSampler(local)
    sampler.start()
    res = {}
    for n in names:
        try:
            res[n] = run_workload(n, WORKLOADS[n], args, rank, world, local, comm, api, torch, stream, sampler, barrier, allmax)
        except Exception as ex:
            if n == names[0]:
                raise
            res[n] = {"error": repr(ex)}   # an extra that does not fit must not lose the main line
    sampler.stop_flag = True
    sampler.join(timeout=1.0)

    if rank == 0:
        main_res = res[names[0]]
        windows = []
        for r in res.values():
            windows += r.pop("_clock_windows", [])
        line = {
            "metric": "training examples/sec", "value": main_res["value"], "unit": "examples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": main_res["config"], "gpu": main_res["gpu"], "clocks": sampler.summary(windows),
            "e2e": main_res["e2e"], "gpu_launches": main_res["gpu_launches"], "roofline": main_res["roofline"],
            "extra": {k: v for k, v in res.items() if k != names[0]},
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                wl = WORKLOADS[names[0]]
                cores = os.cpu_count() or 1
                r = cpu_reference(wl, 16384, 3, cores, max(1, min(32, cores)))
                r1 = cpu_reference(wl, 4096, 1, 1, 1)
                line["cpu_baseline"] = {
                    "value": r["warm"], "unit": "examples/s", "cores": r["cores"], "kind": r["kind"],
                    "cold_table_value": r["cold"],
                    "single_core": {"value": r1["warm"], "cold_table_value": r1["cold"], "cores": 1, "rows": 4096},
                    "sample": "text shard of 16384 rows x %d nnz of the same workload: one cold epoch (empty table) then 3 epochs "
                              "on the warm table (`value`); text parse + update(); %s" % (wl["nnz"], r["how"])}
            except Exception as ex:  # the baseline is reported, never required for the GPU numbers
                line["cpu_baseline"] = {"value": None, "unit": "examples/s", "cores": 0, "kind": "port", "sample": "failed: %r" % (ex,)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        if comm is not None:
            comm.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
