"""Golden case table shared by make_golden.py (generation, needs the reference) and the tests."""

# name -> dict(data, model, opt, epochs, K, block_mb, preinit, latent_rows)
CASES = {
    "small_lr_ftrl_e10": dict(data="small", model="lr", opt="ftrl", epochs=10, K=0),
    "small_lr_ftrl_e60": dict(data="small", model="lr", opt="ftrl", epochs=60, K=0),
    "small_lr_sgd_e60": dict(data="small", model="lr", opt="sgd", epochs=60, K=0),
    "small_fm_sgd_k10_e60": dict(data="small", model="fm", opt="sgd", epochs=60, K=10),
    "small_fm_ftrl_k10_e5": dict(data="small", model="fm", opt="ftrl", epochs=5, K=10, preinit=True),
    "syn_lr_ftrl_e2": dict(data="syn", model="lr", opt="ftrl", epochs=2, K=0, block_mb=1),
    "syn_fm_sgd_k16_e1": dict(data="syn", model="fm", opt="sgd", epochs=1, K=16, block_mb=1),
    # v, nv, zv stored for a seeded sample of latent_rows keys (the whole table would not fit in 1 MB)
    "syn_fm_ftrl_k8_e1": dict(data="syn", model="fm", opt="ftrl", epochs=1, K=8, block_mb=1, preinit=True,
                              latent_rows=2048),
}

SYN = dict(seed=7, rows=3000, nnz_per_row=48, id_space=20000, dist="zipf", zipf_s=1.2)
SYN_TEST = dict(seed=8, rows=500, nnz_per_row=48, id_space=20000, dist="zipf", zipf_s=1.2)

# Reference runs on the syn shards (1 MB blocks) with the reference's own clock-seeded FM initialisation, the
# clock pinned to 1.5e9 s: (model, opt, K, epochs).  Stored for a sample of their keys, see ref_run_name.
REF_RUNS = [("lr", "ftrl", 0, 3), ("lr", "sgd", 0, 3), ("fm", "sgd", 6, 2), ("fm", "ftrl", 4, 2)]


def ref_run_name(model, opt, K, epochs):
    return "syn_refrng_%s_%s_k%d_e%d" % (model, opt, K, epochs)
