#!/usr/bin/env python
"""bench.py - samples/sec of one training step (fwd + loss + bwd + update) of the hot path on synthetic
batches of the BASELINE.json configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--config c2|c3|c4|c5|c2small|c3small|c4small] [--dist uniform|zipf] [--dump-outputs DIR]

Default = BASELINE.json configs[1] (C2: DeepFM, 26 tables x 1M rows, emb_dim 32, batch 65536 per GPU); c3 =
xDeepFM / CIN (128,128), emb_dim 16, batch 32768; c4 = DIN, 100k items, T=50, emb_dim 64, batch 8192; c5 =
DeepFM, 26 x 100M-row tables row-sharded over 8 GPUs (12.5M rows per table per GPU at any world size),
emb_dim 128, batch 32768 per GPU.

Prints ONE JSON line (see the task contract): `value` = device-timed whole-job samples/s with the batch
already resident in HBM; `e2e` = the same step through the public API (`Model.fit(host arrays)`) including the
pinned-H2D copy of the inputs and the D2H read of the loss; `roofline` = the dominant kernel group against the
measured peaks in MEASURED_PEAKS.json (ALGORITHMIC bytes / flops of SURVEY.md section 8(d) over CUDA-event
time); `cpu_baseline` = the CPU oracle (torch-CPU restatement of the reference math) on a bounded sample.
`--impl reference` times the reference's CPU path: real TensorFlow + the reference's deepctr under baseline/_ref if
importable, else the oracle port - on the SAME config, steps and warm-up.
`--dump-outputs DIR` writes what the last timed step left for its caller (see dump_outputs) as DIR/<name>.npy; the
inputs and initial weights are seeded, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HID = (256, 128, 64)
CONFIGS = {
    # BASELINE.json configs[1]
    "c2": dict(kind="deepfm", workload="DeepFM synthetic Criteo: 26 tables x 1M rows, emb_dim=32, batch=65536, 13 dense",
               n_sparse=26, n_dense=13, vocab=1000000, dim=32, batch=65536, hidden=HID),
    "c2small": dict(kind="deepfm", workload="DeepFM synthetic Criteo (small): 26 tables x 10k rows, emb_dim=32, batch=4096",
                    n_sparse=26, n_dense=13, vocab=10000, dim=32, batch=4096, hidden=HID),
    # BASELINE.json configs[2]
    "c3": dict(kind="xdeepfm", workload="xDeepFM (CIN layer_size=[128,128]) synthetic Criteo: 26 tables x 1M rows, "
                                        "emb_dim=16, batch=32768, 13 dense",
               n_sparse=26, n_dense=13, vocab=1000000, dim=16, batch=32768, hidden=HID, cin=(128, 128)),
    "c3small": dict(kind="xdeepfm", workload="xDeepFM (small): 26 tables x 10k rows, emb_dim=16, batch=2048, CIN (128,128)",
                    n_sparse=26, n_dense=13, vocab=10000, dim=16, batch=2048, hidden=HID, cin=(128, 128)),
    # BASELINE.json configs[3] (columns pinned by SURVEY.md section 8d)
    "c4": dict(kind="din", workload="DIN synthetic: 100k items, behaviour seq_len=50, emb_dim=64, batch=8192, att (80,40)",
               vocab=100001, dim=64, maxlen=50, batch=8192, hidden=HID, att=(80, 40), n_sparse=2, n_dense=1),
    "c4small": dict(kind="din", workload="DIN (small): 5k items, seq_len=50, emb_dim=64, batch=1024",
                    vocab=5001, dim=64, maxlen=50, batch=1024, hidden=HID, att=(80, 40), n_sparse=2, n_dense=1),
    # BASELINE.json configs[4]: V = 100M rows per table over 8 GPUs = 12.5M rows per table per GPU (weak)
    "c5": dict(kind="deepfm", workload="DeepFM synthetic Criteo: 26 tables x 100M rows row-sharded over 8 GPUs "
                                       "(12.5M rows per table per GPU), emb_dim=128, batch=32768 per GPU, 13 dense",
               n_sparse=26, n_dense=13, vocab_per_gpu=12500000, dim=128, batch=32768, hidden=HID),
    "c5small": dict(kind="deepfm", workload="C5-shaped (small): 26 tables x 200k rows per GPU, emb_dim=128, batch=8192 per GPU",
                    n_sparse=26, n_dense=13, vocab_per_gpu=200000, dim=128, batch=8192, hidden=HID),
}
LR = 0.01
N_BATCHES = 4      # distinct pre-generated batches cycled through the timed steps
METRIC = {"deepfm": "samples/sec fwd+bwd DeepFM Criteo-synth", "xdeepfm": "samples/sec fwd+bwd xDeepFM Criteo-synth",
          "din": "samples/sec fwd+bwd DIN synth"}


# ================================================================================================
# workloads: feature columns, model, synthetic data
# ================================================================================================
def resolve(cfg, world):
    cfg = dict(cfg)
    if "vocab_per_gpu" in cfg:
        cfg["vocab"] = cfg["vocab_per_gpu"] * world
    return cfg


def feature_columns(cfg, FC=None):
    if FC is None:
        from deepctr_b200 import feature_column as FC
    if cfg["kind"] == "din":
        V, E = cfg["vocab"], cfg["dim"]
        return [FC.SparseFeat("user", V, E), FC.SparseFeat("item_id", V, E), FC.DenseFeat("pay_score", 1),
                FC.VarLenSparseFeat(FC.SparseFeat("hist_item_id", V, E, embedding_name="item_id"),
                                    maxlen=cfg["maxlen"], length_name="seq_length")]
    cols = [FC.SparseFeat("C%d" % (i + 1), cfg["vocab"], cfg["dim"]) for i in range(cfg["n_sparse"])]
    cols += [FC.DenseFeat("I%d" % (i + 1), 1) for i in range(cfg["n_dense"])]
    return cols


def build_model(cfg, M=None, act=None):
    if M is None:
        from deepctr_b200 import models as M
    cols = feature_columns(cfg)
    if cfg["kind"] == "deepfm":
        return M.DeepFM(cols, cols, dnn_hidden_units=cfg["hidden"], l2_reg_linear=0, l2_reg_embedding=0, l2_reg_dnn=0)
    if cfg["kind"] == "xdeepfm":
        return M.xDeepFM(cols, cols, dnn_hidden_units=cfg["hidden"], cin_layer_size=cfg["cin"], l2_reg_linear=0,
                         l2_reg_embedding=0, l2_reg_dnn=0, l2_reg_cin=0)
    return M.DIN(cols, ["item_id"], dnn_hidden_units=cfg["hidden"], att_hidden_size=cfg["att"],
                 att_activation=act or "sigmoid", l2_reg_embedding=0, l2_reg_dnn=0)


class IdSampler(object):
    """uniform ids (worst case for the gather: no reuse; the roofline fraction is computed on these) or
    Zipf(s=1.05) truncated to the vocabulary (Criteo-like skew; SURVEY.md section 8d)."""

    def __init__(self, dist, vocab, rng):
        self.dist, self.vocab, self.rng = dist, vocab, rng
        self.cdf = None
        if dist == "zipf":
            w = 1.0 / np.arange(1, vocab + 1, dtype=np.float64) ** 1.05
            self.cdf = np.cumsum(w)
            self.cdf /= self.cdf[-1]

    def draw(self, shape, low=0):
        if self.cdf is None:
            return self.rng.randint(low, self.vocab, size=shape).astype(np.int32)
        r = np.searchsorted(self.cdf, self.rng.rand(*shape)).astype(np.int64)
        return np.minimum(r + low, self.vocab - 1).astype(np.int32)


def synth_batches(cfg, n, rank=0, dist="uniform", batch=None):
    """-> list of (dict feature name -> host array, labels); seed 2020 + rank; U(0,1) dense, Bernoulli(0.25) labels."""
    rng = np.random.RandomState(2020 + rank)
    B = batch or cfg["batch"]
    ids = IdSampler(dist, cfg["vocab"], rng)
    out = []
    for _ in range(n):
        if cfg["kind"] == "din":
            T = cfg["maxlen"]
            ln = rng.randint(1, T + 1, size=B).astype(np.int32)
            hist = ids.draw((B, T), low=1)
            hist[np.arange(T)[None, :] >= ln[:, None]] = 0
            x = {"user": ids.draw((B,)), "item_id": ids.draw((B,), low=1), "pay_score": rng.rand(B).astype(np.float32),
                 "hist_item_id": hist, "seq_length": ln}
        else:
            idm = ids.draw((B, cfg["n_sparse"]))
            dense = rng.rand(B, cfg["n_dense"]).astype(np.float32)
            x = {"C%d" % (i + 1): np.ascontiguousarray(idm[:, i]) for i in range(cfg["n_sparse"])}
            x.update({"I%d" % (i + 1): np.ascontiguousarray(dense[:, i]) for i in range(cfg["n_dense"])})
            x["__ids__"], x["__dense__"] = idm, dense
        y = (rng.rand(B) < 0.25).astype(np.float32)
        out.append((x, y))
    return out


def user_inputs(x):
    """what a user holds: one contiguous host array per feature."""
    return {k: v for k, v in x.items() if not k.startswith("__")}


def device_inputs(cfg, x, y, dev):
    """the same batch resident in HBM (per-feature views of one id matrix / one dense matrix for Criteo shapes)."""
    import torch
    if cfg["kind"] == "din":
        return {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in user_inputs(x).items()}, \
            torch.from_numpy(y).to(dev)
    ids_d, dense_d = torch.from_numpy(x["__ids__"]).to(dev), torch.from_numpy(x["__dense__"]).to(dev)
    xd = {"C%d" % (i + 1): ids_d[:, i:i + 1] for i in range(cfg["n_sparse"])}
    xd.update({"I%d" % (i + 1): dense_d[:, i:i + 1] for i in range(cfg["n_dense"])})
    return xd, torch.from_numpy(y).to(dev)


# ================================================================================================
# algorithmic bytes / flops per sample (SURVEY.md section 8d)
# ================================================================================================
def algorithmic(cfg):
    E = cfg["dim"]
    a = {}
    if cfg["kind"] == "din":
        T = cfg["maxlen"]
        att = [4 * E] + list(cfg["att"]) + [1]
        a["att_flops_fwd"] = T * 2 * sum(att[i] * att[i + 1] for i in range(len(att) - 1))      # 2 372 000 at C4
        a["att_bytes"] = T * E * 4 + 2 * E * 4 + T * 4
        dims = [3 * E + 1] + list(cfg["hidden"]) + [1]
        a["dnn_flops_fwd"] = 2 * sum(dims[i] * dims[i + 1] for i in range(len(dims) - 1))
        a["gather_fwd_bytes"] = (T + 2) * 4 + (T + 2) * E * 4 * 2
        return a
    F, nd = cfg["n_sparse"], cfg["n_dense"]
    a["gather_fwd_bytes"] = F * 4 + F * E * 4 + F * E * 4 + F * 4                     # 6864 at C2 (6760 + 104)
    a["scatter_bwd_bytes"] = F * 4 + F * E * 4 + 2 * F * E * 4 + 2 * F * 4            # 10296 at C2 (10088 + 208)
    a["scatter_extra_read_bytes"] = F * E * 4        # the X re-read of the fused FM Jacobian: traffic, not algorithm
    dims = [F * E + nd] + list(cfg["hidden"]) + [1]
    a["dnn_flops_fwd"] = 2 * sum(dims[i] * dims[i + 1] for i in range(len(dims) - 1))
    if cfg["kind"] == "xdeepfm":
        m, h, fl = F, F, 0
        for i, n in enumerate(cfg["cin"]):
            fl += 2 * E * (m * h) * n
            h = n // 2 if i != len(cfg["cin"]) - 1 else n
        a["cin_flops_fwd"] = fl                                                       # 9 584 640 at C3
    return a


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                r = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if r.returncode == 0 and r.stdout.strip():
                    self.rows.append([c.strip() for c in r.stdout.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active")
                                                         for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "which": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "which": "fallback"}


def timed_alone(fn, reps=5, flush=None):
    """median CUDA-event duration (us) of fn() launched alone after an L2 flush."""
    import torch
    fn()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def gemm_launch_times(dims, B, precision, dev, reps=5):
    """CUDA-event duration of every GEMM launch of an MLP tower (forward / dgrad / wgrad per layer, operands as
    ops.dense passes them: pre-split planes in bf16x3 mode), each timed alone after an L2 flush.
    Returns [(label, m, n, k, us)]."""
    import torch
    from deepctr_b200 import _lib as L, kernels as K, ops
    prec = L.GEMM_BF16X3 if precision == "bf16x3" else L.GEMM_FP32
    flush = torch.empty(192 << 20, dtype=torch.uint8, device=dev)
    out = []
    for li in range(len(dims) - 1):
        kin, nout = dims[li], dims[li + 1]
        ld = (kin + 3) // 4 * 4
        xw = torch.randn((B, ld), device=dev)
        x, w, dz = xw[:, :kin], torch.randn((kin, nout), device=dev), torch.randn((B, nout), device=dev)
        pl = (lambda t: K.split_planes(t)) if prec == L.GEMM_BF16X3 else (lambda t: None)
        xp, wp, dzp = pl(x), pl(w), pl(dz)
        dxw = torch.empty((B, ld), device=dev)
        calls = [
            ("fwd", B, nout, kin, lambda: K.gemm(x, w, precision=prec, m=B, n=nout, k=kin, a_planes=xp, b_planes=wp)),
            ("dgrad", B, kin, nout, lambda: K.gemm(dz, w, c=dxw[:, :kin], trans_b=True, precision=prec, m=B, n=kin,
                                                   k=nout, a_planes=dzp, b_planes=wp)),
            ("wgrad", kin, nout, B, lambda: K.gemm(x, dz, trans_a=True, precision=prec,
                                                   split_k=ops._split_k(kin, nout, B), m=kin, n=nout, k=B,
                                                   a_planes=xp, b_planes=dzp)),
        ]
        for name, m, n, k, fn in calls:
            out.append(("%s %d->%d" % (name, kin, nout), m, n, k, timed_alone(fn, reps, flush)))
    return out


def op_alone_us(make, reps=5):
    """fwd + bwd of one differentiable op captured as a CUDA graph and replayed alone after an L2 flush (a group of
    many launches timed eagerly would measure the host's launch gaps)."""
    import torch
    from deepctr_b200 import engine as E
    dev = torch.device("cuda", torch.cuda.current_device())
    flush = torch.empty(192 << 20, dtype=torch.uint8, device=dev)

    def run():
        tape = E.Tape()
        with E.recording(tape):
            out, seed = make()
        out.requires_grad = True
        E.add_grad(out, seed)
        tape.backward()
    run()
    run()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run()
    return timed_alone(g.replay, reps, flush)


DUMP_ROWS = 2048          # rows kept per embedding table by --dump-outputs
DUMP_LIMIT = 64 << 20     # bytes


def dump_outputs(out_dir, loss_sum, model):
    """Write, as float32 .npy files, what a training step leaves for its caller: the summed batch loss
    train_step returned (loss_sum.npy) and every weight it trained (<weight name with '/' as '.'>.npy).
    Tables with more than DUMP_ROWS rows are cut to a fixed, seeded sample of DUMP_ROWS rows (the same
    rows in every run) so that the files stay below DUMP_LIMIT bytes.  Under several GPUs these are
    rank 0's weights, i.e. its shard of each row-sharded table."""
    import torch
    arrays = {"loss_sum": loss_sum.detach().reshape(-1).cpu().numpy()}
    rng = np.random.RandomState(0)
    for w in model.weights:
        t = w.data
        if t is None:
            continue
        if t.dim() >= 1 and t.shape[0] > DUMP_ROWS:
            rows = np.sort(rng.choice(t.shape[0], DUMP_ROWS, replace=False))
            t = t.index_select(0, torch.from_numpy(rows).to(t.device))
        arrays[w.name.replace("/", ".")] = t.detach().cpu().numpy().astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes (limit %d)" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ================================================================================================
# CPU arm: the reference math on host cores
# ================================================================================================
def cpu_step_factory(cfg, threads):
    """One SGD step of the oracle (oracle/ops.py: the reference's layer math restated on torch-CPU): fwd + BCE +
    autograd bwd + row-wise SGD on the gathered rows (the reference's dense-Adam-over-tables semantics, SURVEY.md
    App. C, cannot run at these table sizes on any hardware)."""
    import torch
    from oracle import ops as O
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(1024)
    E, V = cfg["dim"], cfg["vocab"]

    def glorot(a, b):
        return (torch.randn(a, b, generator=g) * (2.0 / (a + b)) ** 0.5).requires_grad_()

    def tower(d0):
        dims = [d0] + list(cfg["hidden"])
        return ([glorot(dims[i], dims[i + 1]) for i in range(len(dims) - 1)],
                [torch.zeros(d, requires_grad=True) for d in dims[1:]], glorot(dims[-1], 1))

    def sgd(params):
        with torch.no_grad():
            for p in params:
                p -= LR * p.grad
                p.grad = None

    if cfg["kind"] == "din":
        T = cfg["maxlen"]
        t_user, t_item = torch.randn(V, E, generator=g) * 1e-2, torch.randn(V, E, generator=g) * 1e-2
        ks, bs, wd = tower(3 * E + 1)
        att = [4 * E] + list(cfg["att"])
        lau = {"dnn_kernels": [glorot(att[i], att[i + 1]) for i in range(len(att) - 1)],
               "dnn_biases": [torch.zeros(d, requires_grad=True) for d in att[1:]],
               "kernel": glorot(att[-1], 1), "bias": torch.zeros(1, requires_grad=True)}
        gb = torch.zeros(1, requires_grad=True)
        dense_params = ks + bs + [wd, gb, lau["kernel"], lau["bias"]] + lau["dnn_kernels"] + lau["dnn_biases"]

        def step(x, y):
            iu = torch.from_numpy(x["user"].astype(np.int64))
            ii = torch.from_numpy(x["item_id"].astype(np.int64))
            ih = torch.from_numpy(x["hist_item_id"].astype(np.int64))
            ru = O.embedding_lookup(t_user, iu.reshape(-1, 1)).detach().requires_grad_()
            ri = O.embedding_lookup(t_item, ii.reshape(-1, 1)).detach().requires_grad_()
            rh = O.embedding_lookup(t_item, ih).detach().requires_grad_()
            hist = O.attention_sequence_pooling(ri, rh, ih != 0, lau, "sigmoid", False)
            xin = torch.cat([ru, ri, hist], dim=-1).flatten(1)
            xin = torch.cat([xin, torch.from_numpy(x["pay_score"]).reshape(-1, 1)], dim=-1)
            logit = O.dnn(xin, ks, bs, "relu") @ wd
            loss = O.binary_crossentropy(y, O.prediction(logit, gb, "binary"))
            loss.backward()
            sgd(dense_params)
            with torch.no_grad():
                t_user.index_add_(0, iu, ru.grad[:, 0, :], alpha=-LR)
                t_item.index_add_(0, ii, ri.grad[:, 0, :], alpha=-LR)
                t_item.index_add_(0, ih.reshape(-1), rh.grad.reshape(-1, E), alpha=-LR)
            return float(loss)
        return step

    F, nd = cfg["n_sparse"], cfg["n_dense"]
    tables = [torch.randn(V, E, generator=g) * 1e-2 for _ in range(F)]
    lin = [torch.zeros(V, 1) for _ in range(F)]
    ks, bs, wd = tower(F * E + nd)
    wl = glorot(nd, 1)
    gb = torch.zeros(1, requires_grad=True)
    dense_params = ks + bs + [wd, wl, gb]
    cin_w = None
    if cfg["kind"] == "xdeepfm":
        filters, cbias, h, width = [], [], F, 0
        for i, n in enumerate(cfg["cin"]):
            filters.append((torch.randn(1, F * h, n, generator=g) * (2.0 / (F * h + n)) ** 0.5).requires_grad_())
            cbias.append(torch.zeros(n, requires_grad=True))
            last = i == len(cfg["cin"]) - 1
            width += n if last else n // 2
            h = n if last else n // 2
        cin_w = (filters, cbias, glorot(width, 1))
        dense_params += filters + cbias + [cin_w[2]]

    def step(x, y):
        idx = torch.from_numpy(x["__ids__"].astype(np.int64))
        rows = [O.embedding_lookup(tables[f], idx[:, f]).detach().requires_grad_() for f in range(F)]
        lrows = [O.embedding_lookup(lin[f], idx[:, f]).detach().requires_grad_() for f in range(F)]
        xe = torch.cat(rows, dim=1)
        d = torch.from_numpy(x["__dense__"])
        logit = O.linear(torch.cat(lrows, dim=-1), d, wl)
        h = O.dnn(torch.cat([xe.flatten(1), d], dim=-1), ks, bs, "relu")
        logit = logit + h @ wd
        if cin_w is None:
            logit = logit + O.fm(xe)
        else:
            logit = logit + O.cin(xe, cin_w[0], cin_w[1], tuple(cfg["cin"]), "relu", True) @ cin_w[2]
        loss = O.binary_crossentropy(y, O.prediction(logit, gb, "binary"))
        loss.backward()
        sgd(dense_params)
        with torch.no_grad():
            for f in range(F):
                tables[f].index_add_(0, idx[:, f], rows[f].grad[:, 0, :], alpha=-LR)
                lin[f].index_add_(0, idx[:, f], lrows[f].grad[:, 0, :], alpha=-LR)
        return float(loss)

    return step


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def run_cpu(cfg, steps, warmup, batch, dist):
    """oracle port: `warmup` + `steps` steps of `batch` samples with the best torch intra-op pool size."""
    import torch
    avail = host_cores()
    step = cpu_step_factory(cfg, avail)
    data = synth_batches(cfg, 2, 0, dist, batch=batch)
    # torch's intra-op pool stops scaling far below the core count of a big host for these op sizes: probe
    best, threads = None, avail
    for cand in sorted(set(min(avail, c) for c in (8, 16, 32, 64, avail))):
        torch.set_num_threads(cand)
        step(*data[0])
        t0 = time.perf_counter()
        step(*data[1])
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, threads = dt, cand
    torch.set_num_threads(threads)
    for i in range(warmup):
        step(*data[i % 2])
    t0 = time.perf_counter()
    for i in range(steps):
        step(*data[i % 2])
    dt = time.perf_counter() - t0
    return steps * batch / dt, dt / steps * 1e3, threads


def run_tensorflow(cfg, steps, warmup, batch, dist):
    """The real thing, when it can be imported: TensorFlow + the UNMODIFIED reference package (baseline/_ref)
    - model.train_on_batch on the same synthetic batches, SGD, l2 = 0, all host cores.
    Returns None when TensorFlow / the reference cannot be imported (this image: always)."""
    try:
        import tensorflow as tf                                   # noqa: F401
    except Exception:
        return None
    p = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(p, "deepctr")) and p not in sys.path:
        sys.path.insert(0, p)
    try:
        from deepctr import models as RM, feature_column as RFC
    except Exception:
        return None
    tf.config.set_visible_devices([], "GPU")
    cols = feature_columns(cfg, RFC)
    if cfg["kind"] == "din":
        model = RM.DIN(cols, ["item_id"], dnn_hidden_units=cfg["hidden"], att_hidden_size=cfg["att"],
                       att_activation="sigmoid", l2_reg_embedding=0, l2_reg_dnn=0)
    elif cfg["kind"] == "xdeepfm":
        model = RM.xDeepFM(cols, cols, dnn_hidden_units=cfg["hidden"], cin_layer_size=cfg["cin"], l2_reg_linear=0,
                           l2_reg_embedding=0, l2_reg_dnn=0, l2_reg_cin=0)
    else:
        model = RM.DeepFM(cols, cols, dnn_hidden_units=cfg["hidden"], l2_reg_linear=0, l2_reg_embedding=0, l2_reg_dnn=0)
    model.compile(tf.keras.optimizers.SGD(LR), "binary_crossentropy")
    data = [(user_inputs(x), y) for x, y in synth_batches(cfg, 2, 0, dist, batch=batch)]
    for i in range(warmup):
        model.train_on_batch(*data[i % 2])
    t0 = time.perf_counter()
    for i in range(steps):
        model.train_on_batch(*data[i % 2])
    dt = time.perf_counter() - t0
    return steps * batch / dt, dt / steps * 1e3, host_cores()


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b2ctr", choices=["b2ctr", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--dist", default="uniform", choices=["uniform", "zipf"])
    ap.add_argument("--precision", default=os.environ.get("B2CTR_GEMM", "auto"))
    ap.add_argument("--din-act", default="sigmoid", choices=["sigmoid", "dice"])
    ap.add_argument("--cpu-sample-batch", type=int, default=8192)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b2ctr":
        ap.error("--dump-outputs applies to --impl b2ctr")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = resolve(CONFIGS[args.config], world)
    warmup = max(args.warmup, 3)
    metric = METRIC[cfg["kind"]]

    if args.impl == "reference":
        # the reference's own CPU path on this box's host cores, same config / steps / warm-up as the b2ctr arm;
        # rank 0 alone runs it.  C5 tables (1.3 TB) cannot exist on a host: that config reports unavailable.
        if rank != 0:
            return
        if "vocab_per_gpu" in cfg and cfg["vocab"] * cfg["n_sparse"] * cfg["dim"] * 4 > 48e9:
            print(json.dumps({"impl": "reference", "unavailable": "the %s tables (%.0f GB) do not fit host memory"
                              % (args.config, cfg["vocab"] * cfg["n_sparse"] * cfg["dim"] * 4 / 1e9)}))
            return
        B = cfg["batch"]
        tf_run = run_tensorflow(cfg, args.steps, warmup, B, args.dist)
        kind = "reference" if tf_run is not None else "port"
        v, ms, threads = tf_run if tf_run is not None else run_cpu(cfg, args.steps, warmup, B, args.dist)
        how = ("TensorFlow + the unmodified reference package, model.train_on_batch" if tf_run is not None else
               "oracle port = torch-CPU restatement of the reference layer math (tried `import tensorflow` first: "
               "not installable in this image, no network)")
        line = {"impl": "reference", "metric": metric, "value": v, "unit": "samples/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": cfg["workload"], "global_batch": B, "optimizer": "sgd", "dist": args.dist,
                           "note": "CPU arm (no GPU is used; n_gpus echoes the launch): " + how},
                "cpu_baseline": {"value": v, "unit": "samples/s", "cores": threads, "kind": kind,
                                 "sample": "%d steps x %d samples (the full per-GPU batch) of the %s workload"
                                           % (args.steps, B, args.config)},
                "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the b2ctr path has no CPU fallback "
                         "(use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from deepctr_b200 import _lib as L, kernels as K, ops
    from deepctr_b200.engine import SGD

    precision = args.precision
    if precision == "auto":
        precision = "bf16x3"
    ops.set_gemm_precision(precision)
    model = build_model(cfg, act=args.din_act)
    # the builders leave the output Dense's initializer unseeded, as the reference does; seed it so that every
    # run starts from the same weights
    for i, w in enumerate(model.weights):
        if getattr(w.initializer, "seed", 0) is None:
            w.initializer.seed = i
    model.compile(SGD(LR), "binary_crossentropy", embedding_update="sparse")
    host = synth_batches(cfg, N_BATCHES, rank, args.dist)
    dev = torch.device("cuda", local_rank)
    dev_batches = [device_inputs(cfg, x, y, dev) for x, y in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ------------------------------------------------------------------
    # warm-up: >= `warmup` steps, extended until every distinct batch has its step graph captured (the
    # model replays the whole training step as one CUDA graph per input-buffer set once warm)
    i = 0
    while i < warmup or (i < warmup + N_BATCHES + 4 and model._graph_eligible()
                         and len(model._step_graphs) < N_BATCHES):
        model.train_step(*dev_batches[i % N_BATCHES])
        i += 1
    warmup_done = i
    barrier()
    L.reset_launch_count()
    model.replayed_launches = 0
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        loss_sum = model.train_step(*dev_batches[(warmup_done + i) % N_BATCHES])
    e1.record()
    barrier()
    launches = L.launch_count() + model.replayed_launches
    graph_replays = args.steps if model._step_graphs else 0
    sampler.stop_flag = True
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss_sum, model)
    # per-kernel durations: the same K steps once more, launched eagerly with a CUDA-event pair around every
    # kernel group (the timed region above replays graphs, which cannot carry per-kernel events)
    K.PROFILE = {}
    for i in range(args.steps):
        model.train_step(*dev_batches[(warmup_done + i) % N_BATCHES])
    torch.cuda.synchronize()
    prof = K.profile_summary()
    K.PROFILE = None
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    B = cfg["batch"]
    value = world * B * args.steps / (ms / 1e3)

    # ---- end-to-end through the public API: host arrays in, loss out -------------------------------
    # model.fit(x, y, batch_size=B) over `steps` batches of host arrays: every step packs its inputs into
    # pinned staging buffers, copies them H2D and reads its loss back D2H (asynchronously; the host waits
    # once per epoch, as Keras' fit does between epochs).
    e2e = None
    if not args.no_e2e:
        reps = (args.steps + N_BATCHES - 1) // N_BATCHES
        n_tot = args.steps * B
        host_x = {k: np.concatenate([user_inputs(h[0])[k] for h in host] * reps)[:n_tot] for k in user_inputs(host[0][0])}
        host_y = np.concatenate([h[1] for h in host] * reps)[:n_tot]
        warm = {k: v[:3 * B] for k, v in host_x.items()}
        model.fit(warm, host_y[:3 * B], batch_size=B, epochs=1, shuffle=False, verbose=0)
        model._feeder.h2d_bytes = 0
        model.d2h_bytes = 0
        barrier()
        e0.record()
        model.fit(host_x, host_y, batch_size=B, epochs=1, shuffle=False, verbose=0)
        e1.record()
        barrier()
        e2e_ms = e0.elapsed_time(e1)
        t = torch.tensor([e2e_ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
        e2e = {"value": world * B * args.steps / (e2e_ms / 1e3), "unit": "samples/s",
               "h2d_bytes_per_step": int(model._feeder.h2d_bytes // args.steps),
               "d2h_bytes_per_step": int(model.d2h_bytes // args.steps), "ms_per_step": e2e_ms / args.steps,
               "api": "Model.fit(host arrays, batch_size=%d)" % B}

    alg = algorithmic(cfg)
    peaks = measured_peaks()
    F, E, nd = cfg["n_sparse"], cfg["dim"], cfg["n_dense"]
    # isolation-timed launches of the dominant GEMM-shaped groups (rank 0)
    gemm_times, group_us = [], {}
    if rank == 0:
        if cfg["kind"] == "din":
            dims = [3 * E + 1] + list(cfg["hidden"])
        else:
            dims = [F * E + nd] + list(cfg["hidden"])
        gemm_times = gemm_launch_times(dims, B, precision, dev)
        if cfg["kind"] == "xdeepfm":
            from deepctr_b200 import engine as EN
            xin = torch.randn((B, F, E), device=dev) * 0.1
            cin_layer = [l for l in model.layers if type(l).__name__ == "CIN"][0]

            def make_cin():
                v = EN.Var(xin, requires_grad=True)
                out = ops.cin(v, cin_layer.filters, cin_layer.bias, cin_layer.layer_size, cin_layer.activation,
                              cin_layer.split_half)
                return out, torch.ones_like(out.data)
            group_us["cin"] = op_alone_us(make_cin)
        if cfg["kind"] == "din":
            from deepctr_b200 import engine as EN
            T = cfg["maxlen"]
            att_layer = [l for l in model.layers if type(l).__name__ == "AttentionSequencePoolingLayer"][0]
            qd = torch.randn((B, 1, E), device=dev) * 0.1
            kd = torch.randn((B, T, E), device=dev) * 0.1
            idd = torch.from_numpy(host[0][0]["hist_item_id"]).to(dev)

            def make_att():
                q, k = EN.Var(qd, requires_grad=True), EN.Var(kd, requires_grad=True)
                k.mask = EN.KMask(ids=[idd])
                out = att_layer._invoke([q, k], True)
                return out, torch.ones_like(out.data)
            group_us["din_att"] = op_alone_us(make_att)
    if world > 1:
        model.close()          # step graphs hold NCCL kernels, the planner holds IPC mappings of peer shards
        dist.barrier()
    if rank != 0:
        sys.stdout.flush()
        os._exit(0)

    kernels = {name: {"launches": count, "ms_per_step": total_ms / args.steps} for name, (count, total_ms) in prof.items()}

    def frac_hbm(name, bytes_per_sample, extra=None):
        if name not in prof or prof[name][0] == 0 or not bytes_per_sample:
            return None
        avg_ms = prof[name][1] / prof[name][0]
        a = bytes_per_sample * B / (avg_ms * 1e-3) / 1e9
        r = {"bound": "hbm", "achieved": a, "peak": peaks["hbm_gbs"], "unit": "GB/s",
             "frac": a / peaks["hbm_gbs"], "traffic": None, "kernel": name,
             "avg_launch_ms": avg_ms, "peak_source": peaks["which"] + " (copy bandwidth)",
             "algorithmic_bytes_per_launch": bytes_per_sample * B,
             "timed": "CUDA events around the launch inside an eagerly launched step (dist=%s)" % args.dist}
        if extra:
            r.update(extra)
        return r
    roof_gather = frac_hbm("embed_gather_uniform_fwd", alg.get("gather_fwd_bytes"))
    roof_scatter = frac_hbm("embed_scatter_uniform_bwd", alg.get("scatter_bwd_bytes"),
                            {"design_extra_read_bytes_per_launch": alg.get("scatter_extra_read_bytes", 0) * B,
                             "note": "algorithmic bytes are SURVEY.md 8(d)'s (ids + dOut + row read-modify-write + linear); "
                                     "the fused FM Jacobian re-reads X, which counts as traffic, not as algorithm"})
    # DRAM bytes per launch from committed `ncu --set full` captures of this workload (a static file, NOT measured
    # by this run: see profiles/README.md for the capture commands)
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and world == 1 and args.dist == "uniform":
        traffic = json.load(open(tpath)).get(args.config, {})
        for r in (roof_gather, roof_scatter):
            if r is not None and r["kernel"] in traffic:
                r["traffic"] = traffic[r["kernel"]]
                r["traffic_source"] = "static: profiles/traffic.json (ncu --set full capture)"

    def tensor_roof(name, flops, us, launches, note, per_launch=None):
        a = flops / (us * 1e-6) / 1e12
        r = {"bound": "tensor", "achieved": a, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
             "frac": a / peaks["bf16_tflops"], "traffic": None, "kernel": name, "launches_per_step": launches,
             "avg_launch_ms": us / max(launches, 1) / 1e3, "algorithmic_flops_per_step": flops,
             "tensor_pipe_frac": (3.0 if precision == "bf16x3" else 1.0) * a / peaks["bf16_tflops"],
             "note": note, "peak_source": peaks["which"] + " (dense bf16, BURST: launches timed alone after an L2 flush)"}
        if per_launch:
            r["per_launch_us"] = per_launch
        return r
    roof_gemm = None
    if gemm_times:
        flops = sum(2.0 * m * n * k for _, m, n, k, _ in gemm_times)
        us = sum(t for *_, t in gemm_times)
        roof_gemm = tensor_roof("gemm_planes_ws_kernel (tcgen05 cta_group::2, split-bf16)" if precision == "bf16x3"
                                else "sgemm_kernel (fp32 FFMA)", flops, us, len(gemm_times),
                                "achieved = 2*M*N*K algorithmic flops / CUDA-event launch time; bf16x3 issues 3 bf16 MMAs "
                                "per fp32 product, so frac <= 1/3 and tensor_pipe_frac = 3 x frac",
                                {lab: round(t, 1) for lab, _, _, _, t in gemm_times})
    roof_group = None
    if "cin" in group_us:
        roof_group = tensor_roof("CIN fwd+bwd (ops.cin: outer product + filter contraction)", 3.0 * alg["cin_flops_fwd"] * B,
                                 group_us["cin"], sum(v[0] for k, v in prof.items() if k.startswith("cin:")) // args.steps,
                                 "algorithmic flops = 3 x forward (dZ*W^T and Z^T*dZ in the backward); the backward "
                                 "RECOMPUTES the outer product, which is not counted; graph-replayed alone")
    if "din_att" in group_us:
        roof_group = tensor_roof("DIN local-attention fwd+bwd (AttentionSequencePoolingLayer)", 3.0 * alg["att_flops_fwd"] * B,
                                 group_us["din_att"], sum(v[0] for k, v in prof.items() if k.startswith("din_att:")) // args.steps,
                                 "algorithmic flops = 3 x forward MLP flops T*2*(4E*80+80*40+40); graph-replayed alone")
    group_ms = {tag: sum(v[1] for k, v in prof.items() if k.startswith(tag + ":")) / args.steps for tag in ("cin", "din_att")}
    gemm_ms = sum(v[1] for k, v in prof.items() if k == "gemm")
    shares = {"gather+scatter_ms": sum(prof.get(k, (0, 0))[1] for k in ("embed_gather_uniform_fwd", "embed_scatter_uniform_bwd",
                                                                          "embed_gather_fwd", "embed_scatter_add")) / args.steps,
              "dnn_gemm_ms": (sum(t for *_, t in gemm_times) / 1e3) if gemm_times else gemm_ms / args.steps,
              "group_ms_alone": {k: v / 1e3 for k, v in group_us.items()},
              "group_ms_eager_with_launch_gaps": group_ms, "step_ms": ms_per_step,
              "measured": "eager pass of the same %d steps with a CUDA-event pair per kernel wrapper" % args.steps}
    cands = [(shares["gather+scatter_ms"], max([r for r in (roof_gather, roof_scatter) if r], key=lambda r: r["avg_launch_ms"],
                                                default=None)),
             (shares["dnn_gemm_ms"], roof_gemm)]
    if roof_group is not None:
        cands.append((list(group_us.values())[0] / 1e3, roof_group))
    cands = [c for c in cands if c[1] is not None]
    dominant = max(cands, key=lambda c: c[0])[1] if cands else None

    cpu = None
    if not args.no_cpu_baseline and world == 1:      # rank 0 at N = 1 only (the N > 1 lines carry null)
        sb = min(args.cpu_sample_batch, B)
        v, cms, threads = run_cpu(cfg, 4, 1, sb, args.dist)
        cpu = {"value": v, "unit": "samples/s", "cores": threads, "kind": "port",
               "sample": "4 steps x %d samples of the same workload (oracle port, torch-CPU)" % sb}

    step_bytes = (alg.get("gather_fwd_bytes", 0) + alg.get("scatter_bwd_bytes", 0)) * B / 1e9
    line = {"metric": metric, "value": value, "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config, "global_batch": world * B,
                       "optimizer": "sgd (fused row-wise)", "dist": args.dist, "gemm_precision": precision,
                       "parallelism": ("tables row-sharded over %d GPUs (%s), dense part data-parallel" %
                                       (world, "NVLink peer loads / red.add" if getattr(model.planner, "peer_mode", False)
                                        else "NCCL all-to-all")) if world > 1 else "1 gpu",
                       "l2_flush": "none: %d distinct batches cycle; per step the path touches %.2f GB of "
                                   "randomly addressed table rows + activations, >> 126 MB L2" % (N_BATCHES, step_bytes)},
            "e2e": e2e, "gpu_launches": int(launches), "graph_replays": int(graph_replays), "clocks": sampler.summary(),
            "roofline": dominant, "roofline_gather_fwd": roof_gather, "roofline_scatter_bwd": roof_scatter,
            "roofline_gemm": roof_gemm, "roofline_group": roof_group, "kernel_ms_per_step": kernels, "shares": shares,
            "cpu_baseline": cpu}
    print(json.dumps(line))
    sys.stdout.flush()
    if world > 1:
        os._exit(0)            # all ranks passed the barrier above; skip collective teardown at exit


if __name__ == "__main__":
    main()
