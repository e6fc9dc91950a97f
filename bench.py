#!/usr/bin/env python
"""bench.py — CTR samples/sec, forward+backward, batch 65 536 per GPU (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload deepfm|xdeepfm|fibinet|dcn] [--dump-outputs DIR]
    python bench.py --impl reference ...        # the reference algorithm on the host cores (oracle port)

With the same arguments every run sees the same seeded weights and batches, so the arrays --dump-outputs writes
(see dump_outputs) compare two builds of the project output for output.

A step = one pass of the hot path over one synthetic Criteo-shaped batch:
X[B,39] -> fused gather (+linear, FM) -> interaction + tower -> sigmoid -> BCE(sum) -> backward down
to per-unique-row table gradients.  No optimizer step (the metric is fwd+bwd), l2 = 0 on both arms.

Printed JSON (one line, rank 0): see the task contract — `value` (device-resident inputs, CUDA
events), `e2e` (pinned host X/y copied in, loss read back, every step), `roofline` of the dominant
kernel (CUDA events around its C-ABI entry point in a separate instrumented pass), `cpu_baseline`
(the oracle port timed on this box's host cores, bounded sample), `clocks`, `gpu_launches`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)
REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))

B_PER_GPU = 65536
N_ROTATE = 8          # distinct pre-generated batches: 8 x 109 MB of gathered rows cannot sit in L2

WORKLOADS = {
    # BASELINE.json configs[1..3] + the DCN model the north star names (SURVEY.md §8d)
    "deepfm": dict(model="DeepFM", D=16, B=65536, kw=dict(dnn_hidden_units=[256, 128]),
                   desc="DeepFM 26 sparse x 1M x 16 + 13 dense, DNN (256,128), batch 65536"),
    "xdeepfm": dict(model="xDeepFM", D=16, B=65536,
                    kw=dict(dnn_hidden_units=[256, 256], cin_layer_size=[128, 128], cin_split_half=True),
                    desc="xDeepFM CIN (128,128) split_half, DNN (256,256), batch 65536"),
    "fibinet": dict(model="FiBiNET", D=32, B=32768, kw=dict(bilinear_type="interaction", dnn_hidden_units=[128, 128]),
                    desc="FiBiNET bilinear interaction, 26 sparse dim 32, DNN (128,128), batch 32768"),
    "dcn": dict(model="DCN", D=16, B=65536, kw=dict(cross_num=2, cross_parameterization="vector",
                                                    dnn_hidden_units=[128, 128], l2_reg_cross=0),
                desc="DCN vector x2, DNN (128,128), batch 65536"),
}


def make_cfg(workload, vocab=1000000):
    from oracle import ctr_oracle as O
    w = WORKLOADS[workload]
    cols = [O.sparse_col("C%d" % (i + 1), vocab, w["D"]) for i in range(26)] + \
           [O.dense_col("I%d" % (i + 1)) for i in range(13)]
    return O.make_cfg(w["model"], cols, cols, init_std=0.05, l2_reg_linear=0, l2_reg_embedding=0, **w["kw"])


def algorithmic_bytes_per_sample(D, F=26, C=39):
    """SURVEY.md §8d: each input read once, each output/grad written once:
    4*(C_X + 2*F*(D+1) + 2) bytes per sample (3700 B at D=16)."""
    return 4 * (C + 2 * F * (D + 1) + 2)


def tensor_flops_per_sample(cfg):
    kw = cfg["kwargs"]
    D = cfg["dnn_columns"][0]["dim"]
    F = 26
    in_dim = F * D + 13
    fl = 0
    hidden = list(kw.get("dnn_hidden_units", []))
    if cfg["model"] == "FiBiNET":
        in_dim = F * (F - 1) * D + 13
        fl += 2 * 325 * (2 * D * D)
    prev = in_dim
    for h in hidden:
        fl += 2 * prev * h
        prev = h
    fl += 2 * prev
    if cfg["model"] == "xDeepFM":
        H = F
        sizes = kw["cin_layer_size"]
        for i, n in enumerate(sizes):
            fl += 2 * D * n * H * F
            H = n // 2 if (kw.get("cin_split_half", True) and i != len(sizes) - 1) else n
    if cfg["model"] == "DCN":
        fl += 2 * (F * D + 13) * 2 * kw.get("cross_num", 2)
    return 3 * fl          # backward = 2x forward


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    """(HBM GB/s, bf16 burst TF/s, bf16 sustained TF/s, source)"""
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return (d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0),
                "measured (MEASURED_PEAKS.json)")
    return 6650.0, 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


def measured_traffic():
    """DRAM bytes per launch of the entry points' dominant kernels, from the committed
    `ncu --set full` capture (profiles/traffic.json: {entry point: dram bytes read + written})."""
    path = os.path.join(REPO, "profiles", "traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return {}


def entry_flops_per_sample(cfg):
    """fp32-equivalent FLOPs per sample of each GEMM-shaped C-ABI entry point (forward; backward = 2x)."""
    kw = cfg["kwargs"]
    D = cfg["dnn_columns"][0]["dim"]
    F = 26
    in_dim = F * D + 13
    if cfg["model"] == "FiBiNET":
        in_dim = F * (F - 1) * D + 13
    dnn = 0
    prev = in_dim
    for h in kw.get("dnn_hidden_units", []):
        dnn += 2 * prev * h
        prev = h
    out = {"ctr_dnn_layer_fwd": float(dnn), "ctr_dnn_layer_bwd": 2.0 * dnn, "ctr_dnn_layer_bwd_chain": 2.0 * dnn}
    if cfg["model"] == "xDeepFM":
        cin, H = 0, F
        sizes = kw["cin_layer_size"]
        for i, n in enumerate(sizes):
            cin += 2 * D * n * H * F
            H = n // 2 if (kw.get("cin_split_half", True) and i != len(sizes) - 1) else n
        out["ctr_cin_layer_fwd"] = float(cin)
        out["ctr_cin_layer_bwd"] = 2.0 * cin
    if cfg["model"] == "FiBiNET":
        bil = 2 * 325 * (2 * D * D)
        out["ctr_bilinear_fwd"] = float(bil)
        out["ctr_bilinear_bwd"] = 2.0 * bil
    return out


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation on the host cores
# ------------------------------------------------------------------------------------------------
def host_threads():
    """Threads of the CPU arm: every physical core (torchrun exports OMP_NUM_THREADS=1, which is not what a user
    of the reference would run with); override with CTR_CPU_THREADS."""
    n = int(os.environ.get("CTR_CPU_THREADS", "0") or 0)
    if n <= 0:
        n = max(1, (os.cpu_count() or 2) // 2)
    return n


def load_live_reference():
    """The UNMODIFIED reference package: baseline/_ref (scripts/install_reference.sh) or the source tree named by
    CTR_REFERENCE_ROOT.  None when neither exists (-> oracle port)."""
    sys.path.insert(0, os.path.join(REPO, "tests", "golden"))
    import _ref_loader
    for root in (os.path.join(REPO, "baseline", "_ref"), _ref_loader.REFERENCE_ROOT):
        if root and os.path.isdir(os.path.join(root, "deepctr_torch")):
            _ref_loader.REFERENCE_ROOT = root
            try:
                return _ref_loader.load_reference(), root
            except Exception as ex:          # noqa: BLE001
                print("bench.py: importing the reference from %s failed: %s" % (root, str(ex)[:200]), file=sys.stderr)
    return None, None


def build_reference_model(cfg, l2=0.0):
    """The reference's model class for an oracle-style cfg (same constructor arguments as the GPU arm)."""
    from deepctr_torch import models as RM
    from deepctr_torch.inputs import DenseFeat, SparseFeat
    cols = []
    for c in cfg["dnn_columns"]:
        cols.append(SparseFeat(c["name"], c["vocab"], embedding_dim=c["dim"]) if c["type"] == "sparse"
                    else DenseFeat(c["name"], c["dimension"]))
    kw = dict(cfg["kwargs"])
    for k in ("dnn_hidden_units", "cin_layer_size"):
        if k in kw:
            kw[k] = tuple(kw[k])
    kw["l2_reg_linear"] = kw["l2_reg_embedding"] = l2
    return getattr(RM, cfg["model"])(cols, cols, device="cpu", **kw)


def reference_fwd_bwd(model, X, y, steps, warmup):
    """forward + BCE(sum) + backward of the reference model, the same loop as the GPU arm (SURVEY §8d (ii))."""
    model.train()
    times = []
    for it in range(warmup + steps):
        model.zero_grad(set_to_none=True)
        t0 = time.perf_counter()
        loss = torch.nn.functional.binary_cross_entropy(model(X).squeeze(), y, reduction="sum")
        loss.backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return X.shape[0] * len(times) / sum(times), sum(times) / len(times)


def reference_fit_throughput(cfg, X, y, batch):
    """The reference's own fit(): Adam + default L2 regulariser included (SURVEY §8d (i), BASELINE.md §3)."""
    model = build_reference_model(cfg, l2=1e-5)
    model.compile("adam", "binary_crossentropy")
    names = [c["name"] for c in cfg["dnn_columns"]]
    cols, x, off = cfg["dnn_columns"], {}, 0
    for c in cols:
        w = 1 if c["type"] == "sparse" else c["dimension"]
        x[c["name"]] = X[:, off:off + w].numpy()
        off += w
    t0 = time.perf_counter()
    model.fit(x, y.numpy(), batch_size=batch, epochs=1, verbose=0, shuffle=False)
    return X.shape[0] / (time.perf_counter() - t0), names


def cpu_fwd_bwd_throughput(cfg, state, batch, steps, warmup, seed=2026):
    """fwd + BCE(sum) + bwd of the oracle restatement (port), torch CPU fp32 — used when the reference package
    itself is not importable."""
    from oracle import ctr_oracle as O
    X, y = O.synthetic_batch(cfg, batch, seed=seed)
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in state.items()}
    times = []
    for it in range(warmup + steps):
        for v in leaves.values():
            v.grad = None
        t0 = time.perf_counter()
        logit = O.model_logit(cfg, leaves, X)
        loss = torch.nn.functional.binary_cross_entropy(torch.sigmoid(logit).squeeze(-1), y, reduction="sum")
        loss.backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    total = sum(times)
    return batch * len(times) / total, total / len(times)


def random_state_cpu(cfg, seed=7):
    """Random-init weights of the architecture (fp32), generated table by table on the CPU."""
    from helpers import build_model
    g = torch.Generator().manual_seed(seed)
    m = build_model(cfg, "cpu")
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * 0.05)
    return {k: v.detach() for k, v in m.state_dict().items()}


def workload_config(workload, world):
    """The `config` object: identical in both arms (it names the workload, not the implementation)."""
    w = WORKLOADS[workload]
    vocab = 1538462 if world > 1 else 1000000
    return {"workload": w["desc"], "batch_per_gpu": w["B"], "global_batch": w["B"] * world, "vocab_per_table": vocab,
            "sparse_fields": 26, "dense_fields": 13, "embedding_dim": w["D"], "l2": 0,
            "tables": "single GPU" if world == 1 else "26 x %d rows = 40M rows, row-sharded over %d GPUs" % (vocab, world),
            "algorithmic_bytes_per_sample": algorithmic_bytes_per_sample(w["D"])}


def cpu_arm(workload, steps, warmup, cpu_batch, with_fit):
    """(samples/s, s/step, cpu_baseline dict) of the reference's CPU implementation on this box."""
    from oracle import ctr_oracle as O
    threads = host_threads()
    torch.set_num_threads(threads)
    cfg = make_cfg(workload)
    B = WORKLOADS[workload]["B"]
    if cpu_batch:
        B = min(B, cpu_batch)
    elif workload in ("xdeepfm", "fibinet"):
        B = min(B, 8192)             # the reference materialises [B, H*M, D] / [B, 650, D]: 28 GB RSS at the full batch
    ref, root = load_live_reference()
    X, y = O.synthetic_batch(cfg, B, seed=2026)
    extra = {}
    if ref is not None:
        model = build_reference_model(cfg, l2=0.0)
        g = torch.Generator().manual_seed(7)
        with torch.no_grad():
            for p in model.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)
        sps, sec = reference_fwd_bwd(model, X, y, steps, warmup)
        kind = "reference"
        what = "the unmodified reference package (%s), %s(...).forward + BCE(sum) + backward" % (
            "baseline/_ref" if root.endswith("_ref") else root, cfg["model"])
        del model
        if with_fit:
            try:
                fit_sps, _ = reference_fit_throughput(cfg, X, y, B)
                extra["reference_fit"] = {"value": fit_sps, "unit": "samples/s",
                                          "what": "reference model.fit(batch_size=%d, epochs=1) incl. Adam and the default "
                                                  "L2 regulariser (BASELINE.md §3 item 1), one step" % B}
            except Exception as ex:      # noqa: BLE001
                extra["reference_fit"] = {"error": str(ex)[:200]}
    else:
        sps, sec = cpu_fwd_bwd_throughput(cfg, random_state_cpu(cfg), B, steps, warmup)
        kind, what = "port", "oracle port of the reference (same ATen CPU kernels)"
    cb = {"value": sps, "unit": "samples/s", "cores": threads, "kind": kind,
          "sample": "%d fwd+bwd steps of batch %d after %d warm-up: %s, torch CPU fp32, %d threads (os.cpu_count()=%d)"
                    % (steps, B, warmup, what, threads, os.cpu_count())}
    cb.update(extra)
    return sps, sec, cb


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    sps, sec, cb = cpu_arm(args.workload, args.steps, args.warmup, args.cpu_batch, with_fit=True)
    line = {"impl": "reference", "metric": "CTR samples/sec fwd+bwd", "value": sps, "unit": "samples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, max(world, args.gpus)),
            "cpu_baseline": cb,
            "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def _finish_multi_gpu():
    """Leave without tearing the NCCL communicator down: destroy_process_group() hangs when CUDA graphs
    that captured collectives are still alive (observed on 2 GPUs, run 26).  All ranks meet once more,
    flush, and exit."""
    import torch.distributed as dist
    torch.cuda.synchronize()
    try:
        dist.barrier()
    except Exception:                     # noqa: BLE001
        pass
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


def quick_parity_check(dev):
    """One small DeepFM step on this GPU against the CPU oracle before anything is timed (the checker, never the
    thing measured).  Logits are gated on the ReLU tower (north-star bar 1e-5); gradients are gated on the same
    model with a smooth tower activation (1e-4) — under ReLU a pre-activation within round-off of zero may pick the
    other branch in two correctly rounded implementations, which moves whole gradient rows (DESIGN.md §3)."""
    from helpers import build_model, capture_logit, rel_err
    from oracle import ctr_oracle as O
    cols = [O.sparse_col("C%d" % i, 5000, 16) for i in range(26)] + [O.dense_col("I%d" % i) for i in range(13)]
    out = {"parity_checked": True, "what": "DeepFM (256,128), batch 4096 vs the CPU oracle: logits with the ReLU tower, "
                                           "all gradients with a tanh tower"}
    for act in ("relu", "tanh"):
        cfg = O.make_cfg("DeepFM", cols, cols, dnn_hidden_units=[256, 128], dnn_activation=act, init_std=0.05,
                         l2_reg_linear=0, l2_reg_embedding=0)
        m = build_model(cfg, dev, table_grad="rowwise")
        g = torch.Generator().manual_seed(3)
        with torch.no_grad():
            for p in m.parameters():
                p.copy_((torch.randn(p.shape, generator=g) * 0.05).to(dev))
        X, y = O.synthetic_batch(cfg, 4096, seed=5)
        state = {k: v.detach().cpu() for k, v in m.state_dict().items()}
        ref_logit, _, _, ref_grads = O.loss_and_grads(cfg, state, X, y)
        m.train()
        y_pred, logit = capture_logit(m, X.to(dev))
        torch.nn.functional.binary_cross_entropy(y_pred.squeeze(1), y.to(dev), reduction="sum").backward()
        m.check_ids()
        e_logit = rel_err(logit.cpu(), ref_logit)
        e_grad = max(rel_err((p.grad.to_dense() if p.grad.is_sparse else p.grad).cpu(), ref_grads[k])
                     for k, p in m.named_parameters())
        if act == "relu":
            out["max_rel_err"], out["max_grad_rel_err_relu"] = e_logit, e_grad
        else:
            out["max_rel_err_tanh"], out["max_grad_rel_err"] = e_logit, e_grad
    out["ok"] = out["max_rel_err"] <= 1e-5 and out["max_rel_err_tanh"] <= 1e-5 and out["max_grad_rel_err"] <= 1e-4
    return out


DUMP_LIMIT_BYTES = 64 * 10**6     # on disk, .npy headers included
NPY_HEADER_BYTES = 128
DUMP_TABLE_ROWS = 16384    # most rows of every table whose gradient is written: a fixed seeded sample of the row ids


def table_sample_rows(vocab, fixed_bytes, bytes_per_row):
    """Size of the table row sample: DUMP_TABLE_ROWS, or fewer when the other outputs (``fixed_bytes``) leave less of
    DUMP_LIMIT_BYTES than DUMP_TABLE_ROWS rows of every table need."""
    return max(0, min(DUMP_TABLE_ROWS, vocab, (DUMP_LIMIT_BYTES - fixed_bytes) // bytes_per_row))


def dump_outputs(out_dir, model, loss, y_pred, pending):
    """Write what one step hands its caller as ``out_dir/<name>.npy``: ``loss``, ``y_pred``, ``grad.<parameter>`` of
    every dense parameter and, for every table, the per-unique-row gradients the step leaves for the fused optimizer,
    as ``grad.<table>.rows`` (the table's gradient at the ids of ``table_sample_ids`` that are below the table's size,
    zero where the batch does not touch the row) and ``grad.<table>.sum`` (the sum over all its rows, float64).  A
    table shared by several fields gets the sum of their gradients.  ``table_sample_ids`` is a seeded sample of the
    largest table's row ids, as many as fit in DUMP_LIMIT_BYTES (at most DUMP_TABLE_ROWS); it depends only on the
    workload.  ``n_unique_rows`` counts the distinct ids of every id column.  Values are float32, ids and counts
    float64."""
    import numpy as np
    plan = model._plan
    dev = plan.device
    names = {id(p): k for k, p in model.named_parameters()}
    (lease, rg_emb, rg_lin, n_emb), = pending
    ws = lease.ws
    n_uniq = ws["n_uniq"].cpu()
    # table -> (parameter, [(per-unique-row gradients, plan column) of every field that reads it])
    tables = {}
    slots = [(p, rg_emb[i], plan.emb_plan_col_host[i]) for i, p in enumerate(plan.emb_params) if i < n_emb] + \
            [(p, rg_lin[i].unsqueeze(1), plan.lin_plan_col_host[i]) for i, p in enumerate(plan.lin_params)]
    for p, rg, col in slots:
        tables.setdefault(names[id(p)], (p, []))[1].append((rg, col))
    table_ids = set(id(p) for p in plan.emb_params + plan.lin_params)
    arrays = {"loss": loss.reshape(1), "y_pred": y_pred.reshape(-1), "n_unique_rows": n_uniq.double()}
    for k, p in model.named_parameters():
        if id(p) not in table_ids and p.grad is not None:
            arrays["grad." + k] = p.grad
    for name, (p, fields) in tables.items():
        arrays["grad.%s.sum" % name] = sum(rg[:int(n_uniq[col])].double().sum(0) for rg, col in fields)
    vocab = max(int(p.shape[0]) for p, _ in tables.values())
    n_files = len(arrays) + 1 + len(tables)          # + table_sample_ids + one grad.<table>.rows per table
    fixed = sum(a.numel() * a.element_size() for a in arrays.values()) + n_files * NPY_HEADER_BYTES
    rows = table_sample_rows(vocab, fixed, 8 + sum(4 * int(p.shape[1]) for p, _ in tables.values()))
    if rows == 0:
        raise SystemExit("bench.py: --dump-outputs: the dense outputs alone exceed %d bytes" % DUMP_LIMIT_BYTES)
    sample = np.sort(np.random.RandomState(0).choice(vocab, rows, replace=False))
    arrays["table_sample_ids"] = torch.from_numpy(sample).double()
    sample = torch.from_numpy(sample).to(dev)
    for name, (p, fields) in tables.items():
        ids = sample[sample < p.shape[0]]
        out = torch.zeros(len(ids), p.shape[1], device=dev, dtype=torch.float32)
        for rg, col in fields:
            n = int(n_uniq[col])
            pos = torch.full((p.shape[0],), -1, dtype=torch.int64, device=dev)
            pos[ws["uniq"][col, :n].long()] = torch.arange(n, device=dev)
            at = pos[ids]
            out += torch.where((at >= 0).unsqueeze(1), rg[at.clamp_min(0)], 0.0)
        arrays["grad.%s.rows" % name] = out
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    written = sum(os.path.getsize(os.path.join(out_dir, k + ".npy")) for k in arrays)
    assert written <= DUMP_LIMIT_BYTES, written


def measure_workload(workload, args, world, rank, dev, steps, warmup, full=True):
    """Time one workload on this process' GPU (all ranks call it together when world > 1).  Returns a dict with the
    device-resident step time, (full) the e2e time, the per-entry-point times of an instrumented eager pass."""
    import torch.distributed as dist
    from deepctr_torch_b200 import _lib, ops
    from helpers import build_model
    from oracle import ctr_oracle as O

    w = WORKLOADS[workload]
    B = w["B"]
    if world > 1:
        from deepctr_torch_b200 import sharded
        # BASELINE config #5 shape: total vocabulary 40M rows = 26 tables x 1 538 462 rows, row-sharded
        cfg = make_cfg(workload, vocab=1538462)
        model, parallelism = sharded.build_sharded(cfg, dev, rank, world, batch=B)
    else:
        cfg = make_cfg(workload)
        model = build_model(cfg, dev, table_grad="rowwise")
        parallelism = "single"
        # the step's contract is "per-unique-row gradients written once" (SURVEY §8d): leave (uniq, rowgrad) in
        # the plan's buffers, exactly what the fused optimizer consumes, instead of wrapping them as sparse COO
        model._gather_plan(torch.device(dev)).keep_rowgrads = True
    gen = torch.Generator(device=dev).manual_seed(7 + rank)
    with torch.no_grad():
        for p in model.parameters():
            p.copy_(torch.randn(p.shape, generator=gen, device=dev) * 0.05)
    model.train()
    plan = model._plan

    host_batches = []
    for i in range(N_ROTATE):
        X, y = O.synthetic_batch(cfg, B, seed=2026 + 100 * rank + i)
        host_batches.append((X.pin_memory(), y.pin_memory()))
    dev_batches = [(X.to(dev), y.to(dev)) for X, y in host_batches]
    bce = ops.binary_cross_entropy
    dump_dir = args.dump_outputs if full else None
    last = {}           # what the last eager step returned, for --dump-outputs

    def finish():
        if world > 1:       # dense-grad all-reduce (= barrier for the pushed row gradients) + owner-side combine
            done = model.sharded.finish_step()
            model.sharded.combine_received(done)
            model.sharded.clear_received(done)
        else:
            plan.pending.clear()

    def step_eager(X, y):
        model.zero_grad(set_to_none=True)
        y_pred = model(X)
        loss = bce(y_pred.squeeze(1), y, reduction="sum")
        loss.backward()
        if dump_dir:
            last.update(loss=loss, y_pred=y_pred, pending=list(plan.pending))
        finish()
        return loss

    def step_resident(i):
        return step_eager(*dev_batches[i % N_ROTATE])

    def step_e2e(i):
        Xh, yh = host_batches[i % N_ROTATE]
        return float(step_eager(Xh.to(dev, non_blocking=True), yh.to(dev, non_blocking=True)).item())

    use_graph = not args.no_graph
    gstep, graph_error = None, None
    if use_graph:
        # the whole step (world > 1: row exchange, push, NCCL all-reduce, owner-side combine) captured as CUDA
        # graph(s) through the public API; every rank must agree, otherwise the collectives would not match
        try:
            gstep = model.make_graphed_step(B)
        except Exception as ex:                      # noqa: BLE001
            import traceback
            graph_error = "rank %d: %s" % (rank, "".join(traceback.format_exception_only(type(ex), ex)).strip()[:400])
            print("bench.py: CUDA-graph capture failed on " + graph_error, file=sys.stderr, flush=True)
        if world > 1:
            ok = torch.tensor([0.0 if graph_error else 1.0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if float(ok.item()) == 0.0:
                gstep = None
        if gstep is None:
            if not args.allow_eager:
                raise SystemExit("bench.py: CUDA-graph capture of the step failed (%s); pass --no-graph or --allow-eager "
                                 "to time the eager step instead" % (graph_error or "another rank failed"))
            use_graph = False
    if use_graph:
        def step_resident(i):      # noqa: F811
            X, y = dev_batches[i % N_ROTATE]
            return gstep(X, y)

        def step_e2e(i):           # noqa: F811
            Xh, yh = host_batches[i % N_ROTATE]
            return float(gstep(Xh, yh).item())

        def step_e2e_pipelined(i):
            # one H2D copy per step, like step_e2e, but it is the NEXT step's batch, enqueued on a copy
            # stream before this step's replay so that it travels while the step computes
            if not pipe["primed"]:
                gstep.prefetch(*host_batches[i % N_ROTATE])
                pipe["primed"] = True
            gstep.prefetch(*host_batches[(i + 1) % N_ROTATE])
            return float(gstep.step_prefetched().item())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, n_steps, n_warm):
        for i in range(n_warm):
            step_fn(i)
        barrier()
        l0 = _lib.launch_count() + (gstep.replays * gstep.launches_per_replay if use_graph else 0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n_steps):
            step_fn(n_warm + i)
        e1.record()
        barrier()
        # kernels of libctr_b200.so inside the timed region: eager launches are counted by the library,
        # graph replays launch the kernel nodes recorded at capture time
        timed.launches = _lib.launch_count() + (gstep.replays * gstep.launches_per_replay if use_graph else 0) - l0
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    out = {"cfg": cfg, "parallelism": parallelism, "cuda_graph": bool(use_graph), "graph_error": graph_error, "B": B}
    sampler = ClockSampler(int(dev.split(":")[1])) if (rank == 0 and full) else None
    prof_region = full and os.environ.get("CTR_PROFILE_REGION") == "1"   # `ncu --profile-from-start off`: timed region only
    if prof_region:
        for i in range(warmup):
            step_resident(i)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
    out["ms"] = timed(step_resident, steps, 0 if prof_region else warmup)
    if prof_region:
        torch.cuda.profiler.stop()
    out["clocks"] = sampler.stop() if sampler else None
    out["launches"] = timed.launches
    model.check_ids()
    if dump_dir:            # the outputs of the last timed step, before anything else runs on the model
        if use_graph:
            last.update(loss=gstep.loss, y_pred=gstep.y_pred, pending=list(plan.pending))
        dump_outputs(dump_dir, model, last["loss"], last["y_pred"], last["pending"])
        last.clear()
    if full:
        pipe = {"primed": False}
        out["e2e_mode"] = "copy-then-step"
        ms_e2e = None
        if use_graph and os.environ.get("CTR_BENCH_PREFETCH", "1") != "0":
            try:                                  # input pipeline: H2D of step i+1 overlaps step i
                gstep.enable_prefetch()
                ms_e2e = timed(step_e2e_pipelined, steps, max(3, warmup // 2))
                out["e2e_mode"] = "pipelined: the H2D copy of step i+1 overlaps step i (one copy and one loss read per step)"
            except Exception as ex:               # noqa: BLE001
                print("bench.py: pipelined e2e failed (%s); using the simple path" % str(ex)[:200], file=sys.stderr)
                torch.cuda.synchronize()
                ms_e2e = None
        if ms_e2e is None:
            ms_e2e = timed(step_e2e, steps, max(3, warmup // 2))
        out["ms_e2e"] = ms_e2e

    # instrumented pass: CUDA events around every C-ABI entry point -> dominant kernel + roofline
    if gstep is not None and world > 1 and (gstep.replays & 1):
        gstep(*dev_batches[0])          # leave the receive-list parity where the eager steps expect it
    _lib.enable_timing(True)
    n_inst = min(steps, 10)
    for i in range(n_inst):
        step_eager(*dev_batches[i % N_ROTATE])
    summary = _lib.timing_summary()
    _lib.enable_timing(False)
    out["per_entry"] = {k: {"calls_per_step": v[0] / n_inst, "ms_per_step": v[1] / n_inst} for k, v in summary.items()}
    out["state_cpu"] = None
    del gstep, model, dev_batches, host_batches
    torch.cuda.empty_cache()
    return out


def rooflines(workload, m, steps):
    """(roofline dict of the dominant entry point, hbm kernels) from a measure_workload() result."""
    w = WORKLOADS[workload]
    cfg, B, D = m["cfg"], m["B"], w["D"]
    hbm_peak, bf16_peak, bf16_sustained, peak_src = measured_peaks()
    per_entry = m["per_entry"]
    dom = max(per_entry.items(), key=lambda kv: kv[1]["ms_per_step"])
    # boundary bytes of the HBM-bound entry points (DESIGN.md §kernels) per sample
    blk_w = 26 * D + 13
    ld = (blk_w + 3) // 4 * 4
    gather_bytes = 4 * (39 + 26 * D + 26 + blk_w + 2)                 # X row + rows + linear w + blk + lin/fm
    scatter_bytes = 4 * (2 * ld + 26 * 2 + 26 * D + 26 + 2)             # d_blk + blk + inv/cnt + row grads out
    # duplicate-free plan: id read + hash slot (key CAS + value) + inv written twice + cnt/uniq, per id column —
    # a chain of dependent L2 atomics, reported against HBM bandwidth for lack of a better ceiling
    plan_bytes = 26 * (4 + 8 + 8 + 8)
    hbm_entries = {"ctr_gather_fwd": gather_bytes, "ctr_gather_fwd_exchanged": gather_bytes,
                   "ctr_scatter_bwd_rowwise": scatter_bytes, "ctr_unique_plan": plan_bytes,
                   "ctr_cross_vector_fwd": 4 * (2 * ld + 2), "ctr_cross_vector_bwd": 4 * (4 * ld)}
    roofs = {}
    for name, bps in hbm_entries.items():
        if name in per_entry and per_entry[name]["ms_per_step"] > 0:
            t = per_entry[name]["ms_per_step"] / max(per_entry[name]["calls_per_step"], 1) * 1e-3
            gbs = bps * B / t / 1e9
            roofs[name] = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s",
                           "frac": gbs / hbm_peak, "bytes_per_sample": bps, "ms": t * 1e3}
    fl = tensor_flops_per_sample(cfg)
    a_bytes = algorithmic_bytes_per_sample(D)
    step_s = m["ms"] * 1e-3 / steps
    t_roof_hbm = a_bytes * B / (hbm_peak * 1e9)
    # fp32-equivalent FLOPs (2 per MAC; the 3xTF32 mode issues 3 tensor-core MACs for each) of the
    # GEMM-shaped entry points, per step: backward = 2 x forward (input gradient + weight gradient)
    ef = entry_flops_per_sample(cfg)
    traffic = measured_traffic()
    if dom[0] in roofs:
        roofline = dict(roofs[dom[0]], kernel=dom[0], traffic=traffic.get(dom[0]))
    else:
        t = dom[1]["ms_per_step"] * 1e-3
        flops = ef.get(dom[0], 0.0) * B
        tf = flops / t / 1e12 if t > 0 else 0.0
        roofline = {"bound": "tensor", "achieved": tf, "peak": bf16_sustained, "unit": "TFLOP/s",
                    "frac": tf / bf16_sustained, "kernel": dom[0], "traffic": traffic.get(dom[0]),
                    "flops_per_step": flops, "ms": t * 1e3,
                    "frac_of_3xtf32_ceiling": tf / (bf16_sustained / 6.0),
                    "note": "fp32-equivalent FLOPs of this entry point / its CUDA-event time inside the step, against the "
                            "measured SUSTAINED dense bf16 peak; the parity mode (3xTF32: 3 tf32 MMAs per fp32 MAC, tf32 = "
                            "bf16/2) can reach at most 1/6 of that peak, i.e. frac <= 0.167"}
    roofline["peak_source"] = peak_src
    roofline["hbm_kernels"] = roofs
    roofline["step_vs_hbm_roofline"] = t_roof_hbm / step_s
    roofline["step_vs_composite_roofline"] = max(t_roof_hbm, fl * B * 3.0 / (bf16_sustained * 0.5 * 1e12)) / step_s
    return roofline, fl


def run_gpu_arm(args):
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = "cuda:%d" % local_rank
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))

    # parity first: nothing is timed before this process' kernels agreed with the oracle on this box
    if world > 1:
        from sharded_worker import passed, run_check
        worst = run_check(dev, rank, world, B=1024, optimizer="adagrad")
        parity = {"parity_checked": True, "max_rel_err": worst["logit"], "detail": worst, "ok": passed(worst),
                  "what": "row-sharded DeepFM on %d GPUs: logits, dense grads, combined row grads and one fused optimizer "
                          "step vs the CPU oracle (uniform + skewed ids)" % world}
    else:
        parity = quick_parity_check(dev)
    if not parity["ok"]:
        raise SystemExit("bench.py: parity check failed before timing: %s" % json.dumps(parity))

    m = measure_workload(args.workload, args, world, rank, dev, args.steps, args.warmup, full=True)
    secondary = {}
    if world == 1 and not args.no_secondary and args.workload == "deepfm":
        # the other BASELINE configs (+ DCN) so that the driver's one default line records them too
        for wl in ("xdeepfm", "fibinet", "dcn"):
            try:
                ms2 = measure_workload(wl, args, world, rank, dev, 5, 3, full=False)
                r2, _ = rooflines(wl, ms2, 5)
                secondary[wl] = {"workload": WORKLOADS[wl]["desc"], "value": WORKLOADS[wl]["B"] * 5 / (ms2["ms"] * 1e-3),
                                 "unit": "samples/s", "ms_per_step": ms2["ms"] / 5, "steps": 5, "cuda_graph": ms2["cuda_graph"],
                                 "dominant": {k: r2.get(k) for k in ("kernel", "bound", "achieved", "unit", "frac", "ms")},
                                 "step_vs_composite_roofline": r2["step_vs_composite_roofline"],
                                 "hbm_kernels": {k: round(v["frac"], 4) for k, v in r2["hbm_kernels"].items()},
                                 "per_entry_ms": {k: round(v["ms_per_step"], 4) for k, v in ms2["per_entry"].items()}}
            except Exception as ex:          # noqa: BLE001
                secondary[wl] = {"error": str(ex)[:300]}
                torch.cuda.synchronize()

        # labelled NON-PARITY fast mode (VERDICT r1 item 2): the same DeepFM step with single-pass TF32 tower GEMMs
        # (ctr_set_gemm_passes(1)).  A secondary figure only: the headline above is the 3xTF32 parity mode.
        from deepctr_torch_b200 import _lib
        prev = _lib.load().ctr_set_gemm_passes(1)
        try:
            mf = measure_workload("deepfm", args, world, rank, dev, 10, 3, full=False)
            pf = quick_parity_check(dev)
            secondary["deepfm_fast_tf32"] = {
                "workload": WORKLOADS["deepfm"]["desc"] + " — NON-PARITY fast mode: single-pass TF32 on the tensor cores",
                "value": WORKLOADS["deepfm"]["B"] * 10 / (mf["ms"] * 1e-3), "unit": "samples/s", "ms_per_step": mf["ms"] / 10,
                "steps": 10, "cuda_graph": mf["cuda_graph"],
                "logit_rel_err_vs_oracle": pf["max_rel_err"], "grad_rel_err_vs_oracle": pf["max_grad_rel_err"],
                "meets_parity_bar": bool(pf["ok"]),
                "per_entry_ms": {k: round(v["ms_per_step"], 4) for k, v in mf["per_entry"].items()}}
        except Exception as ex:          # noqa: BLE001
            secondary["deepfm_fast_tf32"] = {"error": str(ex)[:300]}
            torch.cuda.synchronize()
        finally:
            _lib.load().ctr_set_gemm_passes(prev)

    if rank != 0:
        if world > 1:
            _finish_multi_gpu()
        return

    w = WORKLOADS[args.workload]
    B = w["B"]
    total_B = B * world
    value = total_B * args.steps / (m["ms"] * 1e-3)
    e2e_value = total_B * args.steps / (m["ms_e2e"] * 1e-3)
    roofline, fl = rooflines(args.workload, m, args.steps)
    line = {
        "metric": "CTR samples/sec fwd+bwd", "value": value, "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["ms"] / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, world),
        "impl_detail": {"parallelism": m["parallelism"], "table_grad": "rowwise (per-unique-row, SURVEY §8d)",
                        "l2_flush": "8 rotating batches, 109 MB of gathered rows each (> L2 with tables)",
                        "tensor_flops_per_sample": fl,
                        "tower_precision": "3xTF32 on tcgen05, fp32 accumulate (parity mode)" if os.environ.get("CTR_GEMM", "") != "simt" else "fp32 FFMA (parity mode)",
                        "cuda_graph": m["cuda_graph"], "graph_error": m["graph_error"]},
        "parity": parity,
        "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": int(B * 39 * 4 + B * 4),
                "d2h_bytes_per_step": 4, "ms_per_step": m["ms_e2e"] / args.steps, "mode": m["e2e_mode"]},
        "gpu_launches": int(m["launches"]),
        "clocks": m["clocks"], "roofline": roofline, "per_entry_ms": m["per_entry"],
    }
    if secondary:
        line["secondary"] = secondary
    if world == 1 and not args.no_cpu_baseline:
        # a bounded sample of the same workload on this box's host cores (the reference arm alone: --impl reference)
        _, _, cb = cpu_arm(args.workload, 3, 1, args.cpu_batch, with_fit=False)
        line["cpu_baseline"] = cb
    print(json.dumps(line))
    if world > 1:
        _finish_multi_gpu()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="deepfm", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-batch", type=int, default=0, help="batch of the CPU arm (0 = the workload's batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="issue the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--allow-eager", action="store_true", help="fall back to the eager step if graph capture fails")
    ap.add_argument("--no-secondary", action="store_true", help="skip the xdeepfm / fibinet / dcn secondary measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (loss, predictions, gradients; table gradients "
                         "at a fixed sample of rows) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1 or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs needs the b200 arm on one GPU")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the b200 arm has no CPU path); use --impl reference")
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
