#!/usr/bin/env python
"""bench.py — samples/sec of one training step of the hot path on B200.

Default workload = BASELINE.json configs[1]: DeepFM Criteo-shape, 39 categorical fields x 25,641
rows (~1.0 M rows), emb_dim 16, MLP 300-300-300, batch 4096 per GPU (weak scaling).
`--workload dlrm` = configs[4]: DLRM Criteo-1TB-shape, 26 sparse fields, ~200 M rows, emb_dim 16,
dot interaction, top MLP 64-64-64, GLOBAL batch 65,536 split over the GPUs (strong scaling), tables
row-sharded over the GPUs.

A "step" is one pass of the hot path over one synthetic batch = the reference's
BaseModel.train_step (fuxictr/pytorch/models/rank_model.py:307-323): zero_grad -> gather / FM / LR /
interaction / MLP forward -> BCE -> backward (dense-gradient scatter-add, GEMM dgrad/wgrad) ->
clip_grad_norm_(10) -> Adam over every parameter.

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference ...                   # the UNMODIFIED reference (oracle/_ref) on host CPU
    python bench.py --impl reference-gpu ...               # the unmodified reference, eager, on cuda:0

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from collections import OrderedDict

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NF, VOCAB, DIM, HIDDEN, BATCH = 39, 25641, 16, [300, 300, 300], 4096
# C5 (SURVEY.md 8d): 26 categorical fields, Criteo-1TB-like cardinalities summing to ~200 M
DLRM_VOCABS = [19_000_000] * 10 + [625_000] * 16
DLRM_TOP, DLRM_GLOBAL_BATCH = [64, 64, 64], 65536
METRICS = {"deepfm": "samples/sec DeepFM Criteo-shape train_step (fwd+bwd+clip+Adam)",
           "dlrm": "samples/sec DLRM Criteo-1TB-shape train_step (fwd+bwd+clip+Adam), row-sharded tables",
           "dcnv2": "samples/sec DCNv2 Criteo-shape train_step (fwd+bwd+clip+Adam)",
           "din": "samples/sec DIN Taobao-shape train_step (fwd+bwd+clip+Adam)",
           "xdeepfm": "samples/sec xDeepFM Criteo-shape train_step (fwd+bwd+clip+Adam)"}
# per-GPU batch of each BASELINE config (SURVEY.md 8d): C2, C5 (global 65,536), C3, C4, xDeepFM at the C2 shape
DEFAULT_BATCH = {"deepfm": BATCH, "dcnv2": 8192, "din": 2048, "xdeepfm": 4096}
DCN_HIDDEN, DIN_HIDDEN, XDFM_HIDDEN, XDFM_CIN, SEQ_LEN = [500, 500, 500], [500, 500, 500], [400, 400, 400], [16, 16, 16], 50


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-gpu"])
    ap.add_argument("--workload", default="deepfm", choices=["deepfm", "dlrm", "dcnv2", "din", "xdeepfm"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (deepfm: 4096; dlrm: 65536 / gpus)")
    ap.add_argument("--vocab-scale", type=float, default=1.0, help="dlrm: scale every cardinality (smoke runs)")
    ap.add_argument("--graph", type=int, default=1, help="capture the step in a CUDA graph")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--nbatches", type=int, default=64, help="distinct synthetic batches rotated through")
    ap.add_argument("--dp-only", action="store_true",
                    help="N>1: replicate the tables and all-reduce the whole gradient arena instead of row-sharding")
    ap.add_argument("--lazy-adam", type=int, default=0,
                    help="1: evaluate the dense Adam semantics of the tables row-wise and lazily (bit-identical)")
    ap.add_argument("--steps-only", action="store_true", help="skip the per-kernel / stress / CPU legs (profiling)")
    ap.add_argument("--precision", default="tf32x3", choices=["fp32", "tf32x3", "tf32", "bf16"],
                    help="arithmetic of the dense GEMMs: fp32 FFMA, 3xTF32 (fp32-class, the parity mode), 1xTF32, or "
                         "bf16 operands with fp32 accumulation (BASELINE configs[1]) on tcgen05")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned and left behind (its loss and "
                         "the model's floating-point state_dict; --gpus 1) as DIR/<name>.npy; large tensors keep a "
                         "fixed, seeded sample of distinct rows, first those the last timed batch touched, so that the "
                         "dump stays under 64 MB.  The inputs are the same "
                         "on every run, but the backward accumulates with float atomics: two runs agree to rounding "
                         "after the first steps and drift apart as steps add up, so compare builds at a small --steps")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        raise SystemExit("--dump-outputs dumps the b200 arm's training step (--impl b200)")
    if a.dump_outputs and a.gpus != 1:
        raise SystemExit("--dump-outputs dumps one GPU's training step (--gpus 1): a row-sharded rank holds a "
                         "slice of the tables and of the batch")
    if a.batch <= 0:
        a.batch = DEFAULT_BATCH[a.workload] if a.workload != "dlrm" else max(DLRM_GLOBAL_BATCH // max(a.gpus, 1), 1)
    if a.gpus > 1 and a.workload not in ("deepfm", "dlrm"):
        raise SystemExit("--workload %s is a single-GPU line (row-sharding is implemented for deepfm and dlrm)" % a.workload)
    return a


# ------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------
def _cat(name, vocab):
    return (name, {"type": "categorical", "source": "", "padding_idx": 0, "vocab_size": vocab})


def make_specs(args=None):
    """Synthetic FeatureMap of the workload (SURVEY.md 8d)."""
    w = "deepfm" if args is None else args.workload
    if w in ("deepfm", "dcnv2", "xdeepfm"):
        return [_cat("C%d" % i, VOCAB) for i in range(NF)]
    if w == "dlrm":
        return [_cat("C%d" % i, max(int(v * args.vocab_scale), 16)) for i, v in enumerate(DLRM_VOCABS)]
    # C4: Taobao-shape DIN: item / category targets, 23 profile fields, two histories sharing the target tables
    specs = [_cat("item_id", 400000), _cat("cate_id", 10000)] + [_cat("f%d" % i, 20000) for i in range(23)]
    for name, donor, vocab in (("click_history", "item_id", 400000), ("cate_history", "cate_id", 10000)):
        specs.append((name, {"type": "sequence", "source": "", "padding_idx": 0, "vocab_size": vocab, "max_len": SEQ_LEN,
                             "share_embedding": donor, "feature_encoder": None}))
    return specs


def vocabs(args):
    return [sp["vocab_size"] for _, sp in make_specs(args)]


def table_rows(args):
    """Rows of parameter memory: shared tables count once."""
    return sum(sp["vocab_size"] for _, sp in make_specs(args) if "share_embedding" not in sp)


def workload_config(args, n_gpus):
    specs = make_specs(args)
    rows = table_rows(args)
    w = args.workload
    if w == "deepfm":
        name = ("DeepFM Criteo-shape: %d fields x %d rows, emb_dim %d, MLP %s, fp32 Adam" % (NF, VOCAB, DIM, HIDDEN))
    elif w == "dlrm":
        name = ("DLRM Criteo-1TB-shape: %d sparse fields, %.1f M rows total, emb_dim %d, dot interaction, top MLP %s, "
                "dense fp32 Adam over every row" % (len(specs), rows / 1e6, DIM, DLRM_TOP))
    elif w == "dcnv2":
        name = ("DCNv2 Criteo-shape: %d fields x %d rows, emb_dim %d, 3 CrossNetV2 layers (624x624) parallel to DNN %s"
                % (NF, VOCAB, DIM, DCN_HIDDEN))
    elif w == "din":
        name = ("DIN Taobao-shape: 27 fields (25 categorical + 2 histories of length %d sharing the target tables), "
                "emb_dim %d, attention MLP [64] Dice, DNN %s" % (SEQ_LEN, DIM, DIN_HIDDEN))
    else:
        name = ("xDeepFM Criteo-shape: %d fields x %d rows, emb_dim %d, CIN %s, DNN %s" % (NF, VOCAB, DIM, XDFM_CIN, XDFM_HIDDEN))
    if n_gpus == 1:
        par = "single GPU holds all tables"
    elif args.dp_only:
        par = "dp%d (replicated tables, all-reduce of the gradient arena)" % n_gpus
    else:
        par = "tables row-sharded over %d GPUs (P2P push/pull over NVLink) + dense dp all-reduce" % n_gpus
    width = DIM + (1 if w in ("deepfm", "xdeepfm") else 0)          # + the D=1 LogisticRegression tables
    arena_mb = rows * width * 4 / 1e6 / (1 if n_gpus == 1 or args.dp_only else n_gpus)
    return {"workload": name, "global_batch": args.batch * n_gpus, "per_gpu_batch": args.batch, "parallelism": par,
            "cache": "working set (4 fp32 arenas x %.0f MB per GPU: params, grads, Adam m/v) exceeds the 126 MB L2; "
                     "%d distinct index batches are rotated" % (arena_mb, args.nbatches)}


def make_batches(n, batch, seed=0, specs=None):
    """SURVEY.md 8(d): uniform ids in [1, V), sequences post-padded with 0 to a random length in [1, L],
    Bernoulli(0.25) labels, one (B, input_length + 1) float64 matrix per batch — exactly what the
    reference's BatchCollator hands to the model."""
    import torch
    specs = make_specs() if specs is None else specs
    gen = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        cols = []
        for _, sp in specs:
            v = float(sp["vocab_size"])
            width = sp.get("max_len", 1) if sp["type"] == "sequence" else 1
            u = torch.rand(batch, width, generator=gen, dtype=torch.float64)
            ids = (1 + torch.floor(u * (v - 1))).clamp_(max=v - 1)          # uniform in [1, V)
            if width > 1:
                lens = torch.randint(1, width + 1, (batch, 1), generator=gen)
                ids = ids * (torch.arange(width).view(1, -1) < lens)
            cols.append(ids)
        cols.append((torch.rand(batch, 1, generator=gen) < 0.25).double())
        out.append(torch.cat(cols, dim=1))
    return out


def zipf_ids(batch, vs, alpha=1.05, seed=0, device="cpu"):
    """Zipf(alpha) ranks clipped to [1, V_f) (SURVEY.md 8d: Criteo-like skew), inverse-CDF sampled."""
    import torch
    gen = torch.Generator(device=device).manual_seed(seed)
    cols = []
    for v in vs:
        u = torch.rand(batch, generator=gen, device=device, dtype=torch.float64)
        # continuous approximation of the Zipf CDF on [1, V): F(x) = (x^(1-a) - 1) / (V^(1-a) - 1)
        x = (1.0 + u * (float(v) ** (1.0 - alpha) - 1.0)) ** (1.0 / (1.0 - alpha))
        cols.append(torch.floor(x).clamp_(1, v - 1))
    return torch.stack(cols, dim=1)


# ------------------------------------------------------------------------------------------
# clocks / throttle sampling during the timed region
# ------------------------------------------------------------------------------------------
class ClockSampler(object):
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.rows, self.proc, self.dev = [], None, device_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def wait_first(self, seconds=8.0):
        """nvidia-smi takes a second or two to print its first row: wait for it before the timed region."""
        t_end = time.time() + seconds
        while self.proc is not None and not self.rows and time.time() < t_end:
            time.sleep(0.05)

    def count_between(self, t0, t1):
        return sum(1 for t, _ in self.rows if t0 <= t <= t1)

    def stop(self, windows=None):
        """Median SM clock and the throttle reasons over the rows sampled inside `windows`
        (a list of (t0, t1) wall-clock intervals under load); all rows when windows is None."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, r in self.rows:
            if windows is not None and not any(a <= t <= b for a, b in windows):
                continue
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# Reference arms: the UNMODIFIED reference from oracle/_ref (its own model class, its own
# BaseModel.train_step), on the host CPU or eager on cuda:0.  Falls back to the oracle port when
# oracle/_ref is absent.
# ------------------------------------------------------------------------------------------
def build_reference_model(args, gpu):
    """(model, feature_map) of the reference's own class for the workload, from a synthetic FeatureMap."""
    from baseline import refenv
    R = refenv.import_reference()
    import torch
    fm = refenv.synthetic_feature_map(make_specs(args), embedding_dim=DIM)
    common = dict(model_root="/tmp/b2_bench_ref/", metrics=["logloss", "AUC"], verbose=0, optimizer="adam",
                  loss="binary_crossentropy", task="binary_classification", gpu=gpu, learning_rate=1e-3,
                  embedding_dim=DIM, embedding_regularizer=0, net_regularizer=0, net_dropout=0, batch_norm=False)
    R.torch_utils.seed_everything(seed=2019)
    w = args.workload
    if w == "deepfm":
        model = refenv.load_model_class("DeepFM")(fm, model_id="DeepFM_bench", hidden_units=HIDDEN,
                                                  hidden_activations="relu", **common)
    elif w == "dlrm":
        common.pop("net_dropout")
        model = refenv.load_model_class("DLRM")(fm, model_id="DLRM_bench", top_mlp_units=DLRM_TOP,
                                                bottom_mlp_units=[64, 64, 64], top_mlp_activations="ReLU",
                                                bottom_mlp_activations="ReLU", top_mlp_dropout=0, bottom_mlp_dropout=0,
                                                interaction_op="dot", **common)
    elif w == "dcnv2":
        model = refenv.load_model_class("DCNv2")(fm, model_id="DCNv2_bench", model_structure="parallel",
                                                 num_cross_layers=3, parallel_dnn_hidden_units=DCN_HIDDEN,
                                                 dnn_activations="ReLU", **common)
    elif w == "din":
        model = refenv.load_model_class("DIN")(fm, model_id="DIN_bench", dnn_hidden_units=DIN_HIDDEN,
                                               dnn_activations="ReLU", attention_hidden_units=[64],
                                               attention_hidden_activations="Dice", attention_dropout=0, **common)
    else:
        model = refenv.load_model_class("xDeepFM")(fm, model_id="xDeepFM_bench", dnn_hidden_units=XDFM_HIDDEN,
                                                   dnn_activations="ReLU", cin_hidden_units=XDFM_CIN, **common)
    model._max_gradient_norm = 10.0          # BaseModel.fit() sets it (rank_model.py:213); train_step reads it
    model.train()
    return model, fm, torch


def reference_batches(fm, mats):
    """What BatchCollator.__call__ yields (npz_dataloader.py:111-125): column views of one matrix."""
    cols = list(fm.features.keys()) + list(fm.labels)
    return [{c: m[:, fm.get_column_index(c)] for c in cols} for m in mats]     # list index => (B, L) copy, as the collator


def cpu_reference_run(args, steps, warmup, seconds=None, threads=None):
    """Times the reference's own BaseModel.train_step on the host cores.  Thread count: a fixed sweep
    with >= 5 timed steps per candidate, the fastest is used for the sample and reported."""
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
    batch = args.batch
    try:
        model, fm, torch = build_reference_model(args, -1)
        step = model.train_step
        batches = reference_batches(fm, make_batches(4, batch, specs=make_specs(args)))
        kind = "reference"
    except ImportError:       # no oracle/_ref on this machine: the oracle restatement (same ATen ops)
        import torch
        from oracle import fuxictr_oracle as O
        from fuxictr_b200 import zoo
        from fuxictr_b200.schema import FeatureMap
        if args.workload != "deepfm":
            raise
        specs = make_specs(args)
        fm = FeatureMap.from_specs(specs, embedding_dim=DIM)
        torch.manual_seed(2019)
        holder = zoo.DeepFM(fm, gpu=-1, embedding_dim=DIM, hidden_units=HIDDEN)  # parameter container only
        spec_map = OrderedDict(specs)
        tr = O.OracleTrainer(holder.state_dict(),
                             lambda s, X: torch.sigmoid(O.deepfm_logit(spec_map, s, X, len(HIDDEN))), spec_map, ["label"])
        step = tr.train_step
        batches = [fm.batch_dict(m) for m in make_batches(4, batch)]
        kind = "port"
    sweep = {}
    if threads is None:
        # "all the host threads it can use": ATen's intra-op pool stops scaling (and then collapses) long
        # before 100+ threads on ops this small, so the reference gets the count at which IT is fastest.
        # (at 128 threads one 4096-sample step takes 30 s on this path: a candidate whose first step is
        # already 3x slower than the best so far is recorded from that one step and not pursued)
        best_step = None
        for cand in sorted(set(c for c in (8, 16, 32, 64, ncpu) if c <= ncpu)):
            torch.set_num_threads(cand)
            t0 = time.perf_counter()
            step(batches[0])
            first = time.perf_counter() - t0
            if best_step is not None and first > 3.0 * best_step:
                sweep[cand] = batch / first
                continue
            t0 = time.perf_counter()
            for i in range(5):
                step(batches[i % len(batches)])
            per = (time.perf_counter() - t0) / 5
            sweep[cand] = batch / per
            best_step = per if best_step is None else min(best_step, per)
        threads = max(sweep, key=sweep.get)
    torch.set_num_threads(threads)
    for i in range(warmup):
        step(batches[i % len(batches)])
    t0 = time.perf_counter()
    done = 0
    while True:
        step(batches[done % len(batches)])
        done += 1
        el = time.perf_counter() - t0
        if seconds is not None:
            if el >= seconds and done >= 3:
                break
        elif done >= steps:
            break
    return {"value": batch * done / el, "ms_per_step": 1e3 * el / done, "steps": done, "cores": threads,
            "host_cpus": ncpu, "kind": kind, "sweep": {str(k): round(v, 1) for k, v in sweep.items()}}


def cpu_baseline_entry(r, args, how):
    what = ("the unmodified reference (oracle/_ref: model_zoo class + BaseModel.train_step)" if r["kind"] == "reference"
            else "oracle port of the reference's ATen path")
    return {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": r["kind"],
            "sample": "%d train steps of batch %d %s on %d of %d host threads (fastest of the sweep %s); %s"
                      % (r["steps"], args.batch, how, r["cores"], r["host_cpus"], r["sweep"], what)}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    warm = min(args.warmup, 5)
    r = cpu_reference_run(args, steps, warm)
    line = {"impl": "reference", "metric": METRICS[args.workload], "value": r["value"], "unit": "samples/s",
            "n_gpus": args.gpus, "steps": r["steps"], "warmup": warm, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak" if args.workload == "deepfm" else "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, args.gpus),
            "cpu_baseline": cpu_baseline_entry(r, args, "(this run)"),
            "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def reference_gpu_eager(args, steps=30, warmup=5):
    """The unmodified reference on the SAME B200, eager CUDA, no patching: the GPU-vs-GPU bar
    (SURVEY.md 8d).  Reported with the `loss.item()` sync of train_epoch (rank_model.py:342) and without."""
    from fuxictr_b200 import patch
    patch.disable()
    model, fm, torch = build_reference_model(args, 0)
    batches = reference_batches(fm, [m.pin_memory() for m in make_batches(8, args.batch, specs=make_specs(args))])
    out = {}
    for sync in (True, False):
        for i in range(warmup):
            loss = model.train_step(batches[i % len(batches)])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            loss = model.train_step(batches[i % len(batches)])
            if sync:
                loss.item()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out["with_loss_item_sync" if sync else "no_host_sync"] = {"ms_per_step": ms, "value": args.batch / ms * 1e3}
    del model
    torch.cuda.empty_cache()
    return {"unit": "samples/s", "value": out["with_loss_item_sync"]["value"], "detail": out, "steps": steps,
            "what": "unmodified reference model_zoo class + BaseModel.train_step, eager on cuda:0 (per-feature "
                    ".to(device), aten embedding/cuBLAS kernels, torch.optim.Adam)"}


def run_reference_gpu_arm(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    r = reference_gpu_eager(args, steps=args.steps, warmup=max(min(args.warmup, 10), 3))
    print(json.dumps({"impl": "reference-gpu", "metric": METRICS[args.workload], "value": r["value"],
                      "unit": "samples/s", "n_gpus": 1, "higher_is_better": True, "dtype": "f32", "data": "synthetic",
                      "config": workload_config(args, 1), "detail": r}))


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
def time_kernel(fn, reps, stream_sync=None):
    """Average device duration (ms) of `fn` over `reps` back-to-back launches.  The launches are
    captured into one CUDA graph so that host-side (Python/ctypes) launch cost does not leak into
    a microsecond-scale kernel time; CUDA events bracket the replay on the launching stream."""
    import torch
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def profile_step_shares(pipe, dev_batch):
    """Device time of every C-ABI launch of ONE eager step, in step order.  The step is enqueued behind
    a long spin kernel so the whole launch sequence is resident before it starts (host launch cost
    stays out of the event intervals); each call is bracketed by CUDA events on the launching stream."""
    import torch
    from fuxictr_b200 import _lib
    records = []
    orig_call = _lib.call

    def timed_call(name, *a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = orig_call(name, *a)
        e1.record()
        records.append((name, e0, e1))
        return rc

    saved_graph = pipe.graph
    pipe.graph = None
    torch.cuda.synchronize()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(int(2.0e8))            # ~0.1 s at 2 GHz: the queue fills behind it
    _lib.call = timed_call
    try:
        s0.record()
        pipe.step_device(dev_batch)
        s1.record()
    finally:
        _lib.call = orig_call
        pipe.graph = saved_graph
    torch.cuda.synchronize()
    total_us = s0.elapsed_time(s1) * 1e3
    agg = OrderedDict()
    for name, e0, e1 in records:
        ent = agg.setdefault(name, {"launches": 0, "us": 0.0})
        ent["launches"] += 1
        ent["us"] += e0.elapsed_time(e1) * 1e3
    ours = sum(v["us"] for v in agg.values())
    for v in agg.values():
        v["share"] = v["us"] / total_us
    return {"eager_step_us": total_us, "c_abi_us": ours, "other_us (torch fills/copies, NCCL)": total_us - ours,
            "calls": agg}


def kernel_rooflines(model, fm, dev_batch, peaks, args, with_gather=True):
    """Per-kernel achieved bandwidth / flops, measured live with CUDA events (graph-captured
    back-to-back launches): the fused gather (north-star kernel), the dense clip+Adam pass and the
    tensor-core GEMMs of the first MLP layer (forward, dgrad, wgrad shapes)."""
    import ctypes
    import torch
    from fuxictr_b200 import _lib, functional as F2
    out = {}
    hbm = peaks["hbm_gbs"]
    X = OrderedDict((k, v) for k, v in fm.batch_dict(dev_batch).items() if k != "label")
    B = dev_batch.shape[0]
    nf = fm.num_fields
    fed = model.embedding_layer
    fed = getattr(fed, "embedding_layer", fed)          # DIN holds the FeatureEmbeddingDict directly
    if with_gather:
        with torch.no_grad():
            ms = time_kernel(lambda: fed.forward(X), 50, None)
        slots = sum(sp.get("max_len", 1) if sp["type"] == "sequence" else 1 for sp in fm.features.values())
        gbytes = B * (slots * 8 + 2 * slots * DIM * 4)   # SURVEY 8d: per slot 8 (id) + D*4 (row) + D*4 (out)
        out["embed_gather_fwd"] = {"ms": ms, "algorithmic_bytes": gbytes, "GBps": gbytes / ms / 1e6,
                                   "frac_of_measured_hbm": gbytes / ms / 1e6 / hbm,
                                   "note": "B=%d, uniform ids; the launch is latency-bound at this size" % B}
    opt = model._fused_optimizer
    a = model._arena
    st = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731
    P, G, M, V = (ctypes.c_void_p(t.data_ptr()) for t in (a.P, a.G, opt.M, opt.V))
    if a.numel * 16 < 40e9:                  # the timing loop works on copies of the state: skip when they do not fit
        backup = (a.P.clone(), opt.M.clone(), opt.V.clone(), a.G.clone())
        opt.step_dev.add_(1)
        ms = time_kernel(lambda: _lib.call("b2_adam_step", P, G, M, V, a.numel, ctypes.c_void_p(opt.sumsq.data_ptr()),
                                           10.0, 1e-3, 0.9, 0.999, 1e-8, ctypes.c_void_p(opt.step_dev.data_ptr()),
                                           1, st()), 10, None)
        abytes = a.numel * 4 * 8             # 4 reads (p,g,m,v) + 4 writes (p,m,v, g=0) of fp32
        out["adam_step"] = {"ms": ms, "algorithmic_bytes": abytes, "GBps": abytes / ms / 1e6,
                            "frac_of_measured_hbm": abytes / ms / 1e6 / hbm}
        ms = time_kernel(lambda: _lib.call("b2_sumsq", G, a.numel, ctypes.c_void_p(opt.sumsq.data_ptr()), st()), 10, None)
        sbytes = a.numel * 4
        out["grad_sumsq"] = {"ms": ms, "algorithmic_bytes": sbytes, "GBps": sbytes / ms / 1e6,
                             "frac_of_measured_hbm": sbytes / ms / 1e6 / hbm}
        a.P.copy_(backup[0]); opt.M.copy_(backup[1]); opt.V.copy_(backup[2]); a.G.copy_(backup[3])
        opt.step_dev.sub_(1)
        del backup
    mode = F2.get_matmul_precision()
    if mode != "fp32":
        x3 = mode == "tf32x3"
        # dense TF32 = half the measured bf16 rate; bf16 operands are measured against the bf16 rate itself
        tf32_peak = peaks.get("bf16_tflops", 1590.0) / (1.0 if mode == "bf16" else 2.0)
        # the largest dense contraction of the workload: (in, out) widths of that Linear
        K_, N_ = {"deepfm": (nf * DIM, HIDDEN[0]), "dlrm": (DLRM_TOP[0], DLRM_TOP[1]),
                  "dcnv2": (nf * DIM, nf * DIM), "din": (fm.sum_emb_out_dim(), DIN_HIDDEN[0]),
                  "xdeepfm": (nf * DIM, XDFM_HIDDEN[0])}[args.workload]
        x = torch.randn(B, K_, device="cuda"); w = torch.randn(N_, K_, device="cuda"); dz = torch.randn(B, N_, device="cuda")
        xs, ws, dzs = F2.make_aux(x), F2.make_aux(w), F2.make_aux(dz)
        y, dx, dw = torch.empty(B, N_, device="cuda"), torch.empty(B, K_, device="cuda"), torch.empty(N_, K_, device="cuda")
        cases = {
            "gemm_fwd  Y=X.W^T": (lambda: F2.gemm_ex(x, w, y, a_small=xs, b_small=ws), (B, N_, K_)),
            "gemm_dgrad dX=dZ.W (W MN-major)": (lambda: F2.gemm_ex(dz, w, dx, b_mn=True, a_small=dzs, b_small=ws), (B, K_, N_)),
            "gemm_wgrad dW=dZ^T.X (both MN-major)": (lambda: F2.gemm_ex(dz, x, dw, a_mn=True, b_mn=True, a_small=dzs, b_small=xs), (N_, K_, B)),
        }
        for name, (fn, (m_, n_, k_)) in cases.items():
            if K_ % 4 or N_ % 4:
                continue
            ms = time_kernel(fn, 30, None)
            flops = 2.0 * m_ * n_ * k_
            out[name] = {"ms": ms, "shape_MNK": [m_, n_, k_], "passes": 3 if x3 else 1,
                         "TFLOPs_algorithmic": flops / ms / 1e9,
                         "frac_of_tf32_peak_algorithmic": flops / ms / 1e9 / tf32_peak,
                         "frac_of_tf32_peak_counting_passes": flops * (3 if x3 else 1) / ms / 1e9 / tf32_peak,
                         "tf32_peak_TFLOPs": tf32_peak}
    return out


def gather_points(peaks, rows, vs_label):
    """The fused multi-field gather (the metric's own kernel) at B in {4096, 65536, 524288}, uniform and
    Zipf(1.05) ids (SURVEY.md 8d), on F = 39 tables of `rows` rows x 64 B."""
    import torch
    from fuxictr_b200 import functional as F2
    res = []
    F_, D = NF, DIM
    tables = [torch.empty(rows, D, device="cuda").normal_(0, 0.01) for _ in range(F_)]
    plan = F2.GatherPlan([F2.GatherField("C%d" % i, i, D, padding_idx=0) for i in range(F_)])
    for dist_name in ("uniform", "zipf1.05"):
        for B in (4096, 65536, 524288):
            if dist_name == "uniform":
                gen = torch.Generator(device="cuda").manual_seed(B)
                mat = torch.randint(1, rows, (B, F_ + 1), device="cuda", generator=gen).double()
            else:
                mat = torch.cat([zipf_ids(B, [rows] * F_, 1.05, seed=B, device="cuda"),
                                 torch.zeros(B, 1, device="cuda", dtype=torch.float64)], dim=1)
            idx = [mat[:, i] for i in range(F_)]
            nbytes = B * (F_ * 8 + 2 * F_ * D * 4)
            for hot_rows in ((0,) if dist_name == "uniform" else (0, 16)):
                plan.hot_rows = hot_rows
                with torch.no_grad():
                    ms = time_kernel(lambda: F2.embed_gather(plan, idx, tables), 20, None)
                res.append({"ids": dist_name, "batch": B, "hot_rows_in_smem": hot_rows, "ms": ms, "GBps": nbytes / ms / 1e6,
                            "frac_of_measured_hbm": nbytes / ms / 1e6 / peaks["hbm_gbs"]})
            plan.hot_rows = 0
            del mat, idx
    del tables
    torch.cuda.empty_cache()
    return {"tables": vs_label, "table_bytes": rows * D * 4 * F_, "algorithmic_bytes_per_sample": F_ * 8 + 2 * F_ * D * 4,
            "points": res}


DUMP_BYTES = 60 << 20          # under the 64 MB that --dump-outputs promises


def touched_rows(fm, batch, key):
    """Rows of the embedding table `key` (a state_dict key) that the batch matrix indexes, or None."""
    import torch
    if not key.endswith(".weight") or "embedding_layers." not in key:
        return None
    table = key.split("embedding_layers.")[-1][:-len(".weight")]
    cols = []
    for name, sp in fm.features.items():
        if name == table or sp.get("share_embedding") == table:
            idx = fm.column_index[name]
            cols += idx if isinstance(idx, list) else [idx]
    return batch[:, cols].long().flatten().unique() if cols else None


def sample_rows(nrows, n, gen, touched=None):
    """n distinct row indices out of nrows (n < nrows): rows in `touched` first, the rest uniform."""
    import torch
    pick = torch.empty(0, dtype=torch.long)
    if touched is not None:
        pick = touched[torch.randperm(len(touched), generator=gen)[:n]]
    if len(pick) < n:
        rest = (torch.randperm(nrows, generator=gen) if nrows <= 4 * n
                else torch.randint(0, nrows, (2 * n,), generator=gen).unique())
        rest = rest[~torch.isin(rest, pick)]
        pick = torch.cat([pick, rest[torch.randperm(len(rest), generator=gen)[:n - len(pick)]]])
    return pick.sort().values


def dump_outputs(out_dir, loss, model, fm, last_batch):
    """Writes the last timed step's loss and the floating-point state_dict it left as
    out_dir/<name>.npy (float32, float64 kept as such).  An array larger than its even share of
    DUMP_BYTES keeps a sample of distinct rows drawn from a generator seeded with its position in the
    state_dict, embedding tables first from the rows `last_batch` (the last timed step's input)
    updated: the same rows every run, so that two builds can be compared array for array."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    params = [(k, v.detach()) for k, v in model.state_dict().items() if v.is_floating_point()]
    share = DUMP_BYTES // (len(params) + 1)
    arrays = [("loss", torch.tensor([loss], dtype=torch.float32))]
    for i, (k, v) in enumerate(params):
        cap = share // (8 if v.dtype == torch.float64 else 4)
        if v.numel() > cap:
            n = max(cap // max(v[0].numel(), 1), 1)
            rows = sample_rows(v.shape[0], n, torch.Generator().manual_seed(i), touched_rows(fm, last_batch, k))
            v = v.index_select(0, rows.to(v.device))
        arrays.append(("param." + k, v.double() if v.dtype == torch.float64 else v.float()))
    for name, v in arrays:
        np.save(os.path.join(out_dir, name + ".npy"), v.cpu().numpy())


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fd:
            p = json.load(fd)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p.get("bf16_tflops", 1590.0)),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback (B200_PROFILING.md)"}


def build_model(args, local, world):
    """The workload's model on this rank's GPU (row-sharded when world > 1), with the fused optimizer."""
    import torch
    from fuxictr_b200 import zoo
    from fuxictr_b200.schema import FeatureMap
    fm = FeatureMap.from_specs(make_specs(args), embedding_dim=DIM)

    def construct():
        torch.manual_seed(2019)
        # parameters are created directly in HBM: a 200 M-row table set is 12.8 GB, too much to stage
        # through host memory once per rank
        with torch.device("cuda:%d" % local):
            w = args.workload
            if w == "deepfm":
                return zoo.DeepFM(fm, gpu=local, embedding_dim=DIM, hidden_units=HIDDEN)
            if w == "dlrm":
                return zoo.DLRM(fm, gpu=local, embedding_dim=DIM, top_mlp_units=DLRM_TOP, interaction_op="dot")
            if w == "dcnv2":
                return zoo.DCNv2(fm, gpu=local, embedding_dim=DIM, model_structure="parallel", num_cross_layers=3,
                                 parallel_dnn_hidden_units=DCN_HIDDEN)
            if w == "din":
                return zoo.DIN(fm, gpu=local, embedding_dim=DIM, dnn_hidden_units=DIN_HIDDEN, attention_hidden_units=[64],
                               attention_hidden_activations="Dice")
            return zoo.xDeepFM(fm, gpu=local, embedding_dim=DIM, dnn_hidden_units=XDFM_HIDDEN, cin_hidden_units=XDFM_CIN)
    model = construct()
    sharded = world > 1 and not args.dp_only
    if sharded:
        try:
            from fuxictr_b200.sharded import SymmPeerGroup
            model.enable_sharding(SymmPeerGroup(), args.batch, fm.input_length + 1, torch.float64,
                                  want_fm=(args.workload == "deepfm"))
            torch.cuda.empty_cache()
        except Exception as exc:   # no peer-mapped memory on this box: replicated tables + arena all-reduce
            sys.stderr.write("[bench] row-sharding unavailable (%r); using --dp-only\n" % (exc,))
            sharded = False
            args.dp_only = True
            model = construct()
    opt = model.use_fused_optimizer(lazy_tables=bool(args.lazy_adam) and world == 1)
    if world > 1 and not sharded:
        opt.grad_allreduce = True
    model.train()
    return model, fm, sharded


def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run)" % (args.gpus, world))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    from fuxictr_b200 import _lib, functional as F2
    _lib.load()
    F2.set_matmul_precision(args.precision)
    peaks = load_peaks()

    def note(msg):
        if os.environ.get("B2_BENCH_VERBOSE"):
            sys.stderr.write("[bench r%d] %s\n" % (rank, msg))
            sys.stderr.flush()

    model, fm, sharded = build_model(args, local, world)
    width = fm.input_length + 1
    note("model built")
    host_batches = [m.pin_memory() for m in make_batches(args.nbatches, args.batch, seed=1000 + rank, specs=make_specs(args))]
    dev_batches = [m.cuda(non_blocking=True) for m in host_batches]
    # launches per step (our kernels only): counted by wrapping the C-ABI call around one eager step
    from fuxictr_b200.pipeline import TrainPipeline
    pipe = TrainPipeline(model, args.batch, width, torch.float64, graph=False)
    pipe.prime(dev_batches[0])
    counter = {"n": 0}
    orig_call = _lib.call

    def counting_call(name, *a):
        counter["n"] += 1
        return orig_call(name, *a)

    pipe.step_device(dev_batches[0])        # first step: lazy allocations, cuTensorMap entry point, ...
    _lib.call = counting_call
    pipe.step_device(dev_batches[0])
    torch.cuda.synchronize()
    launches = counter["n"]
    _lib.call = orig_call
    shares = None
    if world == 1 and not args.steps_only:
        try:
            shares = profile_step_shares(pipe, dev_batches[1 % len(dev_batches)])
        except Exception as exc:
            shares = {"error": repr(exc)}
    if world > 1:
        dist.barrier()
    if args.graph:
        try:
            pipe.capture(3)     # the constructor does this for graph=True; done late here to count launches first
        except Exception as exc:   # report an eager number rather than none (the JSON line says cuda_graph: false)
            import traceback
            sys.stderr.write("[bench r%d] CUDA-graph capture failed (%r); timing the eager step\n%s\n"
                             % (rank, exc, traceback.format_exc()))
            pipe.graph, pipe.loss_dev = None, None
            torch.cuda.synchronize()
    note("graph captured")

    def run_step(i, e2e):
        if e2e:     # the user-facing call: pinned host matrix -> async H2D (overlapping the previous
            pipe.step(host_batches[i % len(host_batches)])     # step) -> graph replay -> loss D2H
        else:       # inputs already resident in HBM
            pipe.step_device(dev_batches[i % len(dev_batches)])

    def timed(e2e, steps, warmup):
        for i in range(warmup):
            run_step(i, e2e)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            run_step(warmup + i, e2e)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    warmup = max(args.warmup, 3)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_first()
    t_w0 = time.time()
    ms_total = timed(False, args.steps, warmup)
    ms_e2e = timed(True, args.steps, warmup)
    t_w1 = time.time()
    if args.dump_outputs and rank == 0:     # before the untimed clock-sampling steps below change the state
        dump_outputs(args.dump_outputs, pipe.loss(), model, fm, host_batches[(warmup + args.steps - 1) % len(host_batches)])
    windows, clock_note = [(t_w0, t_w1)], "rows sampled inside the two timed regions"
    if ms_total + ms_e2e < 600.0:
        # a few hundred sub-millisecond steps end before nvidia-smi's 100 ms sampling sees them: keep the
        # same step running back to back (untimed, every rank: the count follows from the all-reduced time)
        # for ~0.8 s right after, and sample the clocks over it as well
        n_extra = int(800.0 / max(ms_total / args.steps, 1e-3))
        t_x0 = time.time()
        for i in range(n_extra):
            run_step(i, False)
        torch.cuda.synchronize()
        windows.append((t_x0, time.time()))
        clock_note = ("timed regions (%.0f ms) are shorter than the sampling period: sampled over them plus "
                      "%d further identical steps run back to back right after" % (ms_total + ms_e2e, n_extra))
    clocks = sampler.stop(windows) if rank == 0 else None
    if clocks is not None:
        clocks["sampled"] = clock_note
    final_loss = pipe.loss()
    note("timed regions done")
    if rank != 0:
        # Last collective done.  Leave without NCCL teardown: rank 0 still captures CUDA graphs for
        # its single-rank kernel measurements, and a concurrent communicator finalize hung here.
        sys.stdout.flush()
        os._exit(0)
    samples = args.batch * world * args.steps
    value = samples / (ms_total / 1e3)
    e2e_value = samples / (ms_e2e / 1e3)
    step_ms = ms_total / args.steps
    if args.steps_only:
        print(json.dumps({"value": value, "ms_per_step": step_ms, "e2e": e2e_value, "workload": args.workload,
                          "gpu_launches_per_step": launches, "precision": args.precision, "n_gpus": world}))
        sys.stdout.flush()
        if world > 1:
            os._exit(0)
        return
    kernels = kernel_rooflines(model, fm, dev_batches[0], peaks, args, with_gather=not sharded)
    # dominant kernel = largest share of the profiled step among ALL C-ABI launches (GEMMs included)
    group = {"b2_gemm_tc_ex": "gemm", "b2_gemm_tc": "gemm", "b2_adam_step": "adam_step", "b2_adam_step_sched": "adam_step",
             "b2_sumsq": "grad_sumsq"}
    by_group = {}
    if shares and "calls" in shares:
        for name, v in shares["calls"].items():
            gname = group.get(name, name)
            ent = by_group.setdefault(gname, {"us": 0.0, "launches": 0})
            ent["us"] += v["us"]
            ent["launches"] += v["launches"]
    dom = max(by_group, key=lambda k: by_group[k]["us"]) if by_group else "adam_step"
    share = (by_group[dom]["us"] / shares["eager_step_us"]) if by_group else None
    tf32_peak = peaks["bf16_tflops"] / 2.0
    if dom == "gemm":
        gem = [v for k, v in kernels.items() if k.startswith("gemm_")]
        flops = sum(2.0 * v["shape_MNK"][0] * v["shape_MNK"][1] * v["shape_MNK"][2] for v in gem)
        ms = sum(v["ms"] for v in gem)
        passes = gem[0]["passes"] if gem else 1
        roofline = {"kernel": "gemm_tf32_kernel (first MLP layer: forward + dgrad + wgrad launches)", "bound": "tensor",
                    "achieved": flops / ms / 1e9, "peak": tf32_peak, "unit": "TFLOP/s", "frac": flops / ms / 1e9 / tf32_peak,
                    "frac_counting_3xTF32_passes": flops * passes / ms / 1e9 / tf32_peak, "passes": passes,
                    "algorithmic_flops": flops, "traffic": None,
                    "peak_source": peaks["source"] + ": dense TF32 = measured bf16 / 2"}
    else:
        key = dom if dom in kernels else "adam_step"
        k = kernels.get(key)
        roofline = {"kernel": key, "bound": "hbm", "achieved": k["GBps"] if k else None, "peak": peaks["hbm_gbs"],
                    "unit": "GB/s", "frac": k["frac_of_measured_hbm"] if k else None,
                    "algorithmic_bytes": k["algorithmic_bytes"] if k else None, "traffic": None,
                    "peak_source": peaks["source"]}
    roofline["share_of_step"] = share
    # dram__bytes_read+write of one `ncu --set full` capture of the same command, N = 1 only (a shard of
    # the arena is a different launch: never reuse the N = 1 figure there)
    tpath = os.path.join(ROOT, "profiles", "r2_step_kernels_traffic.json")
    if world == 1 and args.workload == "deepfm" and os.path.exists(tpath):
        with open(tpath) as fd:
            cap = json.load(fd).get({"adam_step": "adam_kernel", "gemm": "gemm_tf32_kernel"}.get(dom, dom))
        if cap:
            roofline["traffic"] = (cap["dram_read_MB"] + cap["dram_write_MB"]) * 1e6
            roofline["traffic_source"] = "profiles/r2_step_kernels_traffic.json (ncu --set full, per launch)"
    line = {"metric": METRICS[args.workload], "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak" if args.workload == "deepfm" else "strong",
            "vs_baseline": None,
            "dtype": {"fp32": "f32", "tf32x3": "f32 (3xTF32 tensor-core GEMMs, fp32 everything else)",
                      "tf32": "tf32 GEMMs, f32 elsewhere",
                      "bf16": "bf16 GEMM operands (fp32 accumulation in TMEM), f32 tables / optimizer"}[args.precision],
            # `config` names the WORKLOAD only (both arms print the same dict); how this arm computes it:
            "data": "synthetic", "config": workload_config(args, world),
            "matmul": args.precision,
            "optimizer_pass": ("dense semantics, lazy row-wise evaluation" if args.lazy_adam and world == 1
                               else "dense pass over the arena"),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "samples/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": pipe.h2d_bytes_per_step * world, "d2h_bytes_per_step": pipe.d2h_bytes_per_step * world,
                    "api": "fuxictr_b200.pipeline.TrainPipeline.step (double-buffered H2D on a copy stream)"},
            "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches,
            "cuda_graph": pipe.graph is not None, "final_loss": final_loss,
            "roofline": roofline, "kernels": kernels, "step_profile": shares}
    if world == 1 and args.workload == "deepfm":
        del pipe, model
        torch.cuda.empty_cache()
        try:
            line["gather"] = {"c2": gather_points(peaks, VOCAB, "39 x 25,641 rows (64 MB: L2-resident)"),
                              "stress": gather_points(peaks, 4_000_000, "39 x 4 M rows (10 GB >> L2)")}
        except Exception as exc:  # e.g. a smaller GPU: report, do not hide
            line["gather"] = {"error": str(exc)}
        try:
            line["reference_gpu_eager"] = reference_gpu_eager(args, steps=args.steps)
        except Exception as exc:
            line["reference_gpu_eager"] = {"unavailable": repr(exc)}
    if world == 1 and not args.no_cpu_baseline and args.workload != "dlrm":
        r = cpu_reference_run(args, 0, 3, seconds=args.cpu_seconds)
        line["cpu_baseline"] = cpu_baseline_entry(r, args, "in %.0f s" % args.cpu_seconds)
    print(json.dumps(line))
    sys.stdout.flush()
    if world > 1:
        os._exit(0)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference_arm(a)
    elif a.impl == "reference-gpu":
        run_reference_gpu_arm(a)
    else:
        run_b200_arm(a)
