#!/usr/bin/env python
"""bench.py -- filtered link-prediction throughput (triples/s) on synthetic KGs.

    python bench.py --gpus N --steps K --warmup W [--workload c2] [--impl reference]

A "step" is ONE full filtered link-prediction evaluation of the workload's test set
(raw + filtered ranks of the true head and of the true tail of every test triple against all
entities) -- the metric BASELINE.json names.  Default workload: c2 = TransE-L2 d=200,
|E|=1M, |R|=1k, 20,466 test triples (the single-GPU configuration the metric is quoted on).
Other workloads: c1 (the reference's CPU-runnable case), c3 (ComplEx d=400), c4 (RotatE d=1000,
|E|=5M, entity table range-partitioned), c5 (DistMult d=200 training step: Bernoulli corruption
fused with scoring + margin loss; a "step" is one forward+backward over a batch).

Our arm (default) prints ONE JSON line on stdout (everything else, NCCL's init lines included,
goes to stderr) with
  value      whole-job triples/s, inputs already on the device (table, indices, filter CSR)
  e2e        the same through the public API (LinkPredictionEvaluator.evaluate) from HOST
             index tensors / filter sets to rank vectors on the host
  roofline   the dominant kernel: algorithmic flops (bytes) per launch / CUDA-event duration
  parity_full  every test triple: ranks of the timed path (tensor-core / approximate
             bound-and-refine) against the exact ATen-order scalar scan
  cpu_baseline  the CPU oracle (a PyTorch-CPU restatement of torchkge's path; the unmodified
             reference itself when oracle/_ref holds it) timed on a bounded sample of the same
             test set on this box's host cores, and a parity check of the GPU ranks on it
With N > 1 (torchrun) the job is decomposed BOTH ways the path allows (SURVEY.md section 8e)
and both are reported: "queries" -- table replicated, test triples sharded, no data-path
collective, rank vectors all-gathered -- and "entities" -- the north star's design: entity
table range-partitioned, every rank scans its rows for every query, ONE all-reduce of the rank
counters.  The headline `value` is the decomposition `config.parallelism` names (queries when
the table fits one GPU); the other one is the sub-record of its name.  Total work is fixed, so
"scaling" is "strong".

--impl reference times the reference's own CPU implementation of the path on a bounded
sample per step (oracle/_ref = the unmodified torchkge package when present, else the oracle
port oracle/kge_oracle.py, which tests/golden pins against it).

--dump-outputs DIR writes what the timed path computed in its last timed step as DIR/<name>.npy
(integers as float64, floating-point results as float32): the four rank vectors of a link-prediction
workload (rank_heads, rank_tails, filt_rank_heads, filt_rank_tails; with --impl reference, of the
last step's sample), or for c5 the loss, the relation gradient table and the gradient rows of a
fixed seeded sample of DUMP_ROWS entities (grad_ent_rows holds their ids).  Inputs are generated
from --seed, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the source tree may be read-only: nothing is written into it

# stdout carries exactly one JSON line: keep a private handle on it and point fd 1 at stderr, so
# that NCCL's INFO lines and any library chatter land on stderr
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)
sys.stdout = sys.stderr

import torch  # noqa: E402


def emit(record):
    _REAL_STDOUT.write(json.dumps(record) + "\n")
    _REAL_STDOUT.flush()


def _count(minimum):
    def parse(text):
        v = int(text)
        if v < minimum:
            raise argparse.ArgumentTypeError("must be >= %d" % minimum)
        return v
    return parse


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_count(1), default=3, help="timed steps")
    ap.add_argument("--warmup", type=_count(0), default=3, help="untimed steps before them")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--cpu-sample", type=int, default=0,
                    help="test triples in the CPU-baseline sample (0: 32 at |E| >= 100k, 1 for c4, else 2048)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the sub-records (second decomposition, reference-KG API, c5 training step)")
    ap.add_argument("--n-test", type=int, default=0, help="use only the first n test triples (0: all)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--split", default="auto", choices=["auto", "queries", "entities"],
                    help="multi-GPU decomposition reported as the headline value")
    ap.add_argument("--batch", type=int, default=32768, help="c5: positives per training step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (see the module docstring)")
    return ap.parse_args()


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the warm-up and timed steps run."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax = float(f[1]); power.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax,
                "power_w_max": max(power) if power else None, "samples": len(sm),
                "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- helpers
RANK_NAMES = ("rank_heads", "rank_tails", "filt_rank_heads", "filt_rank_tails")
DUMP_ROWS = 8192                 # c5: entity gradient rows written by --dump-outputs
DUMP_LIMIT = 64 << 20            # bytes, all files of one --dump-outputs together


def dump_rows(n_ent):
    """The fixed sample of entity rows whose gradients --dump-outputs writes for c5."""
    g = torch.Generator().manual_seed(0)
    return torch.randperm(n_ent, generator=g)[:DUMP_ROWS].sort().values


def dump_outputs(directory, arrays):
    """Write each tensor of `arrays` as directory/<name>.npy: integers as float64 (exact below
    2^53), floating-point values as float32."""
    import numpy as np
    host = {}
    for name, a in arrays.items():
        a = a.detach().cpu()
        host[name] = (a.float() if a.is_floating_point() else a.double()).numpy()
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT))
    os.makedirs(directory, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def dist_info():
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return rank, local, world


def row_bytes(code, dim):
    from torchkge_b200 import _lib
    return (8 if code in (_lib.COMPLEX, _lib.ROTATE) else 4) * dim


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def measured_peaks():
    p = _peaks()
    if "hbm_gbs" in p:
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    p = _peaks()
    if "bf16_tflops_sustained" in p:
        return float(p["bf16_tflops_sustained"]), "measured sustained bf16 (MEASURED_PEAKS.json)"
    return 1400.0, "fallback (B200_PROFILING.md sustained)"


class HostKG:
    """What LinkPredictionEvaluator reads from the REFERENCE's knowledge graph (SURVEY.md
    section 8b): index tensors + defaultdict(set) filter dictionaries."""

    def __init__(self, h, t, r, n_ent, n_rel, dh, dt):
        self.head_idx, self.tail_idx, self.relations = h, t, r
        self.n_ent, self.n_rel, self.n_facts = n_ent, n_rel, h.shape[0]
        self.dict_of_heads, self.dict_of_tails = dh, dt

    def __len__(self):
        return self.n_facts


class TableModel(torch.nn.Module):
    """A model object of the reference's class name wrapping pre-generated tables, so that
    the public evaluator can be driven with synthetic weights of any size."""

    def __init__(self, cls_name, diss, dim, n_ent, n_rel, tabs):
        super().__init__()
        self.__class__ = type(cls_name, (TableModel,), {})
        self.emb_dim, self.n_ent, self.n_rel = dim, n_ent, n_rel
        mk = lambda w: torch.nn.Embedding.from_pretrained(w, freeze=True)  # noqa: E731
        if cls_name == "TransEModel":
            from torchkge_b200.models import l1_dissimilarity, l2_dissimilarity
            self.dissimilarity = l1_dissimilarity if diss == "L1" else l2_dissimilarity
            self.ent_emb, self.rel_emb = mk(tabs["ent0"]), mk(tabs["rel0"])
        elif cls_name == "DistMultModel":
            self.ent_emb, self.rel_emb = mk(tabs["ent0"]), mk(tabs["rel0"])
        elif cls_name == "RESCALModel":
            self.ent_emb, self.rel_mat = mk(tabs["ent0"]), mk(tabs["rel0"])
        elif cls_name == "ComplExModel":
            self.re_ent_emb, self.im_ent_emb = mk(tabs["ent0"]), mk(tabs["ent1"])
            self.re_rel_emb, self.im_rel_emb = mk(tabs["rel0"]), mk(tabs["rel1"])
        elif cls_name == "RotatEModel":
            self.re_ent_emb, self.im_ent_emb = mk(tabs["ent0"]), mk(tabs["ent1"])
            self._planes = (tabs["rel0"], tabs["rel1"])

    def relation_planes(self):
        return self._planes


METRIC = "filtered link-prediction triples/sec (full hits@k/MRR eval)"


def table_bytes(wl):
    return wl["n_ent"] * wl["dim"] * (8 if wl["model"] in ("ComplEx", "RotatE") else 4)


def split_mode(args, wl, world):
    """single | queries (replicated table, test triples sharded) | entities (table range-partitioned)"""
    if world == 1:
        return "single"
    if args.split != "auto":
        return args.split
    return "entities" if table_bytes(wl) > 24e9 else "queries"


def parallelism_text(mode, world):
    return {"single": "single GPU",
            "queries": "test triples sharded x%d, table replicated, no data-path collective "
                       "(rank vectors all-gathered inside the timed region)" % world,
            "entities": "entity table range-partitioned x%d (each rank holds and scans only its rows), query rows "
                        "exchanged by all-reduce, 1 all-reduce of the rank counters (inside the timed region)" % world}[mode]


def workload_config(name, wl, world, mode="single", n_test=None):
    return {"workload": "%s: %s%s dim=%d |E|=%d |R|=%d, %d test triples, full filtered LP (head+tail)" % (
                name, wl["model"], ("-" + wl["diss"]) if wl["diss"] else "", wl["dim"], wl["n_ent"],
                wl["n_rel"], n_test if n_test is not None else wl["n_test"]),
            "n_facts_requested": wl["n_facts"],
            "parallelism": parallelism_text(mode, world),
            "l2_policy": l2_policy(wl)}


def l2_policy(wl):
    mb = table_bytes(wl) / 1e6
    if mb > 126:
        return "inputs larger than L2 (table %.0f MB >> 126 MB)" % mb
    return ("table %.1f MB is L2-resident: plumbing / parity configuration, no L2 flush between steps, "
            "HBM fractions are meaningless here" % mb)


def oracle_params_from_tables(kind, tabs):
    if kind in ("transe_l1", "transe_l2", "distmult"):
        return {"ent": tabs["ent0"], "rel": tabs["rel0"]}
    if kind == "rescal":
        return {"ent": tabs["ent0"], "rel_mat": tabs["rel0"]}
    return {"re_ent": tabs["ent0"], "im_ent": tabs["ent1"], "re_rel": tabs["rel0"], "im_rel": tabs["rel1"]}


# ----------------------------------------------------------------------------- CPU reference
def import_reference():
    """The unmodified torchkge package, if a copy travels with the repo (oracle/_ref, built by
    oracle/make_ref.sh from /root/reference; git-ignored) -- else None."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "torchkge")):
        return None
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    try:
        import torchkge  # noqa: F401
        return torchkge
    except Exception as e:  # a dependency of the reference missing on this box
        print("reference import failed: %r" % (e,), file=sys.stderr)
        return None


def reference_model(torchkge, kind, wl, P):
    """A model of the UNMODIFIED reference holding the synthetic tables."""
    from torchkge.models import ComplExModel, DistMultModel, RESCALModel, TransEModel
    d, ne, nr = wl["dim"], wl["n_ent"], wl["n_rel"]
    if kind in ("transe_l1", "transe_l2"):
        m = TransEModel(d, ne, nr, dissimilarity_type="L1" if kind == "transe_l1" else "L2")
        m.ent_emb.weight.data, m.rel_emb.weight.data = P["ent"], P["rel"]
    elif kind == "distmult":
        m = DistMultModel(d, ne, nr)
        m.ent_emb.weight.data, m.rel_emb.weight.data = P["ent"], P["rel"]
    elif kind == "rescal":
        m = RESCALModel(d, ne, nr)
        m.ent_emb.weight.data, m.rel_mat.weight.data = P["ent"], P["rel_mat"]
    elif kind == "complex":
        m = ComplExModel(d, ne, nr)
        m.re_ent_emb.weight.data, m.im_ent_emb.weight.data = P["re_ent"], P["im_ent"]
        m.re_rel_emb.weight.data, m.im_rel_emb.weight.data = P["re_rel"], P["im_rel"]
    else:
        return None
    return m


class CpuReference:
    """Ranks of test triples from the reference's CPU path.  kind "reference": torchkge's own
    LinkPredictionEvaluator on a torchkge model holding the same tables; kind "port": the oracle
    restatement (RotatE, which the reference does not have, and any box without oracle/_ref)."""

    def __init__(self, kind, wl, P):
        self.kind_name, self.wl, self.P = kind, wl, P
        self.impl = "port"
        self.model = None
        tk_ref = import_reference()
        if tk_ref is not None and kind != "rotate":
            try:
                self.model = reference_model(tk_ref, kind, wl, P)
                self.tk_ref = tk_ref
                if self.model is not None:
                    self.impl = "reference"
            except Exception as e:
                print("reference model construction failed: %r" % (e,), file=sys.stderr)
                self.model = None

    def ranks(self, th, tt, tr, dh, dt, b_size):
        """(rank_heads, rank_tails, filt_rank_heads, filt_rank_tails) CPU int64"""
        if self.impl == "reference":
            from torchkge.evaluation import LinkPredictionEvaluator as RefEvaluator
            kg = HostKG(th, tt, tr, self.wl["n_ent"], self.wl["n_rel"], dh, dt)
            ev = RefEvaluator(self.model, kg)
            ev.evaluate(b_size=b_size, verbose=False)
            return (ev.rank_true_heads, ev.rank_true_tails, ev.filt_rank_true_heads,
                    ev.filt_rank_true_tails)
        from oracle import kge_oracle as oracle
        return oracle.link_prediction(self.kind_name, self.P, th, tt, tr, dh, dt, b_size)


def oracle_ranks_sharded(kind, code, wl, seed, th, tt, tr, dh, dt, dev, n_shards):
    """Oracle ranks for a table too large to score in one piece on the host (c4: 40 GB):
    rank = sum over entity-range shards of #{c in shard : s_c >= s_true} (SURVEY.md section 8e),
    each shard regenerated from its seed, scored with the oracle's all-entity scorer against the
    shard rows plus the query's own head / tail rows (appended, so that s_true comes out of the same
    arithmetic).  Returns (ranks 4-tuple, seconds spent in the oracle's scoring + counting)."""
    from oracle import kge_oracle as oracle
    from torchkge_b200 import synthetic as S
    n = th.numel()
    n_ent, n_rel, dim = wl["n_ent"], wl["n_rel"], wl["dim"]
    hq = S.rows_by_id(code, dim, n_ent, seed, th, dev)
    tq = S.rows_by_id(code, dim, n_ent, seed, tt, dev)
    hq = {k: (v.cpu() if v is not None else None) for k, v in hq.items()}
    tq = {k: (v.cpu() if v is not None else None) for k, v in tq.items()}
    raw = torch.zeros((2, n), dtype=torch.int64)   # tail, head
    sub = torch.zeros((2, n), dtype=torch.int64)
    per = (n_ent + n_shards - 1) // n_shards
    cpu_s = 0.0
    for s in range(n_shards):
        lo, hi = min(n_ent, s * per), min(n_ent, (s + 1) * per)
        if hi <= lo:
            continue
        print("cpu oracle: entity rows [%d, %d) (%d of %d), %.0f s of scoring so far" % (lo, hi, s + 1, n_shards, cpu_s),
              file=sys.stderr, flush=True)
        tabs = S.make_tables(code, dim, n_ent, n_rel, lo, hi, seed, dev)
        tabs = {k: (v.cpu() if v is not None else None) for k, v in tabs.items()}
        rows = hi - lo
        for i in range(n):     # one query at a time: temporaries stay at (rows, dim) floats
            ext = {"ent0": torch.cat([tabs["ent0"], hq["ent0"][i:i + 1], tq["ent0"][i:i + 1]]),
                   "ent1": None if tabs["ent1"] is None else
                   torch.cat([tabs["ent1"], hq["ent1"][i:i + 1], tq["ent1"][i:i + 1]]),
                   "rel0": tabs["rel0"], "rel1": tabs["rel1"]}
            P = oracle_params_from_tables(kind, ext)
            hi_, ti_ = torch.tensor([rows]), torch.tensor([rows + 1])
            for which, side in ((0, "tail"), (1, "head")):
                t0 = time.perf_counter()
                sc = oracle.scores_all(kind, P, hi_, ti_, tr[i:i + 1], side)[0]
                s_true = sc[rows + 1] if side == "tail" else sc[rows]
                shard_sc = sc[:rows]
                raw[which, i] += int((shard_sc >= s_true).sum())
                cpu_s += time.perf_counter() - t0
                true = int(tt[i]) if side == "tail" else int(th[i])
                key = (int(th[i]), int(tr[i])) if side == "tail" else (int(tt[i]), int(tr[i]))
                fset = (dt if side == "tail" else dh).get(key)
                if fset is not None and true in fset:      # get_true_targets' quirk otherwise
                    for c in fset:
                        if c != true and lo <= c < hi:
                            sub[which, i] += int(shard_sc[c - lo] >= s_true) - int(s_true == float("-inf"))
        del tabs
    return (raw[1], raw[0], raw[1] - sub[1], raw[0] - sub[0]), cpu_s


# ----------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    """The reference's CPU path on a bounded sample per step; rank 0 only."""
    if rank != 0:
        return
    from torchkge_b200 import synthetic as S
    if args.workload == "c5":
        return run_reference_c5(args)
    wl = S.WORKLOADS[args.workload]
    code = S.MODEL_CODE[(wl["model"], wl["diss"])]
    kind = S.ORACLE_KIND[code]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    dev = torch.device("cuda:0") if torch.cuda.is_available() else torch.device("cpu")
    big = wl["n_ent"] >= 100000
    graph = S.make_graph(wl["n_ent"], wl["n_rel"], wl["n_facts"], wl["n_test"], args.seed, dev)
    per_step = (2 if args.workload == "c4" else 8) if big else 1024
    total = min(per_step * (args.steps + args.warmup), graph["test_h"].numel())
    per_step = max(1, total // (args.steps + args.warmup))
    dh, dt = S.filters_as_dicts(graph, wl["n_ent"], wl["n_rel"], limit=total)
    th, tt, tr = (graph[k][:total].cpu() for k in ("test_h", "test_t", "test_r"))
    b_size = 4 if big else 256
    sharded = table_bytes(wl) > 8e9
    last = {}
    if sharded:
        impl = "port"

        def step(i):
            lo, hi = i * per_step, (i + 1) * per_step
            last["ranks"], s_ = oracle_ranks_sharded(kind, code, wl, args.seed, th[lo:hi], tt[lo:hi], tr[lo:hi],
                                                     dh, dt, dev, 8)
            return s_
    else:
        tabs = S.make_tables(code, wl["dim"], wl["n_ent"], wl["n_rel"], 0, wl["n_ent"], args.seed, dev)
        P = oracle_params_from_tables(kind, {k: (v.cpu() if v is not None else None) for k, v in tabs.items()})
        ref = CpuReference(kind, wl, P)
        impl = ref.impl

        def step(i):
            lo, hi = i * per_step, (i + 1) * per_step
            t0 = time.perf_counter()
            last["ranks"] = ref.ranks(th[lo:hi], tt[lo:hi], tr[lo:hi], dh, dt, b_size)
            return time.perf_counter() - t0

    for i in range(args.warmup):
        step(i)
    el = 0.0
    for i in range(args.steps):
        el += step(args.warmup + i)
    value = args.steps * per_step / el
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(RANK_NAMES, last["ranks"])))
    sample = "%d test triples per step (b_size %d) of workload %s%s" % (
        per_step, 1 if sharded else b_size, args.workload,
        ", table scored in 8 entity-range pieces (40 GB does not fit the scorer's temporaries)" if sharded else "")
    mode = split_mode(args, wl, world)
    emit({
        "impl": "reference", "metric": METRIC,
        "value": value, "unit": "triples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000 * el / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, wl, world, mode),
        "cpu_baseline": {"value": value, "unit": "triples/s", "cores": cores, "kind": impl,
                         "sample": sample,
                         "what": "unmodified torchkge LinkPredictionEvaluator on CPU (oracle/_ref)"
                                 if impl == "reference" else "oracle port oracle/kge_oracle.py (pinned by tests/golden)"},
        "e2e": {"value": value, "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


def run_reference_c5(args):
    from oracle import kge_oracle as oracle
    from torchkge_b200 import _lib, synthetic as S
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    c5 = S.C5
    b = 4096
    tabs = S.make_tables(_lib.DISTMULT, c5["dim"], c5["n_ent"], c5["n_rel"], 0, c5["n_ent"], args.seed,
                         torch.device("cpu"))
    P = {"ent": tabs["ent0"].requires_grad_(True), "rel": tabs["rel0"].requires_grad_(True)}
    g = torch.Generator().manual_seed(1)
    probs = torch.rand(c5["n_rel"], generator=g) * 0.8 + 0.1

    rows = dump_rows(c5["n_ent"])
    last = {}

    def step():
        h = torch.randint(0, c5["n_ent"], (b,), generator=g)
        t = torch.randint(0, c5["n_ent"], (b,), generator=g)
        r = torch.randint(0, c5["n_rel"], (b,), generator=g)
        t0 = time.perf_counter()
        nh, nt = oracle.corrupt_batch(h, t, r, probs, c5["n_ent"], c5["n_neg"])
        pos, neg = oracle.forward_pos_neg("distmult", P, h, t, r, nh, nt)
        loss = oracle.margin_loss(pos, neg, 1.0)
        loss.backward()
        el_ = time.perf_counter() - t0
        if args.dump_outputs:
            last.update(loss=loss.detach().view(1), grad_ent_rows=rows, grad_ent=P["ent"].grad[rows],
                        grad_rel=P["rel"].grad.clone())
        for p in P.values():
            p.grad = None
        return el_

    for _ in range(args.warmup):
        step()
    steps = args.steps
    el = sum(step() for _ in range(steps))
    value = steps * b / el
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    emit({"impl": "reference", "metric": C5_METRIC, "value": value, "unit": "positives/s", "n_gpus": args.gpus,
          "steps": steps, "warmup": args.warmup, "ms_per_step": 1000 * el / steps,
          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
          "config": {"workload": c5_workload_text(b)},
          "cpu_baseline": {"value": value, "unit": "positives/s", "cores": cores, "kind": "port",
                           "sample": "%d steps at B=%d (oracle: corrupt_batch + forward_pos_neg + margin_loss + "
                                     "autograd backward)" % (steps, b)},
          "e2e": {"value": value, "unit": "positives/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
          "gpu_launches": 0})


# ----------------------------------------------------------------------------- our arm: link prediction
def run_ours(args, rank, local, world):
    import torch.distributed as dist
    from torchkge_b200 import _lib, synthetic as S
    from torchkge_b200.engine import (CudaEngine, EntityShard, ModelSpec, QueryShard,
                                      rank_link_prediction)
    import torchkge_b200.engine as engine_mod
    from torchkge_b200.evaluation import LinkPredictionEvaluator
    from torchkge_b200.data import KnowledgeGraph

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL's init lines (rank count, transport, NVLS) go to stderr with everything else
        if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
            os.environ["NCCL_DEBUG"] = "INFO"          # the image default (VERSION) hides the rank / transport lines
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        dist.init_process_group("nccl", device_id=dev)
    if args.workload == "c5":
        return run_c5(args, rank, world, dev)
    wl = dict(S.WORKLOADS[args.workload])
    code = S.MODEL_CODE[(wl["model"], wl["diss"])]
    n_ent, n_rel, dim = wl["n_ent"], wl["n_rel"], wl["dim"]
    fits = table_bytes(wl) <= 24e9
    primary = split_mode(args, wl, world)
    modes = [primary]
    if world > 1 and fits and not args.no_extras:
        modes.append("entities" if primary == "queries" else "queries")

    graph = S.make_graph(n_ent, n_rel, wl["n_facts"], wl["n_test"], args.seed, dev)
    if args.n_test:
        for k in ("test_h", "test_t", "test_r"):
            graph[k] = graph[k][:args.n_test].contiguous()
    t0 = time.perf_counter()
    csr_t, csr_h = S.make_filters(graph, n_ent, n_rel)
    torch.cuda.synchronize()
    csr_build_s = time.perf_counter() - t0
    n_test = graph["test_h"].numel()
    eng = CudaEngine()
    engine_mod._default_engine = eng  # the evaluator uses the same instance (launch counting)
    peak, peak_src = measured_peaks()
    rb = row_bytes(code, dim)
    full_tabs = {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def measure(mode, clocks):
        """One decomposition: device-resident timing, end-to-end timing, full-test-set parity of the
        timed path against the exact scalar scan."""
        # entity decomposition: every rank generates and HOLDS only its range of rows (the table is
        # range-partitioned for real, also when it would fit one GPU)
        local_storage = mode == "entities"
        shard = EntityShard(n_ent, rank, world, None, local_storage=True) if mode == "entities" else None
        if local_storage:
            lo, hi = shard.lo, shard.hi
            tabs = S.make_tables(code, dim, n_ent, n_rel, lo, hi, args.seed, dev)
        else:
            lo, hi = 0, n_ent
            if not full_tabs:
                full_tabs.update(S.make_tables(code, dim, n_ent, n_rel, 0, n_ent, args.seed, dev))
            tabs = full_tabs
        qshard = QueryShard(n_test, rank, world) if mode == "queries" else QueryShard(n_test, 0, 1)
        my_h, my_t, my_r = qshard.slice(graph["test_h"], graph["test_t"], graph["test_r"])
        my_csr_t, my_csr_h = qshard.csr(csr_t), qshard.csr(csr_h)
        spec = ModelSpec(code, dim, n_ent, n_rel, tabs["ent0"], tabs["ent1"], tabs["rel0"], tabs["rel1"],
                         ent_lo=lo)
        rows_here = (shard.hi - shard.lo) if shard is not None else n_ent
        n_my = qshard.hi - qshard.lo

        def device_step(exact=False):
            lazy = rank_link_prediction(spec, my_h, my_t, my_r, my_csr_t, my_csr_h, shard=shard, engine=eng,
                                        exact=exact, sync=False)
            ranks = qshard.all_gather(lazy.ranks) if mode == "queries" else list(lazy.ranks)
            return ranks, lazy

        # ---- device-resident timing (no host synchronisation inside a step) ----
        if clocks is not None:
            clocks.start()
        for _ in range(args.warmup):
            ranks_dev, lazy = device_step()
        barrier()
        _lib.scan_timing_enable(True)
        for kind_ in (0, 1, 2):
            _lib.scan_timing_read(kind_)
        launches0 = eng.launches
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pending = []
        ev0.record()
        for _ in range(args.steps):
            ranks_dev, lazy = device_step()
            pending.append(lazy)
        ev1.record()
        barrier()
        dev_ms = ev0.elapsed_time(ev1)
        overflowed = sum(int(lz.overflow.item()) for lz in pending if lz.overflow is not None)
        if eng.trace is not None and rank == 0:   # KGE_TRACE=1: where the steps spent their time
            for lab, host_ms, dev_ms_ in eng.trace_report():
                print("trace %-28s host %9.3f ms  device %9.3f ms" % (lab, host_ms, dev_ms_), file=sys.stderr)
        launches = eng.launches - launches0
        scan_n, scan_ms = _lib.scan_timing_read(0)
        tc_n, tc_ms = _lib.scan_timing_read(1)
        rc_n, rc_ms = _lib.scan_timing_read(2)
        _lib.scan_timing_enable(False)
        clock_rec = clocks.stop() if clocks is not None else None
        dev_ms = max_over_ranks(dev_ms)
        value = args.steps * n_test / (dev_ms / 1000.0)
        calls_per_step = 2 * ((n_my + engine_mod.DEFAULT_CHUNK - 1) // engine_mod.DEFAULT_CHUNK)
        near_ties = None
        if eng.tc_stats:
            near_ties = float(sum(int(s_[0]) for s_ in eng.tc_stats[-calls_per_step:]))

        # ---- end-to-end through the public API, host buffers in, host ranks out ----
        model = TableModel(wl["model"] + "Model", wl["diss"], dim, n_ent, n_rel, tabs)
        t0 = time.perf_counter()
        kg = KnowledgeGraph(graph["test_h"].cpu(), graph["test_t"].cpu(), graph["test_r"].cpu(), n_ent, n_rel,
                            filter_facts=(graph["heads"], graph["tails"], graph["rels"]))   # index built on the device
        kg.head_idx, kg.tail_idx, kg.relations = (x.pin_memory() for x in (kg.head_idx, kg.tail_idx, kg.relations))
        filter_index_build_s = time.perf_counter() - t0
        evaluator = LinkPredictionEvaluator(model, kg, shard=qshard if mode == "queries" else shard)
        for _ in range(min(args.warmup, 2)):
            evaluator.evaluate(b_size=256, verbose=False)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            evaluator.evaluate(b_size=256, verbose=False)
        barrier()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        e2e_value = args.steps * n_test / e2e_s
        api_ranks = (evaluator.rank_true_heads, evaluator.rank_true_tails,
                     evaluator.filt_rank_true_heads, evaluator.filt_rank_true_tails)
        same = all(torch.equal(a.cpu(), b) for a, b in zip(ranks_dev, api_ranks))

        # ---- parity at full size: the timed path against the exact ATen-order scalar scan ----
        t0 = time.perf_counter()
        exact_ranks, _ = device_step(exact=True)
        torch.cuda.synchronize()
        exact_s = time.perf_counter() - t0
        names = ["rank_heads", "rank_tails", "filt_rank_heads", "filt_rank_tails"]
        eq = [bool(torch.equal(a, b)) for a, b in zip(ranks_dev, exact_ranks)]
        differing = int(sum((a != b).sum().item() for a, b in zip(ranks_dev, exact_ranks)))
        parity_full = {"n": int(ranks_dev[0].numel()), "ranks_equal": all(eq), "vectors": dict(zip(names, eq)),
                       "rank_entries_differing": differing, "near_tie_pairs": near_ties,
                       "near_tie_list_overflows": overflowed,
                       "timed_path": ("tcgen05 bound-and-refine" if tc_n > 0 else
                                      ("approximate-sqrt bound-and-refine" if code == _lib.ROTATE and eng.tensor_core
                                       else "exact scalar scan (no approximate path for this model)")),
                       "against": "exact ATen-order scalar scan (oracle-validated, bit-exact) on all test triples",
                       "exact_scan_s": exact_s}

        # ---- roofline of the dominant kernel ----
        sm_mhz = (clock_rec or {}).get("sm_mhz") or 1965.0
        if tc_n > 0:
            # tensor-core bound-and-refine scan: split GEMM (3 MMAs per fp32 product)
            k_total = dim * (2 if code == _lib.COMPLEX else 1)
            ms_per_launch = tc_ms / tc_n
            alg_flops = 2.0 * n_my * rows_here * k_total            # the fp32 contraction itself (this rank)
            tensor_peak = measured_tensor_peak()
            ach = alg_flops / (ms_per_launch / 1000.0) / 1e12
            roofline = {
                "kernel": "tc_scan_kernel (tcgen05 split GEMM, 3 MMAs per fp32 product, threshold epilogue)",
                "bound": "tensor", "achieved": ach, "peak": tensor_peak[0], "unit": "TFLOP/s",
                "frac": ach / tensor_peak[0], "peak_source": tensor_peak[1],
                "traffic": TRAFFIC.get((args.workload, world)),
                "traffic_source": "constant copied from the committed ncu --set full capture of this launch shape "
                                  "(profiles/, see DESIGN.md section 5); not measured inside this run",
                "launches_timed": tc_n, "ms_per_launch": ms_per_launch,
                "scan_share_of_step": tc_ms / dev_ms if dev_ms > 0 else None,
                "recheck_ms_per_launch": rc_ms / max(1, rc_n),
                "recheck_share_of_step": rc_ms / dev_ms if dev_ms > 0 else None,
                "near_tie_pairs_per_step": near_ties,
                "near_tie_fraction": (near_ties / (2.0 * max(1, n_my) * rows_here)) if near_ties is not None else None,
                "executed_tflops": 3 * ach, "executed_frac_of_peak": 3 * ach / tensor_peak[0],
                "note": "algorithmic flops = 2 x queries x rows x K (the fp32 contraction); the kernel executes "
                        "3 half-precision MMAs per product (hi*hi + lo*hi + hi*lo), i.e. 3x the algorithmic "
                        "flops, so frac <= 1/3 by construction; near-ties are re-scored exactly so ranks stay "
                        "bit-identical (parity_full)",
            }
        else:
            # scalar fp32 scan.  algorithmic bytes per launch = queries x candidate rows x row_bytes
            # (SURVEY.md 8d: 2*nE*row_bytes per triple = nE*row_bytes per (triple, side) launch unit)
            alg_bytes_per_launch = float(n_my) * rows_here * rb
            scan_ms_per_launch = scan_ms / max(1, scan_n)
            achieved = alg_bytes_per_launch / (scan_ms_per_launch / 1000.0) / 1e9
            refine_rot = code == _lib.ROTATE and eng.tensor_core   # approximate-sqrt bound-and-refine scan
            ops_per_elem = {_lib.TRANSE_L1: 2.5, _lib.TRANSE_L2: 3.5, _lib.DISTMULT: 2.0, _lib.RESCAL: 2.0,
                            _lib.COMPLEX: 4.0, _lib.ROTATE: 5.0 if refine_rot else 16.0}[code]  # fp32 ops per (q,c,k)
            lane_ops = float(n_my) * rows_here * dim * ops_per_elem
            fp32_peak = 148 * 128 * sm_mhz * 1e6
            roofline = {
                "kernel": "scan_kernel (dense rank scan, fp32 pipes)", "bound": "hbm", "achieved": achieved,
                "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                "traffic": None,
                "launches_timed": scan_n, "ms_per_launch": scan_ms_per_launch,
                "scan_share_of_step": scan_ms / dev_ms if dev_ms > 0 else None,
                "recheck_ms_per_launch": rc_ms / max(1, rc_n) if rc_n else None,
                "recheck_share_of_step": (rc_ms / dev_ms) if (rc_n and dev_ms > 0) else None,
                "near_tie_pairs_per_step": near_ties,
                "near_tie_fraction": (near_ties / (2.0 * max(1, n_my) * rows_here)) if near_ties is not None else None,
                "note": "algorithmic bytes = queries x rows x row_bytes per launch; every streamed candidate "
                        "tile is shared by 64 queries per CTA, so DRAM traffic is ~1/64 of this and the "
                        "kernel is fp32-issue bound (see fp32_issue)",
                "fp32_issue": {"achieved_tlaneops": lane_ops / (scan_ms_per_launch / 1000.0) / 1e12,
                               "peak_tlaneops": fp32_peak / 1e12,
                               "frac": lane_ops / (scan_ms_per_launch / 1000.0) / fp32_peak,
                               "ops_per_element": ops_per_elem},
            }
            if refine_rot:
                # one MUFU.SQRT per element at 16 per clock and SM is the binding unit of this form
                elems = float(n_my) * rows_here * dim
                mufu_peak = 148 * 16 * sm_mhz * 1e6
                roofline["mufu"] = {"achieved_telem": elems / (scan_ms_per_launch / 1000.0) / 1e12,
                                    "peak_telem": mufu_peak / 1e12,
                                    "frac": elems / (scan_ms_per_launch / 1000.0) / mufu_peak}
                roofline["kernel"] = "scan_kernel<EL_ROT, APPROX> (approximate-sqrt bound-and-refine, fp32 pipes + MUFU)"
        import hashlib
        flat = torch.cat([x.view(-1) for x in ranks_dev]).cpu()
        digest = hashlib.sha256(flat.numpy().tobytes()).hexdigest()[:16]
        rec = {
            "value": value, "unit": "triples/s", "ms_per_step": dev_ms / args.steps,
            # identical across GPU counts and decompositions iff the rank vectors are (same test set)
            "ranks_sha256_16": digest,
            "ranks_first8": [x[:8].tolist() for x in ranks_dev],
            "parallelism": parallelism_text(mode, world),
            "e2e": {"value": e2e_value, "unit": "triples/s",
                    "h2d_bytes_per_step": evaluator.last_stats.get("h2d_bytes"),
                    "d2h_bytes_per_step": evaluator.last_stats.get("d2h_bytes"),
                    "ms_per_step": 1000 * e2e_s / args.steps,
                    "api": "LinkPredictionEvaluator(model, kg).evaluate(b_size=256), kg = torchkge_b200.KnowledgeGraph "
                           "(pinned host index tensors; sorted-array filter index of all facts, built and resident on the device)",
                    "equals_device_ranks": bool(same)},
            "gpu_launches": launches, "roofline": roofline, "parity_full": parity_full,
            "filter_index_build_s": filter_index_build_s,
        }
        return rec, clock_rec, ranks_dev, tabs, model

    clocks = ClockSampler(local) if rank == 0 else None
    recs = {}
    main_ranks = main_tabs = main_model = clock_rec = None
    for i, mode in enumerate(modes):
        rec, cr, ranks_dev, tabs, model = measure(mode, clocks if i == 0 else None)
        recs[mode] = rec
        if i == 0:
            clock_rec, main_ranks, main_tabs, main_model = cr, ranks_dev, tabs, model

    # ---- CPU baseline on a bounded sample + parity of the headline ranks on that sample ----
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        kind = S.ORACLE_KIND[code]
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        big = n_ent >= 100000
        sharded = table_bytes(wl) > 8e9
        ns = args.cpu_sample or ((1 if sharded else 32) if big else 2048)   # a 40 GB table costs minutes per triple
        ns = min(n_test, ns)
        th, tt, tr = (graph[k][:ns].cpu() for k in ("test_h", "test_t", "test_r"))
        dh, dt = S.filters_as_dicts(graph, n_ent, n_rel, limit=ns)  # reference-style dicts, sample keys
        b_size = 4 if big else 256
        if sharded:
            ref, cpu_s = oracle_ranks_sharded(kind, code, wl, args.seed, th, tt, tr, dh, dt, dev, 8)
            impl, what = "port", ("oracle port, table scored in 8 entity-range pieces regenerated from their "
                                  "seeds (40 GB table); time = scoring + counting only")
        else:
            full = main_tabs if main_tabs["ent0"].shape[0] == n_ent else full_tabs
            if not full:
                full = S.make_tables(code, dim, n_ent, n_rel, 0, n_ent, args.seed, dev)
            P = oracle_params_from_tables(kind, {k: (v.cpu() if v is not None else None) for k, v in full.items()})
            refimpl = CpuReference(kind, wl, P)
            t0 = time.perf_counter()
            ref = refimpl.ranks(th, tt, tr, dh, dt, b_size)
            cpu_s = time.perf_counter() - t0
            impl = refimpl.impl
            what = ("unmodified torchkge LinkPredictionEvaluator on CPU (oracle/_ref)" if impl == "reference"
                    else "oracle port oracle/kge_oracle.py (pinned by tests/golden)")
        got = [x[:ns].cpu() for x in main_ranks]
        equal = [bool(torch.equal(a, b)) for a, b in zip(got, ref)]
        cpu = {"value": ns / cpu_s, "unit": "triples/s", "cores": cores, "kind": impl, "what": what,
               "sample": "first %d test triples, b_size %d, torch %s CPU, %d threads" % (
                   ns, 1 if sharded else b_size, torch.__version__, cores),
               "parity_on_sample": {"ranks_equal": all(equal), "n": ns,
                                    "vectors": dict(zip(["rank_heads", "rank_tails", "filt_rank_heads",
                                                         "filt_rank_tails"], equal))}}

    # ---- extras (single GPU only): the reference's own KnowledgeGraph containers; c5 training step ----
    extras = {}
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            extras["api_reference_kg"] = measure_reference_kg(S, graph, wl, main_model, main_ranks, args)
        except Exception as e:   # never lose the headline over an extra
            extras["api_reference_kg"] = {"error": repr(e)}
        if args.workload == "c2":
            try:
                extras["c5_training_step"] = measure_c5(args, dev, cpu_steps=0 if args.no_cpu_baseline else 1)
            except Exception as e:
                extras["c5_training_step"] = {"error": repr(e)}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    head = recs[primary]
    out = {
        "metric": METRIC, "value": head["value"], "unit": "triples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, wl, world, primary, n_test),
        "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": clock_rec,
        "roofline": head["roofline"], "parity_full": head["parity_full"], "cpu_baseline": cpu,
        "ranks_sha256_16": head["ranks_sha256_16"], "ranks_first8": head["ranks_first8"],
        "filter_csr_build_s": csr_build_s, "filter_index_build_s": head["filter_index_build_s"],
        "mean_filter_set": float(csr_t[1].numel() + csr_h[1].numel()) / (2 * n_test),
    }
    for mode in modes[1:]:
        out[mode] = recs[mode]
    out.update(extras)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(RANK_NAMES, main_ranks)))
    emit(out)
    if world > 1:
        dist.destroy_process_group()


# dram__bytes_read.sum + dram__bytes_write.sum of ONE tc_scan launch, from the committed ncu capture
# profiles/r02_tc_scan_fp16_ncu_summary.md (the 0.9 GB operand image read once + the near-tie list writes)
TRAFFIC = {("c2", 1): 1.025e9 + 0.037e9,
           # profiles/r02_tc_scan_c3_ncu_summary.md: both operand images stream at K = 800 (no resident query image)
           ("c3", 1): 12.975e9 + 0.156e9}


def measure_reference_kg(S, graph, wl, model, ranks_dev, args):
    """The drop-in case: LinkPredictionEvaluator driven with the REFERENCE's containers (index tensors
    + defaultdict(set) dictionaries, as torchkge.data_structures.KnowledgeGraph holds them)."""
    from torchkge_b200.evaluation import LinkPredictionEvaluator
    n_ent, n_rel = wl["n_ent"], wl["n_rel"]
    n_test = graph["test_h"].numel()
    t0 = time.perf_counter()
    dh, dt = S.filters_as_dicts(graph, n_ent, n_rel, limit=None)
    dict_build_s = time.perf_counter() - t0
    kg = HostKG(graph["test_h"].cpu(), graph["test_t"].cpu(), graph["test_r"].cpu(), n_ent, n_rel, dh, dt)
    ev = LinkPredictionEvaluator(model, kg)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ev.evaluate(b_size=256, verbose=False)
    first_s = time.perf_counter() - t0
    steps = max(2, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(steps):
        ev.evaluate(b_size=256, verbose=False)
    steady_s = (time.perf_counter() - t0) / steps
    got = (ev.rank_true_heads, ev.rank_true_tails, ev.filt_rank_true_heads, ev.filt_rank_true_tails)
    same = all(torch.equal(a.cpu(), b) for a, b in zip(ranks_dev, got))
    return {"first_call": {"value": n_test / first_s, "unit": "triples/s", "s": first_s},
            "steady_state": {"value": n_test / steady_s, "unit": "triples/s", "s": steady_s, "calls": steps},
            "equals_device_ranks": bool(same),
            "api": "LinkPredictionEvaluator(model, kg).evaluate(b_size=256) with kg.dict_of_heads / dict_of_tails "
                   "= defaultdict(set) as in torchkge.data_structures.KnowledgeGraph; the first call flattens the "
                   "distinct keys' sets on the host and expands rows on the device, later calls reuse the device CSR "
                   "cached on the graph object",
            "bench_side_dict_build_s": dict_build_s}


# ----------------------------------------------------------------------------- c5: fused training step
C5_METRIC = "training-step positives/sec (Bernoulli corruption n_neg=256 fused with scoring + margin loss, fwd+bwd)"


def c5_workload_text(b):
    from torchkge_b200 import synthetic as S
    c5 = S.C5
    return ("c5: DistMult dim=%d |E|=%d |R|=%d, B=%d positives per step, n_neg=%d, margin 1.0, Bernoulli "
            "corruption; random 800-byte row gathers over an 800 MB table (inputs larger than L2)"
            % (c5["dim"], c5["n_ent"], c5["n_rel"], b, c5["n_neg"]))


def measure_c5(args, dev, cpu_steps=1, batches=(4096, 32768), reps=None, warm=3, outputs=None):
    """C5 (BASELINE.json configs[4]) on one GPU: forward and forward+backward of the fused step,
    HBM roofline on SURVEY.md section 8d's algorithmic bytes ((n_neg + 3) * 4d forward, x3 with
    backward, per positive), parity with supplied negatives against the oracle, CPU baseline.
    `reps` timed and `warm` untimed calls of each form (reps None: --steps clamped to [3, 10]);
    `outputs`, a dict, receives what the last timed forward+backward at batches[-1] computed."""
    import torchkge_b200 as tk
    from torchkge_b200 import synthetic as S
    from torchkge_b200.training import fused_margin_step
    c5 = S.C5
    dim, n_ent, n_rel, n_neg = c5["dim"], c5["n_ent"], c5["n_rel"], c5["n_neg"]
    torch.manual_seed(0)
    model = tk.DistMultModel(dim, 64, n_rel)       # small constructor, then the synthetic tables
    from torchkge_b200 import _lib
    tabs = S.make_tables(_lib.DISTMULT, dim, n_ent, n_rel, 0, n_ent, args.seed, dev)
    model.n_ent = n_ent
    model.ent_emb = torch.nn.Embedding.from_pretrained(tabs["ent0"], freeze=False)
    model.rel_emb = torch.nn.Embedding.from_pretrained(tabs["rel0"], freeze=False)
    model = model.to(dev)
    params = list(model.parameters())
    peak, peak_src = measured_peaks()
    g = torch.Generator(device=dev).manual_seed(1)
    probs = torch.rand(n_rel, generator=g, device=dev) * 0.8 + 0.1
    row = 4 * dim
    out = {"workload": c5_workload_text(batches[-1]), "metric": C5_METRIC, "by_batch": {}}
    calls = [0]
    last = {}

    def timed(fn, reps, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    for b in batches:
        h = torch.randint(0, n_ent, (b,), generator=g, device=dev)
        t = torch.randint(0, n_ent, (b,), generator=g, device=dev)
        r = torch.randint(0, n_rel, (b,), generator=g, device=dev)
        h_host, t_host, r_host = (x.cpu().pin_memory() for x in (h, t, r))

        def fwd():
            calls[0] += 1
            with torch.no_grad():
                return fused_margin_step(model, h, t, r, 1.0, n_neg=n_neg, bern_probs=probs, seed=7, offset=calls[0])

        def fwd_bwd():
            calls[0] += 1
            for p in params:
                p.grad = None
            loss = fused_margin_step(model, h, t, r, 1.0, n_neg=n_neg, bern_probs=probs, seed=7, offset=calls[0])
            loss.backward()
            last["loss"] = loss
            return loss

        def e2e_step():
            # host batch in (pinned), loss value out
            calls[0] += 1
            for p in params:
                p.grad = None
            hd, td, rd = (x.to(dev, non_blocking=True) for x in (h_host, t_host, r_host))
            loss = fused_margin_step(model, hd, td, rd, 1.0, n_neg=n_neg, bern_probs=probs, seed=7, offset=calls[0])
            loss.backward()
            return loss.item()

        if reps is None:
            reps = max(3, min(args.steps, 10))
        ms_f, ms_fb = timed(fwd, reps, warm), timed(fwd_bwd, reps, warm)
        if outputs is not None and b == batches[-1]:
            rows = dump_rows(n_ent)
            outputs.update(loss=last["loss"].detach().view(1), grad_ent_rows=rows,
                           grad_ent=model.ent_emb.weight.grad[rows.to(dev)],
                           grad_rel=model.rel_emb.weight.grad.clone())
        t0 = time.perf_counter()
        for _ in range(reps):
            e2e_step()
        e2e_ms = (time.perf_counter() - t0) / reps * 1e3
        bytes_f = b * (n_neg + 3) * row
        bytes_fb = 3 * bytes_f
        out["by_batch"][str(b)] = {
            "fwd_ms": ms_f, "fwd_bwd_ms": ms_fb,
            "positives_per_s_fwd": b / ms_f * 1e3, "positives_per_s_fwd_bwd": b / ms_fb * 1e3,
            "negatives_per_s_fwd_bwd": b * n_neg / ms_fb * 1e3,
            "e2e": {"value": b / e2e_ms * 1e3, "unit": "positives/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": 3 * 8 * b, "d2h_bytes_per_step": 4,
                    "api": "fused_margin_step(model, h, t, r, margin, n_neg, bern_probs).backward(); "
                           "pinned host int64 batch in, loss.item() out; dense weight.grad tables zero-filled "
                           "by autograd every step (800 MB) are inside this number"},
            "roofline_fwd": {"bound": "hbm", "achieved": bytes_f / ms_f / 1e6, "peak": peak, "unit": "GB/s",
                             "frac": bytes_f / ms_f / 1e6 / peak, "alg_bytes": bytes_f},
            "roofline_fwd_bwd": {"bound": "hbm", "achieved": bytes_fb / ms_fb / 1e6, "peak": peak, "unit": "GB/s",
                                 "frac": bytes_fb / ms_fb / 1e6 / peak, "alg_bytes": bytes_fb,
                                 "note": "includes autograd's zero-fill of the dense gradient tables (%d MB) "
                                         "that the algorithmic bytes do not count" % (sum(p.numel() for p in params) * 4 // 1000000)},
            "peak_source": peak_src}
    # ---- parity with supplied negatives (oracle: forward_pos_neg + margin_loss), B = 1024 ----
    from oracle import kge_oracle as oracle
    bp = 1024
    gc = torch.Generator().manual_seed(5)
    hp = torch.randint(0, n_ent, (bp,), generator=gc)
    tp = torch.randint(0, n_ent, (bp,), generator=gc)
    rp = torch.randint(0, n_rel, (bp,), generator=gc)
    nhp, ntp = oracle.corrupt_batch(hp, tp, rp, probs.cpu(), n_ent, 16)
    rows = torch.unique(torch.cat([hp, tp, nhp, ntp]))
    remap = torch.zeros(n_ent, dtype=torch.int64)
    remap[rows] = torch.arange(rows.numel())
    P = {"ent": tabs["ent0"][rows.to(dev)].cpu().clone().requires_grad_(True),
         "rel": tabs["rel0"].cpu().clone().requires_grad_(True)}
    pos, neg = oracle.forward_pos_neg("distmult", P, remap[hp], remap[tp], rp, remap[nhp], remap[ntp])
    loss_ref = oracle.margin_loss(pos, neg, 1.0)
    loss_ref.backward()
    for p in params:
        p.grad = None
    loss_gpu = fused_margin_step(model, hp.to(dev), tp.to(dev), rp.to(dev), 1.0,
                                 negatives=(nhp.to(dev), ntp.to(dev)))
    loss_gpu.backward()
    g_ent = model.ent_emb.weight.grad[rows.to(dev)].cpu()
    g_rel = model.rel_emb.weight.grad.cpu()
    rel_err = abs(loss_gpu.item() - loss_ref.item()) / max(1e-30, abs(loss_ref.item()))
    out["parity"] = {"loss_rel_err": rel_err, "loss_ok_1e-5": rel_err <= 1e-5,
                     "grad_ent_allclose_rtol1e-4": bool(torch.allclose(g_ent, P["ent"].grad, rtol=1e-4, atol=1e-6)),
                     "grad_rel_allclose_rtol1e-4": bool(torch.allclose(g_rel, P["rel"].grad, rtol=1e-4, atol=1e-6)),
                     "sample": "B=%d, 16 supplied negatives each, oracle forward_pos_neg + margin_loss + autograd" % bp}
    for p in params:
        p.grad = None
    if cpu_steps:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        b = 4096
        Pc = {"ent": tabs["ent0"].cpu().requires_grad_(True), "rel": tabs["rel0"].cpu().requires_grad_(True)}
        hc = torch.randint(0, n_ent, (b,), generator=gc)
        tc_ = torch.randint(0, n_ent, (b,), generator=gc)
        rc = torch.randint(0, n_rel, (b,), generator=gc)
        t0 = time.perf_counter()
        for _ in range(cpu_steps):
            nh, nt = oracle.corrupt_batch(hc, tc_, rc, probs.cpu(), n_ent, n_neg)
            pos, neg = oracle.forward_pos_neg("distmult", Pc, hc, tc_, rc, nh, nt)
            loss = oracle.margin_loss(pos, neg, 1.0)
            loss.backward()
        cpu_s = (time.perf_counter() - t0) / cpu_steps
        out["cpu_baseline"] = {"value": b / cpu_s, "unit": "positives/s", "cores": cores, "kind": "port",
                               "sample": "%d step(s) at B=%d, fwd+bwd (oracle corrupt_batch + forward_pos_neg + "
                                         "margin_loss + autograd), torch %s CPU" % (cpu_steps, b, torch.__version__)}
    return out


def run_c5(args, rank, world, dev):
    """--workload c5: replicas only (SURVEY.md section 8e): every rank runs the same step; the
    line reports rank 0's numbers times the number of replicas."""
    import torch.distributed as dist
    clocks = ClockSampler(dev.index) if rank == 0 else None
    if clocks is not None:
        clocks.start()
    outputs = {} if args.dump_outputs and rank == 0 else None
    rec = measure_c5(args, dev, cpu_steps=0 if (args.no_cpu_baseline or rank != 0) else 3, batches=(4096, args.batch),
                     reps=args.steps, warm=args.warmup, outputs=outputs)
    clock_rec = clocks.stop() if clocks is not None else None
    if world > 1:
        dist.barrier()
    if rank == 0:
        b = rec["by_batch"][str(args.batch)]
        emit({"metric": C5_METRIC, "value": world * b["positives_per_s_fwd_bwd"], "unit": "positives/s",
              "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": b["fwd_bwd_ms"],
              "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
              "config": {"workload": c5_workload_text(args.batch),
                         "parallelism": "single GPU" if world == 1 else "%d independent replicas (no collective)" % world,
                         "l2_policy": "inputs larger than L2 (random rows of an 800 MB table)"},
              "e2e": {k: (v * world if k == "value" else v) for k, v in b["e2e"].items()},
              "gpu_launches": 2 * args.steps, "clocks": clock_rec,
              "roofline": dict(b["roofline_fwd_bwd"], kernel="margin_step_fast_kernel fwd + bwd", traffic=None,
                               forward_only=b["roofline_fwd"]),
              "parity": rec["parity"], "cpu_baseline": rec.get("cpu_baseline"), "by_batch": rec["by_batch"]})
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank, local, world = dist_info()
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("--gpus %d needs torchrun with %d ranks (WORLD_SIZE=%d)" % (
            args.gpus, args.gpus, world))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local, world)


if __name__ == "__main__":
    main()
