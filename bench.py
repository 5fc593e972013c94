#!/usr/bin/env python
"""bench.py — scored triples/sec (train + 1-vs-all eval), FB15k-237 shape, TransE d=200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the UNMODIFIED reference on the host cores

Workload (BASELINE.json configs[1]): TransE, N=14,541 entities, R=237 relations, d=200,
L2 norm (-l1 False), hinge margin 5.0 (pykg2vec/hyperparams/TransE.yaml:10), SGD lr 0.01, batch 512,
neg_rate 1, synthetic FB15k-237-shaped graph (no dataset is obtainable offline), tables
xavier-uniform random-init.

One STEP = what the reference repeats on this path for one batch of each kind:
  * one training batch (Trainer.train_model_epoch body, pykg2vec/utils/trainer.py:269-300):
    512 positive + 512 negative triples scored, hinge loss, backward, SGD update
    -> 1,024 scored triples;
  * one evaluation batch (Evaluator.test, pykg2vec/utils/evaluator.py:309-334) of Q=512 test
    triples, each ranked 1-vs-all against every entity in both directions, raw + filtered
    -> 2*512*14,541 = 14,889,984 scored triples.
`value` = scored triples / second of the whole job with inputs resident in HBM;
`e2e` = the same through the host API (Trainer.train_batch + Evaluator.rank_triples:
host id buffers in, pinned H2D, kernels, D2H of loss and ranks) — copies inside the timing.
`train_triples_per_s` / `eval_scores_per_s` time the two halves separately (the eval half is
99.99 % of the scored triples, so `value` alone says nothing about training).

Multi-GPU (torchrun, one rank per GPU): weak scaling — every rank brings its own training batch and
its own 512 test triples.  Training is data-parallel with replicated tables (pykg2vec_b200/trainer.py:
"grads" = local forward/backward + one gradient all-reduce per table, "ids" = id all-gather for tiny
batches); evaluation shards the test triples with NO collective in the timed step — ranks are gathered
once, after the timing (as a real evaluation gathers once at its end).
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

WORKLOAD = dict(model="transe", dataset="fb15k_237", N=14541, R=237, d=200, l1=False, margin=5.0,
                lr=0.01, B=512, neg=1, Q=512)
# identical in both arms (the driver compares them)
CONFIG = {"workload": "TransE L2 d=200 on FB15k-237 shape (N=14541, R=237): per step one train batch "
                      "B=512 neg=1 hinge(margin 5)+SGD and one 1-vs-all eval batch of Q=512 test triples "
                      "(head+tail, raw+filtered)",
          "scored_triples_per_step_per_gpu": WORKLOAD["B"] * (1 + WORKLOAD["neg"]) + 2 * WORKLOAD["Q"] * WORKLOAD["N"],
          "l2": "flushed before every timed step (256 MiB memset, untimed); tables (11.6 MB) otherwise stay L2-resident"}
L2_FLUSH_BYTES = 256 << 20
METRIC = "scored triples/sec (train + 1-vs-all eval)"
DATA = "synthetic (FB15k-237-shaped random graph, random-init tables)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm": float(d["hbm_gbs"]), "bf16": float(d["bf16_tflops"]), "bf16_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "src": "measured (MEASURED_PEAKS.json)", "sm_max": float(d.get("sm_max_mhz", 1965.0))}
    return {"hbm": 6650.0, "bf16": 1590.0, "bf16_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)", "sm_max": 1965.0}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_graph():
    from pykg2vec_b200.synthetic import SyntheticKnowledgeGraph
    return SyntheticKnowledgeGraph.shaped_like(WORKLOAD["dataset"], seed=0)


def make_batches(kg, nsteps, rank, seed=1):
    """Per step: (pairwise batch of 6 id arrays, Q test triples).  Negatives: head or tail
    corrupted with p=0.5, uniform (pykg2vec/data/generator.py:73-95, 'uniform' sampling)."""
    w = WORKLOAD
    rng = np.random.RandomState(seed + 7919 * rank)
    train, test = kg.arrays["train"], kg.arrays["test"]
    out = []
    for s in range(nsteps):
        sel = rng.randint(len(train), size=w["B"])
        ph, pr, pt = train[sel, 0].copy(), train[sel, 1].copy(), train[sel, 2].copy()
        corrupt_tail = rng.random_sample(w["B"]) > 0.5
        rnd = rng.randint(w["N"], size=w["B"])
        nh = np.where(corrupt_tail, ph, rnd)
        nt = np.where(corrupt_tail, rnd, pt)
        qsel = (np.arange(w["Q"]) + (s * w["Q"] + rank * 4099)) % len(test)
        out.append(([ph, pr, pt, nh, pr.copy(), nt], test[qsel]))
    return out


def build(kg, device):
    import torch
    import pykg2vec_b200
    from pykg2vec_b200.synthetic import SyntheticConfig
    from pykg2vec_b200.trainer import Trainer
    w = WORKLOAD
    cfg = SyntheticConfig(kg, device=device, optimizer="sgd", learning_rate=w["lr"], margin=w["margin"],
                          hidden_size=w["d"], l1_flag=w["l1"], batch_size=w["B"], neg_rate=w["neg"])
    torch.manual_seed(2)
    model = pykg2vec_b200.import_model(w["model"])(**cfg.__dict__)
    tr = Trainer(model, cfg)
    tr.build_model()
    return tr


def event_ms(torch, fn, reps, flush=None):
    """mean CUDA-event time of fn() on the current stream; optional untimed L2 flush before each rep"""
    tot = 0.0
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        tot += a.elapsed_time(b)
    return tot / reps


# DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of ONE `ncu --set full` capture of each
# kernel at exactly the shapes timed here — the summaries are committed under profiles/ (ncu cannot run inside
# this process, and a number printed under ncu is never a bench value).
NCU_TRAFFIC = {
    "tc_sweep_both": (13.101824e6 + 0.0, "profiles/r2_ncu_tc_sweep_final_summary.txt (cold caches: the 12 MB of bf16 "
                                         "candidate operands read once from DRAM; in the step they are L2 hits)"),
    "transe": (6.846856e9 + 19.496704e6, "profiles/r2_ncu_score_fwd_transe_staged_summary.txt"),
    "complex": (6.801099e9 + 11.725824e6, "profiles/r2_ncu_score_fwd_complex_summary.txt"),
}


def gather_score_rooflines(torch, _lib, dev, pk, reps=10):
    """The fused gather+score kernels north_star's >= 60 %-of-HBM target names (TransE, ComplEx; d = 200),
    timed here on tables far larger than the 126 MB L2 with random ids.  Algorithmic bytes count what
    must come from DRAM: the ENTITY rows (2 per triple for TransE, 4 for ComplEx), the 24 B of ids and the
    4 B score — the R=1000 relation rows are L2 hits and are not counted."""
    out = []
    gen = torch.Generator(device=dev).manual_seed(0)
    for name, N, ntab_e, ntab_r, n in (("transe", 2_000_000, 1, 1, 4_000_000), ("complex", 1_000_000, 2, 2, 2_000_000)):
        d, R = 200, 1000
        tabs = [(torch.rand((N, d), device=dev, generator=gen) - 0.5) * 0.2 for _ in range(ntab_e)] + \
               [(torch.rand((R, d), device=dev, generator=gen) - 0.5) * 0.2 for _ in range(ntab_r)]
        desc = _lib.ModelDesc(name, tabs, d, l1_flag=False)
        h = torch.randint(0, N, (n,), device=dev, generator=gen)
        r = torch.randint(0, R, (n,), device=dev, generator=gen)
        t = torch.randint(0, N, (n,), device=dev, generator=gen)
        o = torch.empty(n, dtype=torch.float32, device=dev)
        for _ in range(3):
            _lib.score_fwd(desc, h, r, t, out=o)
        ms = event_ms(torch, lambda: _lib.score_fwd(desc, h, r, t, out=o), reps)
        alg = n * (2 * ntab_e * d * 4 + 24 + 4)
        out.append({"kernel": "score_fwd_kernel<%s> (fused gather+score, %d random triples, %d x %d entity table%s = %.1f GB)"
                              % (name, n, N, d, "s" if ntab_e > 1 else "", ntab_e * N * d * 4 / 1e9),
                    "bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                    "frac": alg / (ms * 1e-3) / 1e9 / pk["hbm"], "peak_source": pk["src"], "launch_ms": ms,
                    "algorithmic_bytes_per_launch": alg,
                    "algorithmic_bytes_per_triple": "entity rows %d x %d B + 24 B ids + 4 B score (relation rows are L2-resident)"
                                                    % (2 * ntab_e, d * 4),
                    "traffic": NCU_TRAFFIC[name][0], "traffic_source": NCU_TRAFFIC[name][1]})
        del tabs, desc, h, r, t, o
        torch.cuda.empty_cache()
    return out


def run_cuda(args):
    import torch
    import torch.distributed as dist
    from pykg2vec_b200 import _lib, sharding
    from pykg2vec_b200.evaluator import build_filter_csr
    rank, world = sharding.init_distributed()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    w = WORKLOAD
    kg = make_graph()
    tr = build(kg, dev)
    ev = tr.evaluator
    hr_t, tr_h = kg.read_cache_data("hr_t"), kg.read_cache_data("tr_h")
    total = args.warmup + args.steps
    steps = make_batches(kg, total, rank)
    host = []   # host-side inputs per step (for the e2e leg)
    devin = []  # device-resident inputs per step (for the HBM-resident leg)
    for ids, q in steps:
        ft = build_filter_csr([(int(h), int(r)) for h, r, t in q], hr_t)
        fh = build_filter_csr([(int(t), int(r)) for h, r, t in q], tr_h)
        host.append((ids, q, ft, fh))
        tod = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(dev)
        devin.append(([tod(a) for a in ids], tod(q[:, 0]), tod(q[:, 1]), tod(q[:, 2]),
                      (tod(ft[0]), tod(ft[1])), (tod(fh[0]), tod(fh[1]))))
    desc = tr.model.kge_desc()
    counts = torch.zeros((w["Q"], 4), dtype=torch.int32, device=dev)
    ws = torch.empty(max(_lib.rank_workspace_bytes(desc, w["Q"]), 16), dtype=torch.uint8, device=dev)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    train_per_step = world * w["B"] * (1 + w["neg"])
    eval_per_step = world * 2 * w["Q"] * w["N"]
    scored_per_step = train_per_step + eval_per_step

    def eval_resident(i):
        _ids, qh, qr, qt, ft, fh = devin[i]
        counts.zero_()
        _lib.rank_1vsall(desc, qh, qr, qt, ft, fh, counts=counts, workspace=ws)

    def train_resident(i):
        tr.train_batch_device(devin[i][0])   # fused step; at world > 1 data-parallel inside the Trainer

    # device tensor holding the loss of the latest resident step (every launch mode points it at its own buffer)
    last = {"loss": None}

    def resident_step(i):
        if graph_step is not None:
            return graph_step(i)
        # multi-GPU "ids" mode: the 24 KB id all-gather is started first and hides behind the evaluation batch
        ex = tr.exchange_batch_async(devin[i][0])
        eval_resident(i)
        last["loss"] = tr.train_batch_device(devin[i][0], exchanged=ex)

    # Single GPU: the resident step is ~12 short kernels, so launch gaps are a visible share of it.  It is
    # captured ONCE as a CUDA graph reading from fixed device buffers; a timed step is then the D2D copies of
    # that step's resident inputs into those buffers plus one replay (all inside the timed region).
    graph_step = None
    kernels_per_replay = None
    if not args.no_graph and (world == 1 or tr._dp == "ids"):
        # every step's resident inputs packed into ONE int64 buffer -> one D2D copy per step into the
        # static buffer the captured kernels read: [6 x B ids][qh qr qt][tail ptr][head ptr][tail idx cap][head idx cap]
        cap_t = max(x[4][1].numel() for x in devin)
        cap_h = max(x[5][1].numel() for x in devin)
        B, Q = w["B"], w["Q"]
        words = 6 * B + 3 * Q + 2 * (Q + 1) + cap_t + cap_h
        packed = []
        for ids, qh, qr, qt, ft, fh in devin:
            buf = torch.zeros(words, dtype=torch.int64, device=dev)
            o = 0
            for a in list(ids) + [qh, qr, qt, ft[0], fh[0]]:
                buf[o:o + a.numel()] = a
                o += a.numel()
            buf[o:o + ft[1].numel()] = ft[1]
            buf[o + cap_t:o + cap_t + fh[1].numel()] = fh[1]
            packed.append(buf)
        s_in = torch.zeros(words, dtype=torch.int64, device=dev)
        s_ids = [s_in[k * B:(k + 1) * B] for k in range(6)]
        o = 6 * B
        s_q = [s_in[o + k * Q:o + (k + 1) * Q] for k in range(3)]
        o += 3 * Q
        s_tp, s_hp = s_in[o:o + Q + 1], s_in[o + Q + 1:o + 2 * Q + 2]
        o += 2 * Q + 2
        s_ti, s_hi = s_in[o:o + cap_t], s_in[o + cap_t:o + cap_t + cap_h]

        def load_inputs(i):
            s_in.copy_(packed[i])

        scratch = tr._grad_scratch
        loss_buf = torch.zeros(1, dtype=torch.float32, device=dev)

        def body_eval():
            counts.zero_()
            _lib.rank_1vsall(desc, s_q[0], s_q[1], s_q[2], (s_tp, s_ti), (s_hp, s_hi), counts=counts, workspace=ws)

        def capture(fn, warm):
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                warm()   # un-captured warm-up (lr = 0: tables untouched)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            k0 = _lib.launch_count()
            # (NCCL's watchdog thread may poll its events while we capture: keep the capture's legality check
            # local to this thread when a process group is alive)
            with torch.cuda.graph(g, capture_error_mode="thread_local" if world > 1 else "global"):
                fn()
            return g, _lib.launch_count() - k0

        load_inputs(0)
        if world == 1:
            def body(lr):
                body_eval()
                _lib.train_pairwise_hinge_sgd(desc, scratch, *s_ids, w["margin"], lr, loss_buf)

            g, kernels_per_replay = capture(lambda: body(w["lr"]), lambda: body(0.0))
            last["loss"] = loss_buf
            # the two halves as graphs of their own, for the separately reported train / eval rates
            g_eval, _ = capture(body_eval, body_eval)
            g_train, _ = capture(lambda: _lib.train_pairwise_hinge_sgd(desc, scratch, *s_ids, w["margin"], w["lr"], loss_buf),
                                 lambda: _lib.train_pairwise_hinge_sgd(desc, scratch, *s_ids, w["margin"], 0.0, loss_buf))

            def graph_step(i):
                load_inputs(i)
                g.replay()

            def train_resident(i):   # noqa: F811 — graph-replayed like the step itself
                load_inputs(i)
                g_train.replay()

            def eval_resident(i):   # noqa: F811
                load_inputs(i)
                g_eval.replay()
        else:
            # data parallel, "ids" mode: the NCCL all-gather of the batch ids (24 KB) stays an eager call, started
            # first; the evaluation graph runs while it is in flight; the training graph (the Trainer's own
            # step on the gathered global batch) follows.  Three host calls per step instead of ~25.
            s_gath = torch.zeros((world * 6, B), dtype=torch.int64, device=dev)
            s_stack = s_in[:6 * B].view(6, B)

            def glob_ids():
                gl = s_gath.view(world, 6, B).permute(1, 0, 2).reshape(6, world * B).contiguous()
                return [gl[k] for k in range(6)]

            def body_train():
                # the call made during capture leaves the graph's own loss buffer here
                last["loss"] = tr.train_batch_device(s_ids, exchanged=glob_ids)

            def warm_train():
                lr0 = tr.config.learning_rate
                tr.config.learning_rate = 0.0
                try:
                    body_train()
                finally:
                    tr.config.learning_rate = lr0

            try:
                dist.all_gather_into_tensor(s_gath, s_stack)
                g_eval, k_eval = capture(body_eval, body_eval)
                g_train, k_train = capture(body_train, warm_train)
                kernels_per_replay = k_eval + k_train

                def graph_step(i):
                    load_inputs(i)
                    work = dist.all_gather_into_tensor(s_gath, s_stack, async_op=True)
                    g_eval.replay()
                    work.wait()
                    g_train.replay()

                def train_resident(i):   # noqa: F811 — exchange + graph, nothing to hide the exchange behind
                    load_inputs(i)
                    dist.all_gather_into_tensor(s_gath, s_stack)
                    g_train.replay()

                def eval_resident(i):   # noqa: F811
                    load_inputs(i)
                    g_eval.replay()
            except Exception as exc:   # capture refused next to a live process group: the eager step still measures
                print("bench: CUDA-graph capture of the data-parallel step failed (%s); timing it kernel by kernel"
                      % (str(exc).splitlines()[0] if str(exc) else type(exc).__name__), file=sys.stderr)
                graph_step = None
                torch.cuda.synchronize()

    def e2e_step(i):
        ids, q, ft, fh = host[i]
        pending_loss = tr.train_batch(ids, sync=False)   # pinned H2D + kernels (+ D2H of the loss) enqueued
        ranks = ev.rank_triples(q[:, 0], q[:, 1], q[:, 2], ft, fh)   # host staging overlaps it; returns host ranks
        return float(pending_loss), ranks                # loss of this step read on the host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, first, n, use_events):
        """n steps starting at index `first`; L2 flushed (untimed) before every step; returns total ms."""
        tot = 0.0
        for i in range(first, first + n):
            flush.zero_()
            barrier()
            if use_events:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn(i)
                b.record()
                torch.cuda.synchronize()
                tot += a.elapsed_time(b)
            else:
                t0 = time.perf_counter()
                fn(i)
                torch.cuda.synchronize()
                tot += (time.perf_counter() - t0) * 1e3
        return tot

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(args.warmup):
        resident_step(i)
        if not args.lite:
            e2e_step(i)
    barrier()

    # ---- self-check (outside every timed region): ranks of this rank's step-0 queries, through the host
    # API, against the CPU oracle on a copy of the current tables
    verified = None
    if not args.lite:
        import oracle
        nv = 16
        ids0, q0, ft0, fh0 = host[0]
        got = ev.rank_triples(q0[:, 0], q0[:, 1], q0[:, 2], ft0, fh0)
        om = oracle.Model("transe", [t_.detach().cpu().numpy() for t_ in tr.model.kge_tables()], w["d"], l1_flag=w["l1"])
        want = oracle.rank_1vsall(om, q0[:nv, 0], q0[:nv, 1], q0[:nv, 2], (ft0[0][:nv + 1], ft0[1][:ft0[0][nv]]),
                                  (fh0[0][:nv + 1], fh0[1][:fh0[0][nv]]))
        verified = bool(np.array_equal(got[:nv], want))
        if not verified:
            raise RuntimeError("bench self-check failed: rank counts differ from the oracle")

    # sustained run (~1.5 s of back-to-back steps) so that nvidia-smi samples clocks UNDER LOAD.  The number of
    # passes is fixed from one timed pass and agreed across ranks (MAX): a time-based loop would let the ranks
    # run different numbers of steps, and the steps contain collectives.  Its training updates are undone
    # afterwards, so that the timed steps start from tables that depend on the arguments only, not on the clock.
    tables0 = [t_.detach().clone() for t_ in tr.model.kge_tables()]
    torch.cuda.synchronize()
    t_p0 = time.perf_counter()
    for i in range(args.warmup, total):
        resident_step(i)
    torch.cuda.synchronize()
    one_pass = max(time.perf_counter() - t_p0, 1e-4)
    n_pass = max(1, int((0.3 if args.lite else 1.5) / one_pass))
    if world > 1:
        t = torch.tensor([n_pass], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        n_pass = int(t.item())
    t_s0 = time.perf_counter()
    for _ in range(n_pass):
        for i in range(args.warmup, total):
            resident_step(i)
        torch.cuda.synchronize()
    ms_sustained = (time.perf_counter() - t_s0) * 1e3 / (n_pass * args.steps)
    with torch.no_grad():
        for t_, t0_ in zip(tr.model.kge_tables(), tables0):
            t_.copy_(t0_)
    del tables0
    barrier()
    import gc
    gc.collect()
    gc.disable()   # no cyclic-GC pause inside a timed leg (a pause on one rank stalls every rank's collective)
    launches0 = _lib.launch_count()
    ms_res = max_over_ranks(timed(resident_step, args.warmup, args.steps, True))
    launches = _lib.launch_count() - launches0
    # what the last timed step returned (this rank's rank counts, the loss) and left behind (the trained tables)
    counts_last = counts.clone()
    dump = None
    if args.dump_outputs and rank == 0:
        names = ("ent_embeddings", "rel_embeddings")
        dump = {"loss": last["loss"].detach().reshape(1).float().cpu().numpy()}
        dump.update({n: t_.detach().float().cpu().numpy() for n, t_ in zip(names, tr.model.kge_tables())})
    if graph_step is not None:
        launches = kernels_per_replay * args.steps   # replays re-execute the captured kernels
    ms_train = max_over_ranks(timed(train_resident, args.warmup, args.steps, True))
    ms_eval = max_over_ranks(timed(eval_resident, args.warmup, args.steps, True))
    # warm-L2 back-to-back variant (tables stay in the 126 MB L2 between steps, as in a real epoch)
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(args.warmup, total):
        resident_step(i)
    b.record()
    torch.cuda.synchronize()
    ms_warm = max_over_ranks(a.elapsed_time(b))
    ms_e2e = max_over_ranks(timed(e2e_step, args.warmup, args.steps, False)) if not args.lite else float("nan")
    gc.enable()
    # multi-GPU: the ranks of all shards (those of the last timed step) are gathered ONCE, after the timing
    # (one all-gather of Q x 4 int32)
    all_counts = sharding.gather_query_shards(counts_last, world * w["Q"]) if world > 1 else counts_last
    if dump is not None:
        dump["rank_counts"] = all_counts.cpu().numpy().astype(np.float64)

    # ---- dominant kernel of the step: the tensor-core sweep, timed alone with CUDA events recorded around
    # the kernel launch itself on its own stream (C-ABI profiling hook), L2 flushed before every launch
    _ids, qh, qr, qt, ft, fh = devin[args.warmup]
    reps = max(args.steps, 10)
    sweep = {"tc": [], "fp32": []}
    # "tc": the product call (both directions: ONE tensor-core launch sweeps them, grid.z = 2);
    # "fp32": one direction of the fp32 sweep it replaces (KGE_RANK_NO_TC), for the comparison
    tc_dirs = 1
    for key, flags in (("tc", _lib.RANK_PROFILE),
                       ("fp32", _lib.RANK_TAIL_ONLY | _lib.RANK_PROFILE | _lib.RANK_NO_TC)):
        for rep in range(reps + 3):
            flush.zero_()
            torch.cuda.synchronize()
            _lib.rank_1vsall(desc, qh, qr, qt, None, None, counts=counts, workspace=ws, flags=flags)
            torch.cuda.synchronize()
            if rep >= 3:
                sweep[key].append(_lib.rank_last_sweep_ms(0))
            if key == "tc":
                tc_dirs = _lib.rank_last_sweep_directions()
    tc_ms, fp32_ms = float(np.mean(sweep["tc"])), float(np.mean(sweep["fp32"]))
    clocks = sampler.stop() if rank == 0 else None
    pk = peaks()
    extra = gather_score_rooflines(torch, _lib, dev, pk) if (rank == 0 and not args.lite) else []
    if rank != 0:
        return None
    alg_flops = tc_dirs * 2.0 * w["Q"] * w["N"] * w["d"]           # the Q x N x d contraction (2 flop per multiply-add) per direction
    kp = ((w["d"] + 3 + 15) // 16) * 16                            # padded contraction length incl. the 3 norm columns
    exec_flops = tc_dirs * 3 * 2.0 * (-(-w["Q"] // 128) * 128) * (-(-w["N"] // 128) * 128) * kp   # three bf16 passes over padded tiles
    cpu = cpu_baseline(sample_train=10, sample_queries=8) if not args.lite else None
    line = {
        "metric": METRIC, "value": scored_per_step * args.steps / (ms_res * 1e-3),
        "unit": "triples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": DATA, "config": CONFIG, "verified": verified,
        "parallelism": "dp%d (%s): tables replicated, test triples sharded, no collective in the eval step"
                       % (world, tr._dp or "single GPU"),
        "resident_step_launch": ("kernel by kernel" if graph_step is None else
                                 "one D2D copy of the step's packed inputs + one CUDA-graph replay" if world == 1 else
                                 "one D2D copy of the step's packed inputs + the NCCL all-gather of the batch ids (eager, started "
                                 "first) + two CUDA-graph replays (evaluation while the ids travel, then the training step)"),
        "train_triples_per_s": train_per_step * args.steps / (ms_train * 1e-3),
        "eval_scores_per_s": eval_per_step * args.steps / (ms_eval * 1e-3),
        "ms_per_train_step": ms_train / args.steps, "ms_per_eval_batch": ms_eval / args.steps,
        "ms_per_step_warm_l2": ms_warm / args.steps,
        "ms_per_step_sustained": ms_sustained,
        "e2e": {"value": scored_per_step * args.steps / (ms_e2e * 1e-3), "unit": "triples/s",
                "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": int(6 * w["B"] * 8 + 3 * w["Q"] * 8 +
                                          sum(x.nbytes for x in host[args.warmup][2]) + sum(x.nbytes for x in host[args.warmup][3])),
                "d2h_bytes_per_step": 4 + w["Q"] * 4 * 4},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"kernel": "tc_sweep_kernel: 1-vs-all tensor-core sweep (%s, Q=512 x N=14541 x d=200 each, "
                               "tcgen05.mma bf16x3 split, fp32 accumulation in TMEM)"
                               % ("tail + head directions in one launch" if tc_dirs == 2 else "tail direction"),
                     "directions_per_launch": tc_dirs,
                     "bound": "tensor", "achieved": alg_flops / (tc_ms * 1e-3) / 1e12, "peak": pk["bf16"], "unit": "TFLOP/s",
                     "frac": alg_flops / (tc_ms * 1e-3) / 1e12 / pk["bf16"], "peak_source": pk["src"] + ", burst bf16 (kernel timed alone)",
                     "launch_ms": tc_ms, "algorithmic_flops_per_launch": alg_flops,
                     "algorithmic_flops_per_unit": "2*d = 400 flop per scored candidate (one length-d contraction)",
                     "executed_tensor_flops_per_launch": exec_flops,
                     "executed_frac": exec_flops / (tc_ms * 1e-3) / 1e12 / pk["bf16"],
                     "traffic": NCU_TRAFFIC["tc_sweep_both"][0] if tc_dirs == 2 else None,
                     "traffic_source": NCU_TRAFFIC["tc_sweep_both"][1] if tc_dirs == 2 else None,
                     "note": "exact fp32 ranks need three bf16 passes (a0b0 + a0b1 + a1b0) over tiles padded to 128 x 128 x 208: "
                             "executed_frac counts those tensor flops, frac only the algorithm's 2*Q*N*d",
                     "fp32_sweep_ms_per_direction": fp32_ms, "speedup_vs_fp32_sweep": fp32_ms * tc_dirs / tc_ms},
        "rooflines_extra": extra,
        "cpu_baseline": cpu,
    }
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    return line


# ------------------------------------------------------------------ CPU reference arm ----
def usable_cores():
    """cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


class RefArm:
    """The UNMODIFIED reference (oracle/_ref, installed by build(): oracle/ref_install.py) on the host cores, driven
    through its own code: pykg2vec.models.pairwise.TransE, Trainer.train_step_pairwise + backward +
    optimizer.step (pykg2vec/utils/trainer.py:147-157,288-300) and Evaluator.test
    (pykg2vec/utils/evaluator.py:309-334: two forwards over all N entities, topk(N), D2H, the Python rank walk
    of MetricCalculator).  None of this repo's models, kernels or engine is on this path."""
    kind = "reference"

    def __init__(self):
        import types
        import torch
        from baseline import ref_loader
        ref_loader.load()
        from pykg2vec.models.pairwise import TransE
        from pykg2vec.utils.evaluator import Evaluator
        from pykg2vec.utils.trainer import Trainer
        from pykg2vec_b200.synthetic import SyntheticConfig
        w = WORKLOAD
        self.torch = torch
        self.cores = usable_cores()
        torch.set_num_threads(self.cores)
        self.kg = make_graph()
        cfg = SyntheticConfig(self.kg, device="cpu", optimizer="sgd", learning_rate=w["lr"], margin=w["margin"],
                              hidden_size=w["d"], l1_flag=w["l1"], batch_size=w["B"], neg_rate=w["neg"])
        cfg.epochs, cfg.debug = 1 << 30, False
        torch.manual_seed(2)
        self.model = TransE(**cfg.__dict__)
        self.trainer = object.__new__(Trainer)                    # its train_step_* methods only read model / config
        self.trainer.model, self.trainer.config = self.model, cfg
        self.optimizer = torch.optim.SGD(self.model.parameters(), lr=w["lr"])   # trainer.py:117-121
        self.evaluator = Evaluator(self.model, cfg)
        self.batches = make_batches(self.kg, 64, 0)
        self.test = self.kg.read_cache_data("triplets_test")
        self.cursor = 0
        self.desc = "torch %s CPU, pykg2vec 0.0.52 from oracle/_ref" % torch.__version__

    def train_steps(self, n):
        torch = self.torch
        self.model.train()
        t0 = time.perf_counter()
        for _ in range(n):
            ids, _q = self.batches[self.cursor % len(self.batches)]
            self.cursor += 1
            self.optimizer.zero_grad()
            tid = [torch.LongTensor(np.asarray(a)) for a in ids]          # trainer.py:288-293
            loss = self.trainer.train_step_pairwise(*tid)
            loss.backward()
            self.optimizer.step()
            loss.item()                                                  # trainer.py:300
        return (time.perf_counter() - t0) / n

    def eval_queries(self, n):
        start = (self.cursor * 7) % (len(self.test) - n)
        self.model.eval()
        import contextlib, io
        with self.torch.no_grad(), contextlib.redirect_stderr(io.StringIO()):   # tqdm's progress bar
            t0 = time.perf_counter()
            self.evaluator.test(self.test[start:start + n], n, epoch=0)
            return (time.perf_counter() - t0) / n


class PortArm:
    """Fallback when oracle/_ref is absent: the torch port of the same op chain (oracle/ref_port.py)."""
    kind = "port"

    def __init__(self):
        import torch
        from oracle import ref_port
        w = WORKLOAD
        self.torch, self.rp = torch, ref_port
        self.cores = usable_cores()
        torch.set_num_threads(self.cores)
        self.kg = make_graph()
        gen = torch.Generator().manual_seed(2)
        self.ent = ref_port.xavier_uniform(w["N"], w["d"], gen).requires_grad_()
        self.rel = ref_port.xavier_uniform(w["R"], w["d"], gen).requires_grad_()
        self.opt = torch.optim.SGD([self.ent, self.rel], lr=w["lr"])
        self.batches = make_batches(self.kg, 64, 0)
        self.hr_t, self.tr_h = self.kg.read_cache_data("hr_t"), self.kg.read_cache_data("tr_h")
        self.cursor = 0
        self.desc = "torch %s CPU port of the reference op chain (oracle/ref_port.py)" % torch.__version__

    def train_steps(self, n):
        torch, rp, w = self.torch, self.rp, WORKLOAD
        t0 = time.perf_counter()
        for _ in range(n):
            ids, _q = self.batches[self.cursor % len(self.batches)]
            self.cursor += 1
            tid = [torch.LongTensor(np.asarray(a)) for a in ids]
            self.opt.zero_grad()
            pos = rp.score("transe", [self.ent, self.rel], tid[0], tid[1], tid[2], l1_flag=w["l1"])
            neg = rp.score("transe", [self.ent, self.rel], tid[3], tid[4], tid[5], l1_flag=w["l1"])
            loss = rp.pairwise_hinge(pos, neg, w["margin"])
            loss.backward()
            self.opt.step()
            loss.item()
        return (time.perf_counter() - t0) / n

    def eval_queries(self, n):
        torch, rp, w = self.torch, self.rp, WORKLOAD
        test = self.kg.arrays["test"]
        q = [tuple(int(x) for x in test[(self.cursor * 7 + k) % len(test)]) for k in range(n)]
        fn = lambda a, b, c: rp.score("transe", [self.ent, self.rel], a, b, c, l1_flag=w["l1"])
        with torch.no_grad():
            t0 = time.perf_counter()
            rp.evaluate(fn, w["N"], q, self.hr_t, self.tr_h)
            return (time.perf_counter() - t0) / n


def make_arm():
    from baseline import ref_loader
    if ref_loader.available():
        try:
            return RefArm()
        except Exception as e:   # noqa: BLE001 — fall back to the port, say why
            sys.stderr.write("reference arm: oracle/_ref unusable (%r), using the port\n" % (e,))
    return PortArm()


def tune_threads(arm):
    """Give the CPU arm its best shot: intra-op thread counts up to the usable cores are
    probed on one train step + one test triple and the fastest is kept (torch CPU kernels
    on small tensors often run faster on fewer threads than cores)."""
    w = WORKLOAD
    cands = sorted({c for c in (arm.cores, 64, 32, 16, 8, 4) if c <= arm.cores}, reverse=True)
    best, best_t = cands[0], float("inf")
    for c in cands:
        arm.torch.set_num_threads(c)
        arm.train_steps(1)
        t0 = time.perf_counter()
        t = arm.train_steps(1) + w["Q"] * arm.eval_queries(1)
        if t < best_t:
            best, best_t = c, t
        if time.perf_counter() - t0 > 20:
            break
    arm.torch.set_num_threads(best)
    arm.cores = best
    return best


def cpu_line_value(t_train, t_query):
    w = WORKLOAD
    step_s = t_train + w["Q"] * t_query
    return (w["B"] * (1 + w["neg"]) + 2 * w["Q"] * w["N"]) / step_s, step_s


def cpu_baseline(sample_train, sample_queries):
    arm = make_arm()
    tune_threads(arm)
    arm.train_steps(2)
    arm.eval_queries(1)
    t_train, t_query = arm.train_steps(sample_train), arm.eval_queries(sample_queries)
    value, _ = cpu_line_value(t_train, t_query)
    return {"value": value, "unit": "triples/s", "cores": arm.cores, "kind": arm.kind,
            "sample": "%d train steps + %d test triples of the same workload timed, extrapolated to one step "
                      "(1 train batch + 512 test triples: every test triple costs the same two forwards over N + "
                      "topk + rank walk); %s" % (sample_train, sample_queries, arm.desc),
            "train_step_ms": t_train * 1e3, "eval_ms_per_test_triple": t_query * 1e3}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    # each step: a bounded sample of the workload — 1 train batch + 32 test triples really evaluated —
    # extrapolated to the step's 512 test triples (said so in cpu_baseline.sample)
    per_step_queries = 32
    tt, tq = [], []
    arm = make_arm()
    cores = tune_threads(arm)
    for s in range(args.warmup + args.steps):
        a, b = arm.train_steps(1), arm.eval_queries(per_step_queries)
        if s >= args.warmup:
            tt.append(a)
            tq.append(b)
    t_train, t_query = float(np.mean(tt)), float(np.mean(tq))
    value, step_s = cpu_line_value(t_train, t_query)
    line = {
        "impl": "reference", "metric": METRIC, "value": value,
        "unit": "triples/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": DATA, "config": CONFIG,
        "cpu_baseline": {"value": value, "unit": "triples/s", "cores": cores, "kind": arm.kind,
                         "sample": "per step 1 train batch + %d test triples really run (Evaluator.test), extrapolated to "
                                   "the step's 512 test triples; %s" % (per_step_queries, arm.desc),
                         "train_step_ms": t_train * 1e3, "eval_ms_per_test_triple": t_query * 1e3},
        "e2e": {"value": value, "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 4, 5],
                    help="2 (default): the BASELINE.json headline step; 4 / 5: the multi-GPU evaluation measurements of "
                         "configs[3] (RotatE FB15k, query-sharded) / configs[4] (ComplEx YAGO3-10, entity rows partitioned "
                         "across the ranks) — bench_sharded.py, one JSON line each, not the driver's contract line")
    ap.add_argument("--no-graph", action="store_true",
                    help="launch the resident step kernel by kernel instead of replaying it as one CUDA graph (N = 1)")
    ap.add_argument("--lite", action="store_true",
                    help="profiling aid: only the HBM-resident leg (no e2e / CPU baseline / self-check); never a bench value")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy: rank_counts "
                         "((GPUs x Q) x 4, the query shards of all ranks in rank order: tail raw, tail filtered, head raw, "
                         "head filtered; float64), rank 0's loss (float32) and the "
                         "trained ent_embeddings / rel_embeddings (float32); the same arguments give the same inputs")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "cuda" or args.config != 2):
        ap.error("--dump-outputs writes the outputs of the CUDA path's headline step (--impl cuda --config 2)")
    if args.config != 2:
        import bench_sharded
        return bench_sharded.main(["--queries", "512" if args.config == 5 else "4096"], only=args.config)
    args.warmup = max(args.warmup, 3) if args.impl == "cuda" else args.warmup
    # stdout carries exactly ONE JSON line: while the run is in progress fd 1 points at stderr so
    # that banners printed by native libraries (e.g. NCCL's INFO lines) cannot end up there
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    line = None
    try:
        line = run_reference(args) if args.impl == "reference" else run_cuda(args)
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    if line is not None:
        print(json.dumps(line), flush=True)
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
