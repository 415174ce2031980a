#!/usr/bin/env python
"""bench.py -- DeepFM training samples/sec on Criteo-39-field synthetic data (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (B200, libctr_b200.so)
  python bench.py --impl reference --gpus N --steps K ...  the reference's CPU path (oracle port:
                                                            TensorFlow is not installable here)

Workload (BASELINE.json configs[1]): DeepFM, 39 fields, 200M-row vocabulary, k=16, batch 8192,
deep_layers 256,128,64, dropout 0.5, Adam(5e-4), l2_reg 1e-4 -- the reference script's defaults.
A "step" is one optimizer.minimize(loss) on one batch with TensorFlow's exact semantics: because
l2_loss(fm_v) densifies the gradient and tf.train.AdamOptimizer is not lazy, EVERY table row moves
every step (SURVEY.md A.4).  The headline runs the exact-deferred update (csrc/epoch.cu): the state
is bit-identical to sweeping the whole table every step, but rows nothing gathered are replayed
lazily, one pass over HBM per 16 steps.  `exact_every_step` reports the plain HBM-bound formulation.
`value`   : inputs resident in HBM, CUDA-event timed, max over ranks.
`e2e`     : same steps fed from pinned HOST buffers through the public API, loss read back per step.
`lazy`    : the same step when only gathered rows are updated (NOT the reference's result; reported
            for context, never as the headline).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# the tree this runs from may be read-only and stays as build() left it: no __pycache__ written from here
sys.dont_write_bytecode = True

CFG = dict(model="DeepFM", field_size=39, feature_size=200_000_000, embedding_size=16, batch_size=8192,
           deep_layers="256,128,64", dropout="0.5,0.5,0.5", l2_reg=1e-4, learning_rate=5e-4, optimizer="Adam")
METRIC = "DeepFM training samples/sec, Criteo-39-field synthetic (39 fields, 200M vocab, k=16, bs=8192)"
N_BATCHES = 16  # distinct pre-staged batches, cycled


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--vocab", type=int, default=CFG["feature_size"], help="override N (debug only)")
    ap.add_argument("--batch", type=int, default=CFG["batch_size"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the lazy/infer side measurements")
    ap.add_argument("--zipf", type=float, default=0.0,
                    help="0 = uniform ids inside each categorical sub-vocabulary (default: the roofline-honest worst "
                         "case); > 0 = heavy-tailed ids (synth.criteo_batch), the secondary distribution of SURVEY 8d")
    ap.add_argument("--tables", default="auto", choices=["auto", "replicated", "sharded"],
                    help="N>1: 'sharded' = rows owned by id %% N, NCCL all-to-all exchange (default); "
                         "'replicated' = data parallel with all-gathered sparse gradients")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the headline timed steps, write what the last of them computed (loss terms, "
                         "probabilities, dense variables, a seeded row sample of fm_v / fm_w) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs needs the b200 arm on one GPU")
    return a


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML during the timed region."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ----------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# ----------------------------------------------------------------------------------------------------
def cpu_vocab(N: int) -> int:
    """Largest vocabulary <= N whose oracle state + temporaries (~10 table-sized fp32 arrays) fit in
    half of the available host RAM."""
    import psutil
    avail = psutil.virtual_memory().available
    n = N
    while n > 1000 and n * (CFG["embedding_size"] + 1) * 4 * 10 > avail * 0.5:
        n //= 2
    return n


def _synth_module():
    """tf_repos_b200/synth.py (pure numpy/torch batch generator) loaded BY PATH: importing the package would dlopen
    libctr_b200.so, and the reference arm must not map any product code."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ctr_synth_standalone", os.path.join(ROOT, "tf_repos_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _interleave_host_memory():
    """set_mempolicy(MPOL_INTERLEAVE, all nodes): the oracle's table-sized arrays are first-touched by one thread and
    would otherwise sit on one NUMA node (the CPU arm moved 4x between boxes in round 1).  Best effort."""
    try:
        import ctypes
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        if len(nodes) < 2:
            return f"{len(nodes)} NUMA node(s)"
        mask = ctypes.c_ulong(sum(1 << int(d[4:]) for d in nodes))
        libc = ctypes.CDLL(None, use_errno=True)
        rc = libc.syscall(238, 3, ctypes.byref(mask), ctypes.c_ulong(8 * ctypes.sizeof(mask)))   # x86_64 set_mempolicy
        return f"{len(nodes)} NUMA nodes, interleave rc={rc}"
    except Exception as e:  # pragma: no cover
        return f"interleave unavailable ({e})"


def run_cpu(steps: int, warmup: int, budget_s: float, N: int, B: int):
    """Times oracle.DeepFM.train_step (TF-exact semantics, all host threads).  Returns
    (samples_per_s, ms_per_step, steps_timed, cores, sample description)."""
    import torch

    from oracle import models as om
    from oracle import tf_semantics as tfs
    synth = _synth_module()

    numa = _interleave_host_memory()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    tfs.FAST_SQRT = True  # multithreaded (non-IEEE) sqrt: fastest honest CPU number
    n_cpu = cpu_vocab(N)
    c = CFG
    m = om.DeepFM(c["field_size"], 1000, c["embedding_size"], deep_layers=c["deep_layers"], dropout=c["dropout"],
                  l2_reg=c["l2_reg"], learning_rate=c["learning_rate"], optimizer=c["optimizer"], seed=0)
    # big tables: cheap normal init (the truncated-normal loop would dominate start-up)
    std = (2.0 / (n_cpu + c["embedding_size"])) ** 0.5
    m.N = n_cpu
    m.params["fm_v"] = torch.randn(n_cpu, c["embedding_size"]) * std
    m.params["fm_w"] = torch.randn(n_cpu) * (1.0 / n_cpu) ** 0.5
    m.init_slots()
    batches = [synth.criteo_batch(B, n_cpu, c["field_size"], seed=1000 + i) for i in range(4)]
    gen = torch.Generator().manual_seed(0)
    widths = [int(w) for w in c["deep_layers"].split(",")]
    keeps = [float(k) for k in c["dropout"].split(",")]

    def one(i):
        ids, vals, labels = batches[i % len(batches)]
        masks = [(torch.rand(B, w, generator=gen) < k).float() for w, k in zip(widths, keeps)]
        return m.train_step({"feat_ids": ids.long(), "feat_vals": vals}, labels, masks)

    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    done = 0
    for i in range(steps):
        one(i)
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    desc = (f"{done} exact-TF train steps of oracle.DeepFM (PyTorch-CPU fp32 restatement of DeepFM.py model_fn), "
            f"B={B}, F=39, k=16, vocab {n_cpu}, {warmup} warm-up steps, {numa}" + ("" if n_cpu == N else f" (cut from {N} to fit host RAM; the "
            f"dense-sweep cost scales with vocab, so this FLATTERS the CPU)"))
    return B * done / dt, dt / done * 1e3, done, cores, desc


def _tf_importable() -> bool:
    """SURVEY 8c: probe at run time; a TensorFlow that could run the reference has never been seen in this image."""
    import importlib.util
    try:
        return importlib.util.find_spec("tensorflow") is not None
    except Exception:
        return False


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # three warm-up steps (first touches of the table-sized scratch arrays) and a wall-clock budget: a
    # full-vocabulary CPU step takes seconds
    wu = max(min(args.warmup, 3), 1)
    sps, ms, done, cores, desc = run_cpu(args.steps, wu, 100.0, args.vocab, args.batch)
    line = {"impl": "reference", "metric": METRIC, "value": sps, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": done, "warmup": wu, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]: DeepFM 39 fields, 200M vocab, k=16, bs=8192 (exact TF semantics)",
                       "note": "TensorFlow 1.4 / Python 2 reference cannot be installed here; oracle port timed",
                       "tensorflow_importable": _tf_importable()},
            "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": cores, "kind": "port", "sample": desc},
            "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------
EPOCH = int(os.environ.get("CTR_BENCH_EPOCH", "16"))  # steps per epoch of the exact-deferred update (csrc/epoch.cu); 16 is the
# reported configuration, the override exists for the epoch-length trade-off measurement in DESIGN.md §6


def main_b200(args):
    import torch
    import torch.distributed as dist

    from tf_repos_b200 import _lib, synth
    from tf_repos_b200.deepfm import DeepFM

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; there is no CPU fallback for the b200 arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    c = CFG
    N, B, F, K = args.vocab, args.batch, c["field_size"], c["embedding_size"]

    sharded = world > 1 and args.tables in ("auto", "sharded")
    if sharded:
        # every rank owns the rows id % world == rank (and sweeps only those); ids / rows / gradient rows
        # travel by NCCL all-to-all.  Same result as one GPU on the concatenated batch (tests/test_gpu_sharded.py).
        from tf_repos_b200.sharded import ShardedDeepFM
        model = ShardedDeepFM(F, N, K, B, deep_layers=c["deep_layers"], dropout=c["dropout"], l2_reg=c["l2_reg"],
                              learning_rate=c["learning_rate"], optimizer=c["optimizer"],
                              update_mode="exact_deferred", epoch_steps=EPOCH, device=dev, seed=0)
    else:
        model = DeepFM(F, N, K, B, deep_layers=c["deep_layers"], dropout=c["dropout"], l2_reg=c["l2_reg"],
                       learning_rate=c["learning_rate"], optimizer=c["optimizer"], update_mode="exact_deferred",
                       epoch_steps=EPOCH, device=dev, seed=0, world=world)
    host = [synth.criteo_batch(B, N, F, seed=rank * 1000 + i, zipf=args.zipf) for i in range(N_BATCHES)]
    devb = [tuple(t.to(dev) for t in b) for b in host]
    pinned = [tuple(t.pin_memory() for t in b) for b in host]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    use_graphs = world == 1 and os.environ.get("CTR_BENCH_GRAPHS", "1") != "0"
    if sharded:      # the compute segment between the two exchanges replays from one CUDA graph (sharded.py)
        model.use_graphs = os.environ.get("CTR_BENCH_GRAPHS", "1") != "0"

    def train(ids, vals, labels):
        # public API either way; the graphed form replays the step's launches from a CUDA graph (same kernels, same
        # results: tests/test_gpu_deferred_headline.py::test_graph_replayed_steps_equal_eager_steps)
        if use_graphs and model.update_mode == "exact_deferred":
            return model.train_step_graphed(ids, vals, labels)
        return model.train_step(ids, vals, labels)

    last = {}

    def step_dev(i):
        ids, vals, labels = devb[i % N_BATCHES]
        last["ids"], last["parts"] = ids, train(ids, vals, labels)

    counts = {}
    step_exact_marker = object()

    def timed(fn, steps, warmup, finish=None):
        """W untimed steps (+ untimed steps up to the next epoch boundary), then EXACTLY `steps` timed
        steps; `finish` (flush of deferred work) runs INSIDE the timed region."""
        i = 0
        for _ in range(warmup):
            fn(i); i += 1
        while model.update_mode == "exact_deferred" and model.epoch_pos != 0:
            fn(i); i += 1
        # CUDA graphs: a position's first visit runs eagerly and its second visit captures; both belong to warm-up
        if use_graphs and model.update_mode == "exact_deferred" and fn is not step_exact_marker:
            for _ in range(3):
                if len(getattr(model, "_graphs", {})) >= EPOCH - 1:
                    break
                for _ in range(EPOCH):
                    fn(i); i += 1
        barrier()
        if model.updater.sweep_events is not None:
            model.updater.sweep_events = []
            model.updater.sweep_steps = []
        counts["n0"] = _lib.launch_count() + getattr(model, "replayed_launches", 0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn(i); i += 1
        if finish is not None:
            finish()
        e1.record()
        counts["launches"] = _lib.launch_count() + getattr(model, "replayed_launches", 0) - counts["n0"]
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    # ---- value: inputs resident in HBM; exact-deferred update (bit-identical state to TF-exact) ------
    sampler = ClockSampler(local)
    model.updater.sweep_events = []
    sampler.start()
    ms_total = timed(step_dev, args.steps, args.warmup, finish=model.flush)
    sampler.stop_flag = True
    launches = counts["launches"]
    sweep_ms = [a.elapsed_time(b) for a, b in model.updater.sweep_events]
    sweep_steps = list(model.updater.sweep_steps)
    model.updater.sweep_events = None
    model.check_ids()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, model, last["parts"], last["ids"])
    ms_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total * 1e-3)

    # ---- e2e: pinned host inputs -> device, loss back to host, every step ----------------------------
    # inputs travel pinned host -> device on a copy stream, double-buffered: batch i+1 is in flight while step i
    # computes (every batch is copied inside the timed region; the step waits on its own batch's event)
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [tuple(torch.empty_like(t) for t in devb[0]) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    free = [torch.cuda.Event() for _ in range(2)]
    for ev in free:
        ev.record()
    in_flight = {"next": -1}
    loss_h = torch.zeros(args.steps + args.warmup + 2 * EPOCH + 8, 3).pin_memory()
    reg_h = torch.zeros(2, EPOCH).pin_memory()

    def prefetch(i):
        b = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(free[b])          # the step that last read this buffer is done with it
            for dst, src in zip(bufs[b], pinned[i % N_BATCHES]):
                dst.copy_(src, non_blocking=True)
            ready[b].record(copy_stream)
        in_flight["next"] = i + 1

    def step_host(i):
        b = i % 2
        if in_flight["next"] <= i:                   # first step of a run: nothing was prefetched for it
            prefetch(i)
        cur = torch.cuda.current_stream()
        cur.wait_event(ready[b])
        prefetch(i + 1)                              # other buffer: overlaps with this step's compute
        parts = train(*bufs[b])
        free[b].record(cur)
        loss_h[i % loss_h.shape[0]].copy_(parts, non_blocking=True)       # CE of this step
        if model.epoch_pos == 0 and not sharded:                          # L2 terms of the epoch just closed
            reg_h.copy_(model.epoch_reg_terms(), non_blocking=True)

    sampler2 = ClockSampler(local)
    model.updater.sweep_events = []
    sampler2.start()
    ms_e2e = timed(step_host, args.steps, 2, finish=model.flush)
    sampler2.stop_flag = True
    e2e_sweep_ms = [a.elapsed_time(b) for a, b in model.updater.sweep_events]
    model.updater.sweep_events = None
    e2e_value = world * B * args.steps / (ms_e2e * 1e-3)
    h2d = sum(t.numel() * t.element_size() for t in pinned[0])
    last_loss = float(loss_h[(args.steps + 1) % loss_h.shape[0]][0] + reg_h[:, -1].sum())

    extras = {}
    exact_sweep_ms = []

    def sweep_stats(ms_list, steps_list):
        full = [m for m, st in zip(ms_list, steps_list) if st == EPOCH]
        part = [(m, st) for m, st in zip(ms_list, steps_list) if st != EPOCH]
        return full, part

    if not args.no_extras and not sharded:
        # ---- heavy-tailed ids (SURVEY 8d secondary distribution) ------------------------------------------------
        if args.zipf == 0.0:
            zb = [tuple(t.to(dev) for t in synth.criteo_batch(B, N, F, seed=7000 + i, zipf=1.05)) for i in range(N_BATCHES)]

            def step_zipf(i):
                train(*zb[i % N_BATCHES])
            ms_z = timed(step_zipf, 2 * EPOCH, 3, finish=model.flush)
            extras["zipf_1.05"] = {"value": world * B * 2 * EPOCH / (ms_z * 1e-3), "unit": "samples/s",
                                   "ms_per_step": ms_z / (2 * EPOCH),
                                   "note": "same workload, heavy-tailed ids inside each categorical sub-vocabulary"}
            del zb

        # ---- e2e from libsvm TEXT: host bytes -> H2D -> device tokenizer (csrc/libsvm_device.cu) -> step ---------
        import io
        from tf_repos_b200 import ops as _ops
        texts = []
        for b in host[:4]:
            buf = io.StringIO()
            ids_n, vals_n, lab_n = (t.numpy() for t in b)
            for r in range(B):
                buf.write("%d " % int(lab_n[r]))
                buf.write(" ".join("%d:%s" % (int(i), ("%.6f" % v) if v != 1.0 else "1") for i, v in zip(ids_n[r], vals_n[r])))
                buf.write("\n")
            raw = buf.getvalue().encode()
            texts.append(torch.frombuffer(bytearray(raw), dtype=torch.uint8).pin_memory())
        text_dev = [torch.empty(max(t.numel() for t in texts), dtype=torch.uint8, device=dev) for _ in range(2)]
        loss_t = torch.zeros(3).pin_memory()

        def step_text(i):
            src = texts[i % len(texts)]
            dst = text_dev[i % 2][: src.numel()]
            dst.copy_(src, non_blocking=True)
            ids_t, vals_t, labels_t, consumed, needs_host = _ops.parse_libsvm_device(dst, F, B, final_chunk=True)
            assert not needs_host and ids_t.shape[0] == B
            parts = train(ids_t, vals_t, labels_t)
            loss_t.copy_(parts, non_blocking=True)
        ms_t = timed(step_text, 2 * EPOCH, 3, finish=model.flush)
        extras["e2e_text"] = {"value": world * B * 2 * EPOCH / (ms_t * 1e-3), "unit": "samples/s",
                              "ms_per_step": ms_t / (2 * EPOCH), "h2d_bytes_per_step": int(texts[0].numel()),
                              "note": "libsvm text in pinned host memory -> H2D -> device tokenizer (decode_libsvm, "
                                      "DeepFM.py:65-81) -> train step, loss read back; one host sync per step (row count)"}
        del texts, text_dev

        # ---- steady state: the tables as they look after a long run -------------------------------------------
        # l2 + Adam pull every row nothing gathers to ~FLT_MIN with a denormal first moment (DESIGN.md section 6;
        # tests/test_fastpath_guard_coverage.py simulates it).  The packed sweep handles that state with its scaled
        # loops; this leg times the same steps from that state.
        model.set_update_mode("exact_deferred")          # closes the open epoch
        g = torch.Generator(device=dev).manual_seed(11)
        CH = 1 << 27
        for t in model.tables:
            flat = [t.var.view(-1), t.slots[0].view(-1), t.slots[1].view(-1)]
            for o in range(0, flat[0].numel(), CH):
                n = min(CH, flat[0].numel() - o)
                u = lambda: torch.rand(n, device=dev, generator=g)
                sgn = lambda: torch.where(u() < 0.5, -1.0, 1.0)
                flat[0][o:o + n] = sgn() * (0.25 + 4.0 * u()) * 2.0 ** -126
                mm = sgn() * u() * 4e-42
                flat[1][o:o + n] = torch.where(u() < 0.2, torch.zeros_like(mm), mm)
                flat[2][o:o + n] = (0.5 + u()) * 1e-24
        model.opt.state[0] = 0.0
        model.opt.state[1] = 0.999 ** 3000
        model.updater.sweep_events = []
        ms_ss = timed(step_dev, 2 * EPOCH, 3, finish=model.flush)
        ss_full, _ = sweep_stats([a.elapsed_time(b) for a, b in model.updater.sweep_events], model.updater.sweep_steps)
        model.updater.sweep_events = None
        extras["steady_state"] = {"value": world * B * 2 * EPOCH / (ms_ss * 1e-3), "unit": "samples/s",
                                  "ms_per_step": ms_ss / (2 * EPOCH),
                                  "sweep_full_pass_ms": (sum(ss_full) / len(ss_full) if ss_full else None),
                                  "note": "same steps from the parked long-run state (var ~FLT_MIN, denormal m, "
                                          "v ~1e-24, lr_t ~ lr)"}
        # back to a fresh table for the side measurements below
        model.set_update_mode("exact_deferred")
        for t in model.tables:
            _ops.init_trunc_normal(t.var, (2.0 / (t.N + t.K)) ** 0.5 if t.K > 1 else (1.0 / t.N) ** 0.5, 3)
            for sl in t.slots:
                _ops.fill(sl, 0.0)

        model.set_update_mode("exact")
        model.updater.sweep_events = []
        ms_ex = timed(step_dev, max(args.steps // 2, 4), 2)
        exact_sweep_ms = [a.elapsed_time(b) for a, b in model.updater.sweep_events][2:]
        model.updater.sweep_events = None
        extras["exact_every_step"] = {"value": world * B * max(args.steps // 2, 4) / (ms_ex * 1e-3), "unit": "samples/s",
                                      "ms_per_step": ms_ex / max(args.steps // 2, 4),
                                      "note": "same results; full-table Adam sweep every step (HBM-bound)"}
        model.set_update_mode("lazy")
        ms_lazy = timed(step_dev, args.steps, 3)
        extras["lazy"] = {"value": world * B * args.steps / (ms_lazy * 1e-3), "unit": "samples/s",
                          "ms_per_step": ms_lazy / args.steps,
                          "note": "gathered rows only (LazyAdam-like): NOT TensorFlow's result; context only"}

        def infer(i):
            (model.predict_graphed if use_graphs else model.predict)(devb[i % N_BATCHES][0], devb[i % N_BATCHES][1])
        ms_inf = timed(infer, args.steps, 3)
        extras["infer"] = {"value": world * B * args.steps / (ms_inf * 1e-3), "unit": "samples/s",
                           "ms_per_step": ms_inf / args.steps}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = peaks()
    n_rows = model.N_local if sharded else N
    table_bytes = n_rows * K * 4 * 6  # Adam: read var,m,v + write var,m,v (24 B/element) per pass over the table
    full_ms, part = sweep_stats(sweep_ms, sweep_steps)
    sweep_avg_ms = sum(full_ms) / max(len(full_ms), 1)
    achieved = table_bytes / (sweep_avg_ms * 1e-3) / 1e9 if full_ms else None
    traffic, issue_pct = None, None
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "sweep_traffic.json")))
        issue_pct = t.get("epoch_issue_active_pct")
        if t.get("n_elem") == n_rows * K:
            traffic = t.get("epoch_dram_bytes_per_launch")
    except Exception:
        pass
    line = {"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]: DeepFM 39 fields, 200M vocab, k=16, bs=8192 per GPU, Adam, l2 1e-4, "
                                   "dropout 0.5, exact TensorFlow update semantics (every row moves every step); "
                                   f"exact-deferred update, epoch of {EPOCH} steps (state bit-identical to sweeping "
                                   "every step); the timed region ends with a flush of all deferred work",
                       "vocab": N, "batch_per_gpu": B, "id_distribution": ("uniform" if args.zipf == 0.0 else f"heavy-tailed (zipf={args.zipf})"), "l2_flush": "inputs larger than L2: every epoch streams the "
                       "whole 38.4 GB fm_v/m/v state; 16 distinct pre-staged batches are cycled",
                       "parallelism": ("single GPU" if world == 1 else
                                       f"dp{world} batches, tables row-sharded by id % {world}: NCCL all-to-all of ids / "
                                       "rows / gradient rows, all-reduce of dense gradients" if sharded else
                                       f"dp{world}: replicated tables, all-gather of sparse gradients, all-reduce of "
                                       "dense gradients")},
            "e2e": {"value": e2e_value, "unit": "samples/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 12 + 8, "last_loss": last_loss,
                    "sweep_avg_ms": (sum(e2e_sweep_ms) / len(e2e_sweep_ms) if e2e_sweep_ms else None),
                    "clocks": sampler2.summary()},
            "gpu_launches": launches, "clocks": sampler.summary(),
            "roofline": {"kernel": f"epoch_sweep_adam_kernel on fm_v ({EPOCH} Adam steps per element per pass; CUDA events around the pass incl. the ~1 ms second pass over the rows gathered during the epoch)",
                         "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak if achieved else None), "traffic": traffic,
                         "algorithmic_bytes_per_launch": table_bytes, "avg_launch_ms": sweep_avg_ms,
                         "launches_timed": len(full_ms), "peak_source": peak_src,
                         # passes that replayed fewer steps (the flush that ends the timed region): same bytes, less
                         # arithmetic -- reported apart, NOT averaged into `achieved`
                         "partial_passes": [{"steps": st, "ms": m, "GBps": table_bytes / (m * 1e-3) / 1e9} for m, st in part],
                         "kernel_share_of_step": (sum(sweep_ms) / ms_total if sweep_ms else None),
                         # the same work in the every-step formulation (EPOCH passes of 24 B/element): what HBM
                         # would have to deliver to match this launch -- context, not the roofline fraction
                         "per_step_formulation_equiv_GBps": (EPOCH * achieved if achieved else None),
                         "issue_active_pct_ncu": issue_pct,
                         "fma_pipe_active_pct_ncu": (json.load(open(os.path.join(ROOT, "profiles", "sweep_traffic.json"))).get("epoch_fma_pipe_active_pct") if os.path.exists(os.path.join(ROOT, "profiles", "sweep_traffic.json")) else None),
                         "note": "by design NOT HBM-bound: the pass replays 16 optimizer steps per element in registers (IEEE "
                                 "div+sqrt recurrence: 21 fp32 operations + 2 MUFU per element-step, bit-identical to the every-step "
                                 "formulation) to cut HBM traffic 16x; its limiter is instruction issue on the packed fp32 pipe "
                                 "(FFMA2-class instructions hold the port 2 cycles: profiles/r02_ubench_f32x2.txt, "
                                 "profiles/r02_ncu_sweep_adam_packed.txt).  `frac` is computed from full 16-step passes only; the "
                                 "flush that ends the timed region is listed under partial_passes.  The HBM-bound formulation of the "
                                 "same update is reported under exact_every_step; the same steps from the long-run (parked) table "
                                 "state under steady_state."}}
    if exact_sweep_ms:
        ex_avg = sum(exact_sweep_ms) / len(exact_sweep_ms)
        tr = None
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", "sweep_traffic.json")))
            if t.get("n_elem") == N * K:
                tr = t["dram_bytes_per_launch"]
        except Exception:
            pass
        extras["exact_every_step"]["roofline"] = {
            "kernel": "opt_dense_sweep_kernel<ADAM> on fm_v (one Adam step per element per pass)", "bound": "hbm",
            "achieved": table_bytes / (ex_avg * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
            "frac": table_bytes / (ex_avg * 1e-3) / 1e9 / peak, "traffic": tr, "avg_launch_ms": ex_avg,
            "launches_timed": len(exact_sweep_ms)}
    line.update(extras)
    if world == 1 and not args.no_extras:
        # ---- BASELINE.json configs[2] (DCN) and configs[3] (DIN), same engine, same update semantics ---------
        del model
        torch.cuda.empty_cache()
        model = None
        line.update(side_models(torch, dev, synth, args.vocab))
    if world == 1 and not args.no_cpu_baseline:
        del model
        torch.cuda.empty_cache()
        sps, ms, done, cores, desc = run_cpu(50, 1, 20.0, N, B)
        line["cpu_baseline"] = {"value": sps, "unit": "samples/s", "cores": cores, "kind": "port", "sample": desc,
                                "ms_per_step": ms}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_ROWS = 1 << 17  # table rows of each kind in --dump-outputs: rows the last step gathered, rows drawn at random


def dump_outputs(out_dir, model, parts, ids):
    """Writes what the last timed step computed as float32 / float64 DIR/<name>.npy (about 20 MB here; at most 64 MB).
    Inputs, initial state and dropout masks follow from fixed seeds, so two builds run with the same arguments can be
    compared file by file.  The 200M-row tables are sampled with a fixed seed: up to DUMP_ROWS rows the last step
    gathered (their gradient moved them) plus DUMP_ROWS uniform rows (only the l2 term moved them)."""
    import numpy as np
    import torch

    g = torch.Generator().manual_seed(0)

    def sample(x, n):
        return x if x.numel() <= n else x[torch.randperm(x.numel(), generator=g)[:n].sort().values]

    variables = model.variables()
    gathered = sample(torch.unique(ids.reshape(-1).long().cpu()), DUMP_ROWS)
    rows = torch.unique(torch.cat([gathered, torch.randint(0, model.N, (DUMP_ROWS,), generator=g)]))
    rows_dev = rows.to(model.device)
    # the step's loss, left to right: mean CE, then the l2 terms of the tables, which the exact-deferred update
    # computes in its sweep rather than in the step's returned tensor
    pos = (model.epoch_pos - 1) % model.epoch_steps
    n_tab = len(model.tables)
    out = {"loss_terms": torch.cat([parts[:-n_tab], model.epoch_reg_terms()[:, pos]]),
           "prob": sample(model.pred[: model.B].cpu(), 1 << 20),
           "sample_rows": rows.double(),
           "fm_v_sample_rows": variables["fm_v"][rows_dev],
           "fm_w_sample_rows": variables["fm_w"][rows_dev]}
    out.update({name.replace("/", "."): v for name, v in variables.items() if name not in ("fm_v", "fm_w")})
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v.detach().cpu().numpy())


def side_models(torch, dev, synth, vocab):
    """DCN (cross_layers=6) and DIN (seq_len 100, 100M items, k=32, bs=4096) training samples/s, exact-deferred update,
    inputs resident in HBM, CUDA-event timed over one epoch of 16 steps + the closing sweep."""
    out = {}

    def timeit(step, m, steps, graphed=False):
        for i in range(3):
            step(i)
        while m.epoch_pos != 0:
            step(0)
        if graphed:      # a position's first visit is eager, its second visit captures the CUDA graph: both are warm-up
            for i in range(2 * EPOCH):
                step(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step(i)
        m.flush()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    try:
        from tf_repos_b200.dcn import DCN
        B, F, K, L = 8192, 39, 16, 6
        bt = [synth.criteo_batch(B, vocab, F, seed=50 + i, device=dev) for i in range(8)]
        m = DCN(F, vocab, K, B, cross_layers=L, update_mode="exact_deferred", epoch_steps=EPOCH, device=dev)
        ms = timeit(lambda i: m.train_step_graphed(*bt[i % 8]), m, 2 * EPOCH, graphed=True)
        out["configs[2]_dcn"] = {"value": B / ms * 1e3, "unit": "samples/s", "ms_per_step": ms,
                                 "config": f"DCN 1xB200, B={B} F={F} vocab={vocab} k={K} cross_layers={L}, Adam, l2 1e-4, "
                                           "dropout 0.5, exact TF update semantics (exact-deferred)"}
        del m, bt
        torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001
        out["configs[2]_dcn"] = {"error": repr(e)[:300]}
    try:
        from tf_repos_b200.din import DIN
        B, Fp, N, K, P = 4096, 11, 100_000_000, 32, 100
        bt = []
        for i in range(4):
            b, l = synth.din_batch(B, N, Fp, P, 8, seed=i)
            bt.append(({k: v.to(dev) for k, v in b.items()}, l.to(dev)))
        m = DIN(Fp, N, K, B, P, max_a_int=8, update_mode="exact_deferred", epoch_steps=EPOCH, device=dev)
        ms = timeit(lambda i: m.train_step(*bt[i % 4]), m, EPOCH)
        out["configs[3]_din"] = {"value": B / ms * 1e3, "unit": "samples/s", "ms_per_step": ms,
                                 "config": f"DIN 1xB200, B={B} F'={Fp} seq_len={P} (lengths ~U[1,100]) items={N} k={K}, "
                                           "attention hidden 256, Adam, l2 1e-4, dropout 0.5, exact-deferred update"}
        del m, bt
        torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001
        out["configs[3]_din"] = {"error": repr(e)[:300]}
    return out


if __name__ == "__main__":
    a = parse()
    # stdout carries exactly ONE line (the JSON): anything a library prints on fd 1 meanwhile (NCCL's version
    # banner, ...) goes to stderr
    sys.stdout.flush()
    _saved_stdout = os.dup(1)
    os.dup2(2, 1)
    _real_print = print

    def print(*args, **kw):  # noqa: A001 -- the JSON lines below are the only print() calls that reach stdout
        sys.stdout.flush()
        os.dup2(_saved_stdout, 1)
        _real_print(*args, **kw)
        sys.stdout.flush()
        os.dup2(2, 1)

    if a.impl == "reference":
        main_reference(a)
    else:
        main_b200(a)
