#!/usr/bin/env python
"""bench.py — QA-rounds/s of one pass of the hot path over one synthetic VisDial-shaped batch (BASELINE.json metric).

  --config C4 (default, the headline): `mn-att-ques-im-hist + disc` training step, B = 32 dialogs per GPU
           C1 lf-ques+gen (B=4, V=1k) | C2 lf-ques-im-hist+disc (fc7) | C3 hrea-ques-im-hist+gen — training steps
           C5 the 100-option disc ranker (eval step: encoder + option LSTM + scores + ranks), sweep B = 32..1024 per GPU

A training "step" = Model:trainIteration minus data loading (model.lua:66-106): zeroGradParameters, forward, criterion,
backward, [gradient all-reduce], clamp(-5,5), adam.

  value        : whole-job QA-rounds/s with the batch already resident in HBM (device-timed, max over ranks)
  e2e          : the same step through the reference-facing Model.trainIteration with HOST (pinned) batch buffers: the
                 H2D of the batch and the D2H loss read are inside the timed region
  roofline     : the dominant kernel class (the option-LSTM step), EXECUTED FLOP / CUDA-event time on its stream
  rank_agreement: eval ranks of the benched math mode vs the engine's fp32 mode on the benched batch
  cpu_baseline : the oracle ("port" of the reference's CPU path) on a bounded sample, rank 0, N=1 only

`--impl reference` times the reference's own CPU structure (oracle/, torch CPU fp32, thread count chosen by a sweep)
for the same metric and config; it imports numpy / torch / oracle only — never visdial_b200, so the product library is
not loaded into the reference process.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

FWD_FLOP_PER_ROUND_C4 = 7311261696          # SURVEY.md §8d (C4), forward; training = 3x
LSTM_STEP_KEYS = ("lstm_step", "lstm_step_bwd")

# opts.lua:6-40 defaults (kept here as a plain dict so that the reference arm needs no visdial_b200 import;
# tests/test_host.py checks it against visdial_b200.engine.DEFAULT_PARAMS)
DEFAULTS = dict(
    encoder="lf-ques-hist", decoder="gen", vocabSize=0, embedSize=300, rnnHiddenSize=512, numLayers=2,
    imgFeatureSize=4096, imgSpatialSize=14, imgEmbedSize=300, commonEmbeddingSize=512,
    numAttentionLayers=1, maxQuesCount=10, numOptions=100, dropout=0.5, gpuid=0,
    batchSize=40, learningRate=1e-3, lrDecayRate=0.9997592083, minLRate=5e-5, useGt=True, imgNorm=1,
)

CONFIGS = {
    "C1": dict(encoder="lf-ques", decoder="gen", batch=4, vocabSize=1000, mode="train",
               workload="C1 lf-ques+gen train step (no image/history, 10 rounds, 20-token sequences, V=1000)"),
    "C2": dict(encoder="lf-ques-im-hist", decoder="disc", batch=32, vocabSize=10000, mode="train", imgFeatureSize=4096,
               workload="C2 lf-ques-im-hist+disc train step (VGG fc7 4096-d, concatenated history, 10 rounds, 100 options x 20 tokens, V=10000)"),
    "C3": dict(encoder="hrea-ques-im-hist", decoder="gen", batch=32, vocabSize=10000, mode="train", imgFeatureSize=4096,
               workload="C3 hrea-ques-im-hist+gen train step (VGG fc7 4096-d, hierarchical LSTM + attention over history, V=10000)"),
    "C4": dict(encoder="mn-att-ques-im-hist", decoder="disc", batch=32, vocabSize=10000, mode="train", imgFeatureSize=512,
               workload="C4 mn-att-ques-im-hist+disc train step (pool5 14x14x512, 10 rounds, 100 options x 20 tokens, V=10000)"),
    "C5": dict(encoder="mn-att-ques-im-hist", decoder="disc", batch=32, vocabSize=10000, mode="eval", imgFeatureSize=512,
               sweep=(32, 64, 128, 256, 512, 1024),
               workload="C5 disc 100-option ranker eval step (mn-att-ques-im-hist encoder + option LSTM + dot-product scores + ranks), batch sweep"),
}


def config_params(name, gpuid=0):
    c = CONFIGS[name]
    p = dict(DEFAULTS)
    p.update(encoder=c["encoder"], decoder=c["decoder"], vocabSize=c["vocabSize"], gpuid=gpuid)
    if "imgFeatureSize" in c:
        p["imgFeatureSize"] = c["imgFeatureSize"]
    enc = p["encoder"]                                   # opts.lua:55-67
    p["useHistory"], p["useIm"], p["concatHistory"] = "hist" in enc, "im" in enc, "lf" in enc
    if "att" in enc:
        p["imgNorm"] = 0
    return p


def metric_name(name):
    c = CONFIGS[name]
    return "QA-rounds/sec %s+%s %s" % (c["encoder"], c["decoder"], "train step" if c["mode"] == "train" else "ranker eval step")


def workload_config(name, batch, world):
    return {"workload": CONFIGS[name]["workload"], "dialogs_per_gpu": batch, "global_batch_dialogs": batch * world,
            "parallelism": "dp%d" % world,
            "l2": "per-step working set (LSTM gates/activations, GBs) >> 126 MB L2; 4 rotating input batches"}


def load_synthetic():
    """visdial_b200/synthetic.py is numpy-only: load it by path so that the package (and its ctypes binding) stays out."""
    spec = importlib.util.spec_from_file_location("vd_synthetic", os.path.join(ROOT, "visdial_b200", "synthetic.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"bf16_sustained": d.get("bf16_tflops_sustained", 1449.3), "bf16_burst": d.get("bf16_tflops", 1693.7),
                "hbm": d.get("hbm_gbs", 6579.6), "src": "measured"}
    return {"bf16_sustained": 1400.0, "bf16_burst": 1590.0, "hbm": 6650.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md).  The sampler runs from
    before the warm-up; only samples whose nvidia-smi timestamp falls inside the marked window are kept."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc, self.t0, self.t1 = gpu_index, [], None, None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def mark_begin(self):
        import datetime
        self.t0 = datetime.datetime.now()

    def mark_end(self):
        import datetime
        self.t1 = datetime.datetime.now()

    def stop(self):
        import datetime
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.t.join(timeout=2)
        keep = []
        for r in self.rows:
            if len(r) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f")
            except ValueError:
                continue
            if self.t0 is None or (self.t0 <= ts <= self.t1):
                keep.append(r)
        num = lambda x: x.replace(".", "", 1).isdigit()
        sm = [float(r[1]) for r in keep if num(r[1])]
        mx = [float(r[2]) for r in keep if num(r[2])]
        pw = [float(r[3]) for r in keep if num(r[3])]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in keep for i in range(4) if r[4 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": reasons, "samples": len(sm)}


def dump_sample(a, n=1 << 22):
    """`a` flattened; past n entries, a fixed seeded sample of n of them (same indices for the same length)."""
    a = np.asarray(a).ravel()
    if a.size <= n:
        return a
    return a[np.sort(np.random.default_rng(0).choice(a.size, n, replace=False))]


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array as out_dir/<name>.npy, float64 kept, everything else as float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    return rank, local, world


def barrier(world):
    if world > 1:
        import torch
        import torch.distributed as dist
        dist.barrier()
        torch.cuda.synchronize()


def max_over_ranks(x, world):
    if world <= 1:
        return x
    from visdial_b200 import dist as vdist
    return vdist.max_over_ranks(x)


# ------------------------------------------------------------------------------------------------ CPU arm (oracle only)
class CpuArm:
    """The oracle (CPU restatement of the reference, torch fp32) on one config: numpy / torch / oracle imports only."""

    def __init__(self, cfg_name):
        import torch
        from oracle import layout as OL
        self.torch, self.OL = torch, OL
        self.name, self.cfg = cfg_name, CONFIGS[cfg_name]
        self.p = config_params(cfg_name)
        self.synth = load_synthetic()
        self.flat = OL.init_parameters(self.p, seed=1234)
        self.W = torch.from_numpy(self.flat)
        self.state = {}
        self.it = 0

    def _tb(self, B, seed):
        torch = self.torch
        nb = self.synth.make_batch(self.p, B, seed=seed)
        out = {}
        for k, v in nb.items():
            t = torch.from_numpy(np.ascontiguousarray(v))
            out[k] = t.long() if v.dtype.kind in "iu" else t
        return out

    def step(self, B, structure):
        """One pass over B dialogs; returns seconds (batch creation excluded)."""
        from oracle import philox, visdial_oracle as O
        torch = self.torch
        self.it += 1
        tb = self._tb(B, 1234 + self.it)
        P = {k: torch.from_numpy(v) for k, v in self.OL.split_parameters(self.p, self.W.numpy()).items()}
        t0 = time.perf_counter()
        if self.cfg["mode"] == "train":
            out = O.forward_backward(O.Ctx(train=True, mask_fn=philox.make_mask_fn(1234, self.it), structure=structure), self.p, P, tb)
            dW = torch.from_numpy(self.OL.flat_from_named(self.p, out["grads"]))
            O.clamp_adam(self.W, dW, self.state, 1e-3)
        else:
            O.retrieve_batch(O.Ctx(train=False, structure=structure), self.p, P, tb, use_gt=True)
        return time.perf_counter() - t0

    def sweep_threads(self, B, structure, candidates=(8, 16, 32, 64, 128)):
        """QA-rounds/s of one step at increasing thread counts (one untimed step first); returns (best, table).  The sweep
        stops at the first count that is slower than the best so far: the reference structure is a chain of small
        per-timestep ops, and on the 128-vCPU GPU host over-subscribed counts take MINUTES per step (r01: 8 threads
        1.4 s, 32 threads 4.1 s, 128 threads did not finish), so an exhaustive sweep would not be a bounded sample."""
        torch = self.torch
        ncpu = os.cpu_count() or 1
        cands = sorted({min(c, ncpu) for c in candidates})
        torch.set_num_threads(cands[0])
        self.step(min(B, 2), structure)                      # page in / allocator warm-up
        table = {}
        for t in cands:
            torch.set_num_threads(t)
            sec = self.step(B, structure)
            table[t] = B * 10 / sec
            if table[t] < 0.95 * max(table.values()):
                break
        best = max(table, key=table.get)
        torch.set_num_threads(best)
        return best, table


def run_reference(args):
    """The reference's own CPU path for the same metric/config: oracle in REFERENCE structure (per-timestep addmm, 100
    sequential option-LSTM passes, materialised repeatTensor), thread count from a sweep, the GPU arm's batch size when
    the whole --steps/--warmup run fits the time budget (else 8 dialogs, stated in `config`)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    arm = CpuArm(args.config)
    cfgB = CONFIGS[args.config]["batch"] if args.batch <= 0 else args.batch
    probeB = min(cfgB, 8)
    if args.cpu_threads > 0:
        threads, table = min(args.cpu_threads, os.cpu_count() or 1), {}
        arm.torch.set_num_threads(threads)
        arm.step(min(cfgB, 2), "reference")
    else:
        threads, table = arm.sweep_threads(probeB, "reference", candidates=(4, 8, 16, 32, 64, 128))
    total_steps = args.steps + args.warmup
    B = args.ref_batch
    if B <= 0:
        t_probe = arm.step(probeB, "reference")
        est = t_probe * cfgB / probeB                         # per-step time grows at most linearly in B
        B = cfgB if est * total_steps <= args.ref_budget_s else min(cfgB, 8)
    times = []
    for i in range(total_steps):
        dt = arm.step(B, "reference")
        if i >= args.warmup:
            times.append(dt)
    sec = float(np.median(times))
    val = B * 10 / sec
    # the "batched CPU" figure (BASELINE.md §3): same maths with the 100 option passes stacked into one LSTM pass
    batched = None
    if not args.no_batched:
        arm.step(min(B, 2), "batched")
        sb = arm.step(B, "batched")
        batched = {"value": B * 10 / sb, "unit": "QA-rounds/s", "cores": threads, "kind": "port",
                   "sample": "%d dialogs, 1 timed step, oracle batched structure (torch CPU fp32)" % B}
    line = {"impl": "reference", "metric": metric_name(args.config), "value": val, "unit": "QA-rounds/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.config, B, max(world, args.gpus)),
            "cpu_baseline": {"value": val, "unit": "QA-rounds/s", "cores": threads, "kind": "port",
                             "sample": "%d dialogs (%d QA rounds) per step, median of %d steps, oracle reference-structure, torch CPU "
                                       "fp32, %d threads of %d host CPUs" % (B, B * 10, len(times), threads, os.cpu_count() or 1)},
            "thread_sweep_qa_rounds_per_s": {str(k): v for k, v in table.items()}, "thread_sweep_dialogs": probeB,
            "cpu_baseline_batched": batched,
            "native_so_loaded": sorted({l.split()[-1] for l in open("/proc/self/maps") if "visdial_b200" in l}),
            "e2e": {"value": val, "unit": "QA-rounds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def run_ours(args, rank, local, world):
    from visdial_b200 import VD_MATH_F16, VD_MATH_FP32, VD_MATH_TF32, Batch, Model
    from visdial_b200 import dist as vdist
    from visdial_b200.engine import pinned_empty
    from visdial_b200.synthetic import make_batch

    cfg = CONFIGS[args.config]
    train = cfg["mode"] == "train"
    p = config_params(args.config, gpuid=local)
    B = cfg["batch"] if args.batch <= 0 else args.batch
    p["batchSize"] = B
    model = Model(p, seed=1234)                       # same seed on every rank -> identical replicas
    eng = model.engine
    MODES = {"fp32": VD_MATH_FP32, "tf32": VD_MATH_TF32, "f16": VD_MATH_F16}
    eng.set_math_mode(MODES[args.math])
    vdist.attach_engine(eng, rank, world)
    if not train:
        eng.set_training(0)

    def make_batches(nb_dialogs, n=4):
        host = []
        for i in range(n):
            nb = make_batch(p, nb_dialogs, seed=1234 + 1000 * rank + i)
            pinned = {}
            for k, v in nb.items():
                if k in ("option_in", "option_out"):
                    continue
                buf = pinned_empty(v.shape, v.dtype)
                buf[...] = v
                pinned[k] = buf
            host.append(Batch(pinned))
        return host, [b.to_device(eng) for b in host]

    class Loader:
        def __init__(self, batches):
            self.b, self.i = batches, 0

        def getTrainBatch(self, params):
            self.i += 1
            return self.b[self.i % len(self.b)]

    last = {}                                         # what the most recent step returned to its caller

    def one_step(loader):
        if train:
            last["loss"] = model.trainIteration(loader)
        else:
            last["ranks"] = eng.retrieve(loader.getTrainBatch(p), use_gt=True)

    def timed(loader, steps, profile):
        barrier(world)
        eng.synchronize()
        eng.profile_reset()
        eng.profile(profile)
        l0 = eng.launch_count()
        t_wall = time.perf_counter()
        eng.timer_start()
        for _ in range(steps):
            one_step(loader)
        ms = eng.timer_stop()
        eng.synchronize()
        wall = (time.perf_counter() - t_wall) * 1e3
        barrier(world)
        eng.profile(False)
        return ms, wall, eng.launch_count() - l0

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    if not train:                                     # ---- C5: ranker sweep
        sweep, outputs = {}, {}
        for Bs in cfg["sweep"]:
            host_b, dev_b = make_batches(Bs, n=2)
            dl, hl = Loader(dev_b), Loader(host_b)
            for _ in range(max(args.warmup, 3)):
                one_step(dl)
            one_step(hl)
            if rank == 0 and Bs == cfg["sweep"][0]:
                sampler.mark_begin()
            ms, _, launches = timed(dl, args.steps, 0)
            outputs["ranks_b%d" % Bs] = last["ranks"]
            ms_h, wall_h, _ = timed(hl, args.steps, 0)
            ms = max_over_ranks(ms, world)
            ms_h = max_over_ranks(max(ms_h, wall_h), world)
            sweep[Bs] = {"value": Bs * 10 * world * args.steps / (ms * 1e-3), "ms_per_step": ms / args.steps,
                         "e2e": Bs * 10 * world * args.steps / (ms_h * 1e-3), "h2d": host_b[0].h2d_bytes,
                         "d2h": Bs * 10 * 4, "launches": int(launches)}
            del host_b, dev_b
        if rank == 0:
            sampler.mark_end()
        clocks = sampler.stop() if rank == 0 else None
        if rank != 0:
            return
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        best = max(sweep, key=lambda k: sweep[k]["value"])
        line = {"metric": metric_name(args.config), "value": sweep[best]["value"], "unit": "QA-rounds/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": sweep[best]["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.math, "data": "synthetic",
                "config": workload_config(args.config, best, world),
                "e2e": {"value": sweep[best]["e2e"], "unit": "QA-rounds/s", "h2d_bytes_per_step": sweep[best]["h2d"],
                        "d2h_bytes_per_step": sweep[best]["d2h"]},
                "gpu_launches": sweep[best]["launches"], "clocks": clocks,
                "sweep_dialogs_per_gpu": {str(k): {"QA-rounds/s": v["value"], "e2e QA-rounds/s": v["e2e"], "ms_per_step": v["ms_per_step"]}
                                          for k, v in sweep.items()}}
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(args)
        print(json.dumps(line), flush=True)
        return

    # ---- training configs
    host_batches, dev_batches = make_batches(B)
    dev_loader, host_loader = Loader(dev_batches), Loader(host_batches)
    for _ in range(args.warmup):
        one_step(dev_loader)
    for _ in range(3):                      # the host-batch path has its own first-use costs (staging buffers, copy stream)
        one_step(host_loader)

    if rank == 0:
        sampler.mark_begin()
    if args.ncu_range:                      # `ncu --profile-from-start off`: profile exactly the timed steps
        eng.profiler_range(True)
    # level 2 = only the roofline kernel class (the big LSTM-step launches) is bracketed by CUDA events inside the timed
    # region; every other launch runs un-instrumented
    ms_dev, wall_dev, launches = timed(dev_loader, args.steps, 0 if args.ncu_range else 2)
    if args.ncu_range:
        eng.profiler_range(False)
    if args.dump_outputs and rank == 0:         # replicas are identical after the all-reduce: rank 0 speaks for all
        # the weights and gradients are 9-25 M entries per config: a sample of each keeps the dump under 64 MB
        dump_outputs(args.dump_outputs, {"loss": np.float64([last["loss"]]), "weights": dump_sample(model.wrapperW.numpy()),
                                         "gradients": dump_sample(model.wrapperdW.numpy())})
    stats_shared = {k: eng.kernel_stats(k) for k in LSTM_STEP_KEYS}
    ms_e2e, wall_e2e, _ = timed(host_loader, args.steps, 0)
    # Roofline pass: in the timed region above the option-LSTM kernels share the GPU with the encoder's concurrent
    # streams, so a CUDA-event bracket around one launch also contains the SM time it ceded.  The same K steps are
    # therefore run once more on ONE timeline (reference order: encoder, then decoder) and the dominant kernel's launch
    # duration is taken from there; the shared-machine figure is kept as `achieved_in_overlapped_step`.
    eng.set_option_overlap(False)
    one_step(dev_loader)
    ms_iso, _, _ = timed(dev_loader, args.steps, 2)
    stats = {k: eng.kernel_stats(k) for k in LSTM_STEP_KEYS}
    eng.set_option_overlap(True)
    one_step(dev_loader)
    # SURVEY §8(f) row 2: the same step fed by the HBM-resident corpus (dataloader.lua:324-478 on the device)
    resident = None
    if args.resident and args.config == "C4":
        resident = resident_corpus_arm(args, p, eng, model, timed, rank, world)
    if rank == 0:
        sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    # informational per-class breakdown from a separate, fully instrumented pass (classes on concurrent streams overlap,
    # so the entries do not add up to the step time)
    nprof = min(3, args.steps)
    timed(dev_loader, nprof, 1)
    breakdown = {k: round(eng.kernel_stats(k)["ms"] / nprof, 3) for k in
                 LSTM_STEP_KEYS + ("lstm_step_first", "lstm_step_bwd_last", "lstm_step_small", "lstm_step_bwd_small", "gemm",
                                   "gemm_wgrad", "embed_grad_segsum", "allreduce")}
    # rank fidelity of the benched math mode: eval ranks vs the engine's own fp32 mode on the benched batch
    agreement = None
    if cfg["decoder"] == "disc" and rank == 0 and not args.no_rank_check and args.math != "fp32":
        b0 = dev_batches[0]
        eng.set_training(0)
        r_mode = eng.retrieve(b0, use_gt=False)
        eng.set_math_mode(VD_MATH_FP32)
        r_f32 = eng.retrieve(b0, use_gt=False)
        eng.set_math_mode(MODES[args.math])
        eng.set_training(1)
        agreement = {"vs": "fp32 math mode of the same engine, same batch", "entries": int(r_mode.size),
                     "rank_agreement": float((r_mode == r_f32).mean()),
                     "top1_agreement": float(((r_mode == 1).argmax(1) == (r_f32 == 1).argmax(1)).mean()),
                     "max_rank_move": int(np.abs(r_mode.astype(np.int64) - r_f32).max())}

    ms_dev = max_over_ranks(ms_dev, world)
    ms_e2e = max_over_ranks(max(ms_e2e, wall_e2e), world)     # e2e includes host time: take the wall clock if larger
    if resident is not None:
        resident["ms"] = max_over_ranks(resident["ms"], world)
    rounds = B * 10 * world * args.steps
    value = rounds / (ms_dev * 1e-3)
    e2e = rounds / (ms_e2e * 1e-3)
    if rank != 0:
        return

    peaks = measured_peaks()
    f16 = args.math == "f16"
    # kind::f16 runs at the bf16 rate the driver measured with cuBLAS; TF32 operands at half of it (no TF32 peak was
    # measured by the driver; tools/measure_tf32_peak.py measures this repo's own 8192^3 TF32 kernel for comparison)
    peak = peaks["bf16_sustained"] if f16 else peaks["bf16_sustained"] / 2.0
    roofline = None
    n_l = sum(stats[k]["launches"] for k in LSTM_STEP_KEYS)
    if n_l > 0:
        fl = sum(stats[k]["flops"] for k in LSTM_STEP_KEYS)
        by = sum(stats[k]["bytes"] for k in LSTM_STEP_KEYS)
        t_ms = sum(stats[k]["ms"] for k in LSTM_STEP_KEYS)
        achieved = fl / (t_ms * 1e-3) / 1e12 if t_ms > 0 else 0.0
        per = {k: {"launches": stats[k]["launches"], "avg_launch_ms": stats[k]["ms"] / max(stats[k]["launches"], 1),
                   "TFLOP/s": stats[k]["flops"] / max(stats[k]["ms"] * 1e-3, 1e-12) / 1e12,
                   "algorithmic_GB/s": stats[k]["bytes"] / max(stats[k]["ms"] * 1e-3, 1e-12) / 1e9} for k in LSTM_STEP_KEYS}
        hbm_gbs = by / max(t_ms * 1e-3, 1e-12) / 1e9
        kernel_desc = ("k_lstm16<fwd|bwd>: option-LSTM step, fp16 operands (recurrent gate GEMM on tcgen05 kind::f16, CTA pairs, "
                       "fp32 TMEM accumulators + SeqLSTM pointwise epilogue)" if f16 else
                       "k_tc_gemm<256,LSTM_FWD|LSTM_BWD,2>: option-LSTM step (recurrent gate GEMM on tcgen05 kind::tf32 + SeqLSTM "
                       "pointwise epilogue)") + ", %d launches per training step" % (n_l // args.steps)
        # SURVEY.md §8(d) convention (algorithmic FLOP: the forward step is credited with the D = embedSize x-projection
        # 2*R*4H*(H+D) although it executes as a table gather) — reported NEXT TO the executed figure, never instead of it
        R_opt = B * p["maxQuesCount"] * p["numOptions"]
        fl_conv = fl + stats["lstm_step"]["launches"] * 2.0 * R_opt * 4 * p["rnnHiddenSize"] * p["embedSize"]
        conv = fl_conv / (t_ms * 1e-3) / 1e12 if t_ms > 0 else 0.0
        tensor = {"achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                  "flops_counted": "executed tensor-core FLOP only (2*R*4H*H per launch): the gathered x-projection and the K=0 first/"
                                   "last steps are not credited",
                  "peak_source": "%s bf16_tflops_sustained%s" % (peaks["src"], "" if f16 else " / 2 (TF32 operands)"),
                  "executed_flop_per_launch": fl / max(n_l, 1),
                  "achieved_survey_convention": conv, "frac_survey_convention": conv / peak,
                  "achieved_in_overlapped_step": (sum(stats_shared[k]["flops"] for k in LSTM_STEP_KEYS) /
                                                  max(sum(stats_shared[k]["ms"] for k in LSTM_STEP_KEYS) * 1e-3, 1e-12) / 1e12)}
        hbm = {"achieved": hbm_gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": hbm_gbs / peaks["hbm"],
               "bytes_counted": "algorithmic HBM bytes per launch (DESIGN.md §9): forward fp16 gates out + fp32 c in/out + fp16 h in/out = "
                                "10 KB per option row (the fp16 projection-table gather is L2-resident, not counted); backward fp16 gates "
                                "in + fp16 da in/out + fp32 c_{t-1}, c_t in + fp32 dc in/out = 20 KB per row",
               "peak_source": "%s hbm_gbs (MEASURED_PEAKS.json)" % peaks["src"], "algorithmic_bytes_per_launch": by / max(n_l, 1)}
        # VD_MATH_F16: the class sits nearer the HBM roof than the tensor roof (ncu: backward step DRAM 61 % / tensor 31 %, forward
        # 40 % / 34 %), so HBM is the binding roofline; the TF32 kernels are nearer their (assumed) tensor roof.  Both are always given.
        head = hbm if f16 else tensor
        roofline = {"bound": "hbm" if f16 else "tensor", "kernel": kernel_desc,
                    "achieved": head["achieved"], "peak": head["peak"], "unit": head["unit"], "frac": head["frac"],
                    "launches": n_l, "avg_launch_ms": t_ms / max(n_l, 1), "share_of_step": t_ms / max(ms_iso, 1e-9),
                    "per_direction": per, "hbm": hbm, "tensor": tensor,
                    "measured_in": "a second pass of the same %d steps with the option stream serialised behind the encoder "
                                   "(%.3f ms/step), CUDA events around every launch of this kernel class on its stream" % (args.steps, ms_iso / args.steps),
                    "traffic": None}
        tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")   # dram bytes per launch from the committed ncu --set full capture
        if os.path.exists(tpath):
            t = json.load(open(tpath)).get(args.math)
            if t:
                roofline["traffic"] = t["dram_bytes_per_launch_avg"]
                roofline["traffic_source"] = t["source"]
    line = {"metric": metric_name(args.config), "value": value, "unit": "QA-rounds/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": {"f16": "f16 operands + f16 saved state for the option LSTM, tf32 operands elsewhere; fp32 accumulate, fp32 cell state / "
                             "gradients / optimiser", "tf32": "tf32", "fp32": "f32"}[args.math],
            "data": "synthetic", "config": workload_config(args.config, B, world),
            "e2e": {"value": e2e, "unit": "QA-rounds/s", "h2d_bytes_per_step": host_batches[0].h2d_bytes,
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "rank_agreement": agreement,
            "kernel_ms": breakdown, "wall_ms_per_step": wall_dev / args.steps}
    if args.config == "C4":
        step_flops = 3.0 * FWD_FLOP_PER_ROUND_C4 * B * 10
        line["step_tflop_algorithmic"] = step_flops / 1e12
        line["step_tflops_achieved"] = step_flops / (ms_dev / args.steps * 1e-3) / 1e12
    if resident is not None:
        line["e2e_resident_corpus"] = resident_line(resident, rounds, peaks, args)
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline(args)
    print(json.dumps(line), flush=True)


def cpu_baseline(args):
    """Bounded CPU sample for the GPU arm's line (rank 0, N = 1): thread sweep at 2 dialogs, then one timed step of the
    oracle in reference structure at `--cpu-batch` dialogs (about 10-30 s of CPU work on the GPU host)."""
    arm = CpuArm(args.config)
    Bc = min(args.cpu_batch, CONFIGS[args.config]["batch"])
    if args.cpu_threads > 0:
        threads = min(args.cpu_threads, os.cpu_count() or 1)
        arm.torch.set_num_threads(threads)
        arm.step(min(Bc, 2), "reference")
        table = {}
    else:
        threads, table = arm.sweep_threads(min(Bc, 2), "reference", candidates=(4, 8, 16, 32, 64))
    sec = arm.step(Bc, "reference")
    return {"value": Bc * 10 / sec, "unit": "QA-rounds/s", "cores": threads, "kind": "port",
            "sample": "%d dialogs (%d QA rounds), 1 timed step of the oracle in reference structure (torch CPU fp32, %d threads of %d "
                      "host CPUs; thread sweep at 2 dialogs: %s)" % (Bc, Bc * 10, threads, os.cpu_count() or 1,
                                                                     {k: round(v, 1) for k, v in table.items()})}


def resident_corpus_arm(args, p, eng, model, timed, rank, world):
    from visdial_b200.dataloader import Dataloader
    from visdial_b200.synthetic import make_corpus
    raw = make_corpus(p, num_threads=args.corpus_dialogs, num_opt_list=8000, seed=99 + rank)
    dl = Dataloader(eng, seed=7 + rank).initialize(dict(p, imgNorm=0, maxHistoryLen=60), ["train"], {"train": raw})
    del raw
    for _ in range(2):
        model.trainIteration(dl)
    ms_res, wall_res, _ = timed(dl, args.steps, 0)
    nb = 200
    eng.synchronize()
    eng.profile_reset()
    eng.profile(1)
    by = 0
    t_host = time.perf_counter()
    for _ in range(nb):
        dl.getTrainBatch(p)
        by += dl.corpus["train"].batch_bytes()[0]
    t_host = (time.perf_counter() - t_host) / nb
    eng.synchronize()
    st = eng.kernel_stats("corpus_gather")
    eng.profile(False)
    nl = dl.corpus["train"].batch_bytes()[1]
    dl.close()
    return {"ms": max(ms_res, wall_res), "asm_us": st["ms"] / nb * 1e3, "bytes": by / nb, "launches": nl, "host_us": t_host * 1e6}


def resident_line(resident, rounds, peaks, args):
    gbs = resident["bytes"] / (resident["asm_us"] * 1e-6) / 1e9
    return {"value": rounds / (resident["ms"] * 1e-3), "unit": "QA-rounds/s", "h2d_bytes_per_step": 4 * CONFIGS[args.config]["batch"],
            "d2h_bytes_per_step": 4,
            "what": "Model.trainIteration fed by visdial_b200.dataloader.Dataloader (corpus of %d dialogs resident in HBM, batch "
                    "gathered + trimmed on the device)" % args.corpus_dialogs,
            "batch_assembly": {"device_us_per_batch": resident["asm_us"], "host_us_per_call": resident["host_us"],
                               "kernel_launches": resident["launches"], "algorithmic_bytes": resident["bytes"], "GB/s": gbs,
                               "frac_of_hbm_peak": gbs / peaks["hbm"], "bound": "hbm"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C4", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="dialogs per GPU (0 = the config's: 32 for C2-C4, 4 for C1)")
    ap.add_argument("--math", default="f16", choices=["f16", "tf32", "fp32"])
    ap.add_argument("--cpu-batch", type=int, default=8, help="dialogs of the bounded cpu_baseline sample in the GPU arm's line")
    ap.add_argument("--ref-batch", type=int, default=0, help="dialogs per reference step (0 = the GPU arm's batch if the run fits --ref-budget-s, else 8)")
    ap.add_argument("--ref-budget-s", type=float, default=900.0, help="time budget of the whole --impl reference run")
    ap.add_argument("--cpu-threads", type=int, default=0, help="0 = pick by a sweep over 8/16/32/64/128 threads")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-batched", action="store_true", help="reference arm: skip the batched-CPU figure")
    ap.add_argument("--no-rank-check", action="store_true")
    ap.add_argument("--resident", action="store_true", help="also time the HBM-resident-corpus arm (e2e_resident_corpus)")
    ap.add_argument("--no-resident", action="store_true", help=argparse.SUPPRESS)      # accepted for old command lines
    ap.add_argument("--corpus-dialogs", type=int, default=256, help="dialogs in the synthetic resident corpus per rank")
    ap.add_argument("--ncu-range", action="store_true", help="bracket the timed steps with cudaProfilerStart/Stop")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (training: loss, and a "
                    "seeded sample of the weights and gradients after it; C5: the ranks of each batch size) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return
    rank, local, world = dist_setup(args.gpus)
    try:
        run_ours(args, rank, local, world)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
