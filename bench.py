#!/usr/bin/env python
"""Benchmark of the BEVBert hybrid-map encoder hot path (BASELINE.json metric: pre-train samples/s, R2R, bf16).

  python bench.py --gpus N --steps K --warmup W            # our sm_100a path (one process per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU cores (oracle port)

A "step" = one pre-training step of `GlocalTextPathCMTPreTraining` on one synthetic R2R batch (BASELINE config 2:
batch 32/GPU, 80-token instruction, 36 views x 768, 21x21 BEV, <=20 topological nodes): BEV lift-splat + forward +
backward (+ NCCL gradient all-reduce under DDP) + AdamW update, tasks cycling through the reference's
mlm:sap:masksem = 5:5:1 mix (scripts/pt_r2r.bash:4), dropout 0.1 everywhere as `set_dropout` leaves it
(pretrain_src/utils/misc.py:19-25).  Prints ONE JSON line on rank 0.
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

import torch  # noqa: E402

MIX = ["mlm", "sap"] * 5 + ["masksem"]          # scripts/pt_r2r.bash:4  --task_ratio mlm.5.sap.5.masksem.1
FLOPS_PER_SAMPLE_FWD_BWD = 130e9               # SURVEY.md 8(d): 5:5:1 mix, 43.4 GF forward x 3
# attention-GEMM subset of SURVEY.md 8(d) (projections + QK^T + PV + output projection, FFN excluded), forward, per sample at
# L=80, D^2=441, G=20, P=6: SAP 23.07 GF (the survey's figure), MLM 15.15 GF (language + panorama encoders, 4 + 4
# lang<-visn layers), MASKSEM 21.72 GF (SAP without the global branch); 5:5:1 mix = 19.35 GF forward, x3 with backward
ATTN_GEMM_FLOPS_MIX_FWD_BWD = 58.0e9


def host_cores():
    """CPU cores this process may actually use: scheduler affinity capped by the cgroup CPU quota
    (os.cpu_count() reports the whole host inside a container and oversubscribes the oracle's thread pool)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, int(q / per + 0.5)))
        except Exception:
            pass
    return max(1, min(n, int(os.environ.get("BEVBERT_CPU_THREADS", "64"))))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d.get("bf16_tflops"), "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
                "hbm_gbs": d.get("hbm_gbs"), "source": "MEASURED_PEAKS.json"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


WORKLOAD = "r2r"
WORKLOADS = {
    # BASELINE.json configs[1] (the headline): scripts/pt_r2r.bash:4 --task_ratio mlm.5.sap.5.masksem.1
    "r2r": dict(mix=["mlm", "sap"] * 5 + ["masksem"], model={}, synth={},
                name="R2R pre-train step, BASELINE configs[1]: batch 32/GPU, 80-token instruction, 36 views x 768, 21x21 BEV, "
                     "<=20 topo nodes"),
    # configs[3]: XLM-R vocabulary / positions (configs/rxr_model.json:20,30), 512-token instructions, same task mix
    # (scripts/pt_rxr.bash:4)
    "rxr": dict(mix=["mlm", "sap"] * 5 + ["masksem"], model=dict(vocab_size=250002, max_position_embeddings=514),
                synth=dict(txt_len=512, vocab_lo=1000, vocab_hi=250000, n_mask_tokens=77),
                name="RxR pre-train step, BASELINE configs[3]: XLM-R vocab 250002, 512-token instruction, 36 views x 768, "
                     "21x21 BEV, <=20 topo nodes"),
    # configs[4]: object tokens (configs/rvr_model.json obj_feat_size 768, rvr_pretrain.json max_objects 20),
    # scripts/pt_rvr.bash:4 --task_ratio mlm.1.mrc.1.sap.1.og.1
    "reverie": dict(mix=["mlm", "mrc", "sap", "og"], model=dict(obj_feat_size=768, obj_prob_size=1000,
                                                                 pretrain_tasks=["mlm", "mrc", "sap", "og"]),
                    synth=dict(obj_feat_size=768, obj_max=20, obj_prob_size=1000),
                    name="REVERIE pre-train step, BASELINE configs[4]: 36 pano views + <=20 object tokens x 768, object "
                         "grounding / region classification heads, 21x21 BEV"),
}


def full_config():
    from bevbert_b200.config import make_config
    # reference model config with the north_star's 768-d view features; dropout as set_dropout(model, 0.1) leaves it
    return make_config(hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, feat_dropout=0.1,
                       **WORKLOADS[WORKLOAD]["model"])


def synth_config(batch_size):
    from bevbert_b200 import synth
    return synth.SynthConfig(batch_size=batch_size, **WORKLOADS[WORKLOAD]["synth"])


# ====================================================================================== reference arm (CPU oracle)
def run_reference(args, rank):
    """The reference's algorithm on the host cores: oracle/bevbert_ref.py (validated line by line against the
    unmodified reference in the build container; /root/reference cannot travel to the GPU box)."""
    if rank != 0:
        return
    from bevbert_b200 import synth
    from bevbert_b200.model.pretrain_cmt import GlocalTextPathCMTPreTraining
    from oracle import bevbert_ref as R
    cores = host_cores()
    torch.set_num_threads(cores)
    cfg = full_config()
    model = synth.det_init_(GlocalTextPathCMTPreTraining(cfg), seed=3)
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in model.state_dict().items()}
    del model
    ocfg = R.OracleConfig(cfg, drop_p=0.1, feat_drop_p=0.1)
    Bs = args.ref_batch
    scfg = synth_config(Bs)
    batches = {t: synth.make_batch(scfg, seed=1234, task=t) for t in set(MIX)}

    def step(i):
        t = MIX[i % len(MIX)]
        for v in sd.values():
            v.grad = None
        loss = R.forward(sd, synth.clone_batch(batches[t]), t, ocfg)
        loss.mean().backward()
    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
    dt = time.perf_counter() - t0
    val = Bs * args.steps / dt
    sample = "%d steps of batch %d (R2R 21x21 BEV, mix cycling mlm,sap x5 + masksem), fwd+bwd, fp32, dropout 0.1" % (
        args.steps, Bs)
    print(json.dumps({
        "impl": "reference", "metric": "pretrain_samples_per_s", "value": val, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "R2R pre-train step (BASELINE configs[1] shapes, CPU batch %d)" % Bs, "global_batch": Bs},
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ====================================================================================== our arm
def bind_to_gpu_numa_node(local_rank):
    """Pin this rank (and therefore its pinned host buffers, first-touch) to the CPUs of the NUMA node its GPU hangs
    off: with 8 ranks x ~130 MB of H2D per step the copies otherwise cross the socket interconnect (round 1: e2e
    scaling 0.765 at N=8).  Best effort: returns the node or None."""
    try:
        props = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (getattr(props, "pci_domain_id", 0), props.pci_bus_id, props.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception:
        pass
    return None


def tensor_bytes(batch):
    return sum(v.numel() * v.element_size() for v in batch.values() if torch.is_tensor(v))


def pin_batch(batch):
    return {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in batch.items()}


DUMP_PER_PARAM = 4096       # sampled elements per parameter tensor: 1.2M in all on the R2R model (4.7 MB)


def dump_outputs(out_dir, loss, model, opt):
    """Writes what the last timed step computed as float32 .npy files under `out_dir`: its loss, the total gradient
    norm it clipped with (own AdamW only) and the parameters it left behind, sampled at fixed, seeded DUMP_PER_PARAM
    positions of every parameter (all of a smaller one) and concatenated in `named_parameters()` order.  fp32 atomics in
    the weight-gradient reductions make the step differ from run to run in the last bits, and the steps before it
    amplify that (B200 at 1000 W, R2R, --steps 22 --warmup 5: loss up to 1e-2, gradient norm 5e-2 and parameters
    3e-4 relative apart)."""
    import numpy as np
    params = [p for _, p in model.named_parameters()]
    idx = [torch.arange(p.numel()) if p.numel() <= DUMP_PER_PARAM else
           torch.randint(p.numel(), (DUMP_PER_PARAM,), generator=torch.Generator().manual_seed(i))
           for i, p in enumerate(params)]
    out = {"loss": loss.detach().reshape(-1),
           "params": torch.cat([p.detach().reshape(-1)[j.to(p.device)] for p, j in zip(params, idx)])}
    if not isinstance(opt, torch.optim.Optimizer):
        out["grad_norm"] = opt.total_grad_norm().reshape(-1)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from bevbert_b200 import kernels as K
    from bevbert_b200 import synth
    from bevbert_b200.model.pretrain_cmt import GlocalTextPathCMTPreTraining
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the hot path has no CPU implementation "
                           "(use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        # NCCL prints its version banner to the C-level stdout when the first communicator is created: route fd 1 to
        # stderr while the process group comes up so that stdout carries exactly one JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            import datetime
            dist.init_process_group("nccl", device_id=dev,
                                    timeout=datetime.timedelta(seconds=int(os.environ.get("BEVBERT_NCCL_TIMEOUT_S", "600"))))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    cfg = full_config()
    model = synth.det_init_(GlocalTextPathCMTPreTraining(cfg), seed=3).to(dev).train()
    net = model
    reduce_grads = None
    if world > 1:
        if args.ddp:        # the reference's wrapping (utils/misc.py:70); heavier on the host
            net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank], find_unused_parameters=True,
                                                            gradient_as_bucket_view=True)
        else:               # one flat NCCL all-reduce of the gradients per step (bevbert_b200/parallel.py)
            from bevbert_b200.parallel import FlatGradAllReduce, broadcast_parameters
            broadcast_parameters(model)
            reduce_grads = FlatGradAllReduce(model.parameters(), world)
    if not args.ddp:
        from bevbert_b200.parallel import direct_param_grads, enable_side_stream
        direct_param_grads(True)    # blocks assign p.grad themselves (no per-parameter AccumulateGrad nodes)
        if args.side_stream:
            enable_side_stream(True)    # weight-gradient GEMMs + bias column sums on a second stream
    if args.torch_optim:
        opt = torch.optim.AdamW(model.parameters(), lr=5e-5, weight_decay=0.01, fused=True)
    else:   # own multi-tensor AdamW + grad-norm clip kernel with the reference's update rule and hyper-parameters
        #         (optim/adamw.py:53-112, train_r2r.py:298 grad_norm 5.0, optim/misc.py no-decay groups); it also writes
        #         the bf16 weight shadows the next forward reads
        from bevbert_b200.optim import AdamW, build_param_groups
        opt = AdamW(build_param_groups(model, 0.01), lr=5e-5, betas=(0.9, 0.98), eps=1e-6, max_grad_norm=5.0,
                    runtime=model.rt)
    Bs = args.batch
    if args.strong:          # north_star's strong-scaling figure: the 32-sample global batch is split over the ranks
        if args.batch % world:
            raise SystemExit("--strong: --batch %d is not divisible by %d ranks" % (args.batch, world))
        Bs = args.batch // world
    scfg = synth_config(Bs)
    from bevbert_b200.model.ops import prepare_batch
    # prepare_batch = collate-time host index building (DataLoader-worker work in the reference's pipeline)
    host = {t: [prepare_batch(pin_batch(synth.make_batch(scfg, seed=1234 + 97 * rank + 13 * j, task=t))) for j in range(2)]
            for t in set(MIX)}
    resident = {t: [synth.batch_to(b, dev) for b in bs] for t, bs in host.items()}
    # end-to-end leg: the same batches in the 16-bit wire format (grid / view features as bf16 on the host, as they are
    # stored on disk; everything else unchanged) unless --wire fp32
    wire = torch.bfloat16 if args.wire == "bf16" else None
    host_e2e = host if wire is None else {t: [prepare_batch(b, wire_dtype=wire) for b in bs] for t, bs in host.items()}

    from bevbert_b200 import blocks as Bk

    def eager_step(batch, task):
        loss = net(batch, task).mean()
        loss.backward()
        if reduce_grads is None:
            Bk.join_side()           # side-stream mode: weight gradients landed (the reducer / optimizer also join)
        if reduce_grads is not None:
            reduce_grads()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss

    graphed = None
    if args.graphs and not args.ddp and not args.torch_optim:
        # whole-step CUDA-graph replay (bevbert_b200/graphs.py): one graph per (task, static batch buffers)
        from bevbert_b200.graphs import GraphedTrainStep
        graphed = GraphedTrainStep(net, opt, reduce_grads)
    train_step = graphed if graphed is not None else eager_step

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # The step loop allocates thousands of short-lived Python objects per step; like most production training loops
    # we keep the cyclic garbage collector out of the timed regions (reference counting still frees everything).
    import gc
    gc.collect()
    gc.freeze()
    gc.disable()

    # Setup, untimed: one step per resident (task, batch) pair so that every tensor shape of the cycle has been seen by
    # the caching allocator and the per-task gradient arenas are sized before the W warm-up steps start
    setup_reps = 4 if graphed is not None else 1      # graph mode: two eager steps, the capture and a first replay
    for t in sorted(set(MIX)):
        for j in range(2):
            for _ in range(setup_reps):
                train_step(resident[t][j], t)
    torch.cuda.synchronize()

    # ------------------------------------------------------------------ device-resident throughput ("value")
    for i in range(args.warmup):
        train_step(resident[MIX[i % len(MIX)]][i % 2], MIX[i % len(MIX)])
    sync_all()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    K.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    host_t0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        loss = train_step(resident[MIX[i % len(MIX)]][i % 2], MIX[i % len(MIX)])
    e1.record()
    host_enqueue_ms = (time.perf_counter() - host_t0) * 1e3 / args.steps     # host time to enqueue a step
    sync_all()
    ms = e0.elapsed_time(e1)
    launches = K.launch_count()          # kernels launched eagerly (host-counted) ...
    if graphed is not None:              # ... plus the kernels inside every replayed graph
        for i in range(args.steps):
            n = graphed.launches(resident[MIX[i % len(MIX)]][i % 2], MIX[i % len(MIX)])
            launches += n or 0
    clk = clocks.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    value = Bs * world * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, model, opt)

    # ------------------------------------------------------------------ end to end: pinned host -> device each step
    # Static device input buffers (one set per resident batch), filled from pinned host memory on a copy stream one
    # step ahead -- the reference's PrefetchLoader (data/loader.py:90-125) without per-step allocations.
    copy_stream = torch.cuda.Stream()
    dev_in = {(t, j): {k: (torch.empty(v.shape, dtype=v.dtype, device=dev) if torch.is_tensor(v) else v) for k, v in host_e2e[t][j].items()}
              for t in host_e2e for j in range(2)}
    last_use = {}

    def fetch(i):
        t, j = MIX[i % len(MIX)], i % 2
        with torch.cuda.stream(copy_stream):
            if (t, j) in last_use:
                copy_stream.wait_event(last_use[(t, j)])      # previous consumer of this buffer set has finished
            for k, v in host_e2e[t][j].items():
                if torch.is_tensor(v) and not os.environ.get("BENCH_E2E_NOCOPY"):      # (diagnosis switch)
                    dev_in[(t, j)][k].copy_(v, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(copy_stream)
        return dev_in[(t, j)], t, ev, (t, j)
    h2d = sum(tensor_bytes(host_e2e[MIX[i % len(MIX)]][i % 2]) for i in range(args.steps)) / args.steps
    loss_host = torch.zeros(args.steps, dtype=torch.float32).pin_memory()
    if graphed is not None:                          # untimed: capture the graphs of the static e2e input buffers
        for t in sorted(set(MIX)):
            for j in range(2):
                for k, v in host_e2e[t][j].items():
                    if torch.is_tensor(v):
                        dev_in[(t, j)][k].copy_(v, non_blocking=True)
                for _ in range(setup_reps):
                    train_step(dev_in[(t, j)], t)
        sync_all()
    for i in range(min(args.warmup, 3)):            # untimed: first use of the wire-format kernels / copy stream
        b, t, ev, key = fetch(i)
        torch.cuda.current_stream().wait_event(ev)
        train_step(b, t)
        done = torch.cuda.Event()
        done.record()
        last_use[key] = done
    sync_all()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    nxt = fetch(0)
    # every step's loss is read back into pinned host memory with an async copy on the compute stream (4 bytes per
    # step, inside the timed region); the values are consumed after the loop, so the host is never blocked on the GPU
    for i in range(args.steps):
        b, t, ev, key = nxt
        torch.cuda.current_stream().wait_event(ev)
        if i + 1 < args.steps:
            nxt = fetch(i + 1)
        loss = train_step(b, t)
        done = torch.cuda.Event()
        done.record()
        last_use[key] = done
        loss_host[i:i + 1].copy_(loss.detach().reshape(1), non_blocking=True)
    e3.record()
    sync_all()
    losses = loss_host.tolist()
    ms_e2e = e2.elapsed_time(e3)
    if world > 1:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t)
    e2e_value = Bs * world * args.steps / (ms_e2e * 1e-3)

    gc.enable()

    # ------------------------------------------------------------------ roofline of the dominant kernel (tcgen05 GEMM)
    peaks = load_peaks()
    roof = None
    if rank == 0 or world == 1:
        if reduce_grads is not None:
            reduce_grads.enabled = False     # rank-local pass: the overlapped reducer must not issue collectives
        had_side = K.side_stream() is not None
        if had_side:
            enable_side_stream(False)        # serialise the GEMMs: a launch's span must not include a concurrent one
        K.gemm_profile(True)
        try:
            for i in range(len(MIX)):
                loss = model(resident[MIX[i]][0], MIX[i]).mean()     # un-wrapped module: no collective in this pass
                loss.backward()
                Bk.join_side()
                Bk.PENDING_ADDS.clear()
                model.zero_grad(set_to_none=True)
            torch.cuda.synchronize()
        finally:
            K.gemm_profile(False)
            if had_side:
                enable_side_stream(True)
            if reduce_grads is not None:
                reduce_grads.enabled = True
        rec = [(2.0 * d[0] * d[1] * d[2] * d[3], ms_, d) for ms_, d in K.gemm_profile_records()]
        flops = sum(r[0] for r in rec)
        tms = sum(r[1] for r in rec)
        achieved = flops / (tms * 1e-3) / 1e12
        peak = peaks["bf16_tflops_sustained"] or peaks["bf16_tflops"]
        by_shape = {}
        for r in rec:
            d = by_shape.setdefault(r[2], [0, 0.0, 0.0])
            d[0] += 1
            d[1] += r[1]
            d[2] += r[0]
        top = sorted(by_shape.items(), key=lambda kv: -kv[1][1])[:14]
        shape_rows = [{"MNKb_amn_bmn": list(k), "launches": v[0], "ms": round(v[1], 3),
                       "tflops": round(v[2] / (v[1] * 1e-3) / 1e12, 1)} for k, v in top]
        if os.environ.get("BEVBERT_BENCH_VERBOSE"):      # every shape, to stderr (for profiles/)
            for k, v in sorted(by_shape.items(), key=lambda kv: -kv[1][1]):
                print("gemm-shape M,N,K,batch,a_mn,b_mn=%s launches=%d ms=%.3f tflops=%.1f" % (
                    list(k), v[0], v[1], v[2] / (v[1] * 1e-3) / 1e12), file=sys.stderr)
        roof = {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05, all %d launches of one 11-step mix cycle)" % len(rec),
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "peak_source": "%s bf16_tflops_sustained (kernel timed inside a long step)" % peaks["source"],
                # the timed region is short and runs at the maximum SM clock, so the burst figure is shown beside it
                "peak_burst": peaks["bf16_tflops"],
                "frac_of_burst_peak": (achieved / peaks["bf16_tflops"]) if peaks["bf16_tflops"] else None,
                "traffic": None, "gemm_ms_per_step": tms / len(MIX), "gemm_flops_per_step": flops / len(MIX),
                # the two model-level figures use SURVEY 8(d)'s flop counts of the R2R configuration
                "model_flops_frac": (value / world * FLOPS_PER_SAMPLE_FWD_BWD / 1e12 / peak) if WORKLOAD == "r2r" else None,
                # north_star "achieved fraction of the attention-GEMM roofline": attention-GEMM flops the job retires
                # per second (mix-weighted, fwd + bwd) over the bf16 peak
                "attn_gemm_roofline_frac": (value / world * ATTN_GEMM_FLOPS_MIX_FWD_BWD / 1e12 / peak)
                if WORKLOAD == "r2r" else None}

    # ------------------------------------------------------------------ CPU baseline (rank 0, N == 1, bounded sample)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import bevbert_ref as R
        cores = host_cores()
        torch.set_num_threads(cores)
        sd = {k: v.detach().float().cpu().clone().requires_grad_(True) for k, v in model.state_dict().items()}
        ocfg = R.OracleConfig(cfg, drop_p=0.1, feat_drop_p=0.1)
        cb = args.ref_batch
        cbatches = {t: synth.make_batch(synth_config(cb), seed=1234, task=t) for t in set(MIX)}
        per_task = {}
        for t in ("mlm", "sap", "masksem"):
            ts = []
            for it in range(2):                      # first iteration warms the allocator / threads
                for v in sd.values():
                    v.grad = None
                t0 = time.perf_counter()
                R.forward(sd, synth.clone_batch(cbatches[t]), t, ocfg).mean().backward()
                ts.append(time.perf_counter() - t0)
            per_task[t] = min(ts) / cb
        per_sample = (5 * per_task["mlm"] + 5 * per_task["sap"] + per_task["masksem"]) / 11.0
        cpu = {"value": 1.0 / per_sample, "unit": "samples/s", "cores": cores, "kind": "port",
               "sample": "oracle/bevbert_ref.py fwd+bwd, fp32, batch %d per task (best of 2), mix-weighted 5:5:1; "
                         "s/sample mlm %.3f sap %.3f masksem %.3f" % (cb, per_task["mlm"], per_task["sap"],
                                                                       per_task["masksem"])}

    if rank == 0:
        out = {
            "metric": "pretrain_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if args.strong else "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "%s; batch %d/GPU; lift-splat + fwd + bwd%s + grad-norm clip + AdamW (reference update "
                                   "rule); tasks cycle %s; dropout 0.1" % (
                                       WORKLOADS[WORKLOAD]["name"], Bs, " + NCCL grad all-reduce" if world > 1 else "",
                                       ",".join(MIX)),
                       "global_batch": Bs * world, "parallelism": "dp%d" % world,
                       "l2": "per-step inputs (%.0f MB) and saved activations exceed the 126 MB L2" % (h2d / 1e6)},
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                    "wire": "bf16 grid/view features, other inputs as collated" if wire is not None else "fp32 as collated",
                    "ms_per_step": ms_e2e / args.steps, "last_loss": losses[-1] if losses else None},
            "numa_node": numa, "gpu_launches": int(launches), "host_enqueue_ms_per_step": round(host_enqueue_ms, 3),
            "step_mode": "cuda-graph replay per (task, static batch)" if graphed is not None else "eager launches",
            "clocks": clk, "roofline": roof, "cpu_baseline": cpu,
        }
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=22)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="samples per GPU per step")
    ap.add_argument("--ref-batch", type=int, default=2, help="batch of the bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default="r2r", choices=sorted(WORKLOADS), help="workload: r2r = BASELINE configs[1] "
                    "(headline), rxr = configs[3], reverie = configs[4]")
    ap.add_argument("--side-stream", type=int, default=1, help="1: weight-gradient GEMMs on a second stream (default)")
    ap.add_argument("--graphs", type=int, default=1, help="1: replay each (task, batch) step as one CUDA graph (default); 0: eager launches")
    ap.add_argument("--torch-optim", action="store_true", help="torch.optim.AdamW(fused=True) instead of bevbert_b200.optim.AdamW")
    ap.add_argument("--wire", choices=("bf16", "fp32"), default="bf16",
                    help="host dtype of the large feature tensors in the end-to-end leg")
    ap.add_argument("--ddp", action="store_true", help="wrap with torch DDP instead of the flat gradient all-reduce")
    ap.add_argument("--strong", action="store_true",
                    help="strong scaling: --batch is the GLOBAL batch, split over the ranks (default: weak, --batch per GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last one's loss, gradient norm and a fixed sample of the "
                         "parameters it left behind to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3)
    # dropout masks derive from torch's seed (blocks.Runtime, graphs.GraphedTrainStep): fixed, so that runs with the
    # same arguments compute the same step
    torch.manual_seed(0)
    global WORKLOAD, MIX
    WORKLOAD = args.config
    MIX = list(WORKLOADS[WORKLOAD]["mix"])
    if WORKLOAD == "reverie":
        args.graphs = 0      # the object-token path sizes its tensors from device data (host sync): not capturable
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
