"""Headline benchmark: BEV queries/sec of the BEVFormer encoder hot path (bevformer_base, 200x200x256,
6 cameras, 4 levels, temporal self-attention with prev_bev), forward + backward, bf16.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle)
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write the last step's outputs to DIR

One "step" = one full encoder forward + backward (all layers, point sampling included, gradients for
every parameter, bev_query and the camera features) over one synthetic sample per GPU.  Rank 0
prints one JSON line (contract in the task statement): `value` with inputs resident in HBM, `e2e`
through the public plugin call with pinned HOST inputs copied in every step and the loss read back,
`roofline` for the dominant kernel (the SCA sampler backward) timed live with CUDA events,
`cpu_baseline` = the oracle restatement on the host cores over a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from bevformer_b200 import synthetic as syn  # noqa: E402
from bevformer_b200.dist import average_gradients_flat  # noqa: E402

METRIC = "BEV queries/sec (bevformer_base 200x200x256, 6 cams) fwd+bwd"
UNIT = "BEV queries/s"
WORKLOAD = "base"
# BASELINE.json configs[1..3] (parity-test cases; `--config tiny|small` prints their bench lines for
# BASELINE.md §5, the default and the driver's run stay on configs[3] = base)
CONFIGS = {
    "base": dict(workload="base", dtype="bf16", backward=True,
                 metric=METRIC),
    "small": dict(workload="small4", dtype="bf16", backward=True,
                  metric="BEV queries/sec (bevformer_small 150x150x256, 6 cams, 4 synthetic levels) fwd+bwd"),
    "tiny": dict(workload="tiny", dtype="f32", backward=False,
                 metric="BEV queries/sec (bevformer_tiny 50x50x256, 6 cams, 1 level) fwd"),
}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback"


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle restatement on the host cores, bounded sample
# ------------------------------------------------------------------------------------------------
def cpu_threads() -> int:
    """Threads for the CPU arm.  PyTorch's CPU kernels on this path stop scaling (and then regress)
    well before 128 threads (measured on the B200 host: 8 thr 1165 q/s, 16 thr 1539, 32 thr 1500, 64 thr 846,
    128 thr 196), so the arm uses min(host cores, BEVF_CPU_THREADS or 16) and reports that
    number as `cores`."""
    cap = int(os.environ.get("BEVF_CPU_THREADS", "16"))
    return max(1, min(os.cpu_count() or 1, cap))


def cpu_reference_step_factory(layers_in_sample=1, bev_div=1):
    """Returns (step_fn, queries_equivalent_per_step).  Sample = `layers_in_sample` of the 6 encoder
    layers, forward + backward, on the full base inputs (optionally a bev_div-times coarser BEV
    grid); reported q/s scales the sample time to all layers of the full grid."""
    from oracle import torch_ref
    w = syn.WORKLOADS[WORKLOAD]
    if bev_div > 1:
        import dataclasses
        w = dataclasses.replace(w, bev_h=w.bev_h // bev_div, bev_w=w.bev_w // bev_div)
    torch.set_num_threads(cpu_threads())
    sd = {k: v.requires_grad_(True) for k, v in syn.make_state_dict(w).items()}
    inp = syn.make_encoder_inputs(w, bs=1, seed=0)
    inp.bev_query.requires_grad_(True)
    inp.feat.requires_grad_(True)
    proj = torch.randn(1, w.num_query, w.embed_dims, generator=torch.Generator().manual_seed(11))

    def step():
        for t in list(sd.values()) + [inp.bev_query, inp.feat]:
            t.grad = None
        out = torch_ref.encoder_forward(sd, layers_in_sample, inp.bev_query, inp.feat,
                                        use_c_oracle=False, **inp.kwargs())
        (out * proj).sum().backward()

    frac = layers_in_sample / syn.WORKLOADS[WORKLOAD].num_layers
    return step, w.num_query * frac, w


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = cpu_threads()
    step, q_per_step, w = cpu_reference_step_factory(1, 1)
    t0 = time.perf_counter(); step(); first = time.perf_counter() - t0
    bev_div = 1
    if first * (args.steps + args.warmup) > 300.0:      # keep the whole run within a few minutes
        bev_div = 2 if first * (args.steps + args.warmup) < 1200.0 else 4
        step, q_per_step, w = cpu_reference_step_factory(1, bev_div)
    for _ in range(max(args.warmup - (1 if bev_div == 1 else 0), 0)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    value = q_per_step / dt
    sample = (f"1 of 6 encoder layers fwd+bwd on the base inputs, BEV grid {w.bev_h}x{w.bev_w}; "
              f"q/s = grid queries / (6 x sample time)")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": {"workload": "bevformer_base encoder (6 layers, 200x200 BEV, 6 cams, 4 levels), "
                               "reference CPU path = pure-PyTorch restatement of the reference modules "
                               "(grid_sample fallback), bounded sample"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampling
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        rows = [r for t, r in self.rows if self.t0 is None or (self.t0 <= t <= (self.t1 or t) + 0.05)]
        if len(rows) < 3:                       # very short timed region: fall back to every sample taken
            rows = [r for _, r in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------
def sca_alg_bytes(w, pairs, bwd):
    """SURVEY.md §8d compulsory bytes of the SCA sampler at bf16 storage, active pairs only."""
    c, m = w.embed_dims, w.num_heads
    lp = len(w.levels) * w.sca_points
    value = w.num_cams * w.num_value * c * 2
    la = pairs * m * lp * 12
    io = pairs * c * 2
    if not bwd:
        return value + la + io
    return value + la + io + w.num_cams * w.num_value * c * 4 + la


SEED = 0
DUMP_MAX_ELEMENTS = 1 << 21    # per array (8 MB of float32): at most 5 arrays, 40 MB in all


def dump_outputs(path, last):
    """--dump-outputs: writes what the last timed step handed its caller as <path>/<name>.npy in float32:
    the encoder output `out` and the `loss`, and with a backward pass the gradients of bev_query, of the
    camera features and of every parameter (`grad_params`: flattened, concatenated in named_parameters()
    order).  An array of more than DUMP_MAX_ELEMENTS elements is stored as that many of its elements,
    flattened, at fixed seeded positions (the same in every run), so that two builds of the project can be
    compared output for output."""
    torch.cuda.synchronize()
    arrays = {"out": last["out"], "loss": last["loss"]}
    if last["bev_query"].grad is not None:
        arrays.update(grad_bev_query=last["bev_query"].grad, grad_feat=last["feat"].grad,
                      grad_params=torch.cat([g.reshape(-1).float() for g in last["grads"]]))
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMENTS:
            pos = torch.randint(t.numel(), (DUMP_MAX_ELEMENTS,), generator=torch.Generator().manual_seed(0))
            t = t.reshape(-1)[pos.sort().values.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def run_ours(args):
    import torch.distributed as dist
    from bevformer_b200 import _lib, ops
    from bevformer_b200.plugin import build_transformer_layer_sequence

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # PyTorch seeds its generators at random in every process; the step draws from them (the loss
    # projection `proj`; the dropout keys derive from the CPU generator's seed, ops._next_seed).  A fixed
    # seed makes every run with the same arguments compute the same thing.
    torch.manual_seed(SEED)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this framework has no CPU path "
                         "(use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"

    lib = _lib.load()
    if args.dense is not None:
        _lib.check(lib.bevf_msda_set_dense_backward(args.dense), lib)
    elif os.environ.get("BEVF_MSDA_DENSE", "") == "2":
        _lib.check(lib.bevf_msda_set_dense_backward(2), lib)
    dense_mode = int(lib.bevf_msda_get_dense_backward())
    cfg = CONFIGS[args.config]
    w = syn.WORKLOADS[cfg["workload"]]
    dtype = torch.bfloat16 if cfg["dtype"] == "bf16" else torch.float32
    do_bwd = cfg["backward"]
    enc = build_transformer_layer_sequence(syn.encoder_cfg(w))
    enc.load_state_dict(syn.make_state_dict(w))
    enc = enc.to(dev, dtype)
    enc = enc.train() if do_bwd else enc.eval()   # training step: dropout active, as the configs set it
    model = enc
    use_graph = not args.no_graph
    if world > 1 and not use_graph:
        model = torch.nn.parallel.DistributedDataParallel(enc, device_ids=[local],
                                                          gradient_as_bucket_view=True)
    params = [p for p in enc.parameters()]
    # graph mode: all parameter gradients accumulate in one flat arena (one memset + one conversion per step
    # instead of ~150 small fills / casts); its bf16 result is also the all-reduce bucket
    arena = enc.enable_grad_arena(overlap=not args.no_overlap) if (use_graph and do_bwd and not args.no_arena) else None
    if arena is not None and world > 1:
        arena.defer_conversion = True

    def allreduce_grads():
        """Graph-replayed step: one flat-bucket NCCL all-reduce (eager mode uses torch DDP instead)."""
        if arena is not None:
            arena.all_reduce_mean(world)              # fp32 average of the flat accumulator, then one conversion
        else:
            average_gradients_flat(params, world)
    # one synthetic sample per GPU (weak scaling), different per rank
    host = syn.make_encoder_inputs(w, bs=1, seed=rank)
    pin = {k: getattr(host, k).to(dtype).pin_memory()
           for k in ("bev_query", "feat", "bev_pos", "prev_bev")}
    # the camera rig of the frame: every step reads its projection matrices from HERE (device buffer,
    # refreshed from pinned host memory in the e2e loop), runs point sampling and builds the in-view pair
    # list on the device -- nothing of the step is prepared outside the timed region
    pin_l2i = torch.as_tensor(np.asarray([m["lidar2img"] for m in host.img_metas], dtype=np.float32)).pin_memory()
    l2i_dev = pin_l2i.to(dev)
    h2d_bytes = sum(t.numel() * t.element_size() for t in pin.values()) + pin_l2i.numel() * 4
    dev_in = {k: t.to(dev) for k, t in pin.items()}
    shift = host.shift.to(dev)
    ss, lsi = host.spatial_shapes.to(dev), host.level_start_index.to(dev)
    proj = torch.randn(1, w.num_query, w.embed_dims, device=dev, dtype=dtype)
    last = {}     # tensors the most recent step handed its caller (--dump-outputs); detached, so that no
                  # step's autograd graph outlives it

    def step(inputs):
        bq = inputs["bev_query"].requires_grad_(do_bwd)
        ft = inputs["feat"].requires_grad_(do_bwd)
        for p in enc.parameters():
            p.grad = None
        with torch.set_grad_enabled(do_bwd):
            out = model(bq, ft, ft, bev_h=w.bev_h, bev_w=w.bev_w, bev_pos=inputs["bev_pos"],
                        spatial_shapes=ss, level_start_index=lsi, prev_bev=inputs["prev_bev"],
                        shift=shift, img_metas=host.img_metas, lidar2img=l2i_dev)
            loss = (out * proj).sum()
        if do_bwd:
            loss.backward()
        last.update(out=out.detach(), loss=loss.detach(), bev_query=bq, feat=ft,
                    grads=[p.grad for p in enc.parameters()])
        return loss

    def step_resident():
        return step({k: v.detach() for k, v in dev_in.items()})

    # ---- CUDA-graph mode: the whole step -- point sampling, the device-side pair list, all layers
    # forward + backward -- is captured once and replayed; the host then issues one launch per step instead
    # of ~600.  The graph is frame-valid: a replay reads the current contents of l2i_dev (a new camera rig
    # just changes the pair list the graph builds; tests/test_plan_gpu.py replays one graph with two rigs).
    graph, graph_outputs = None, last
    if use_graph:
        static_in = {k: v.clone() for k, v in dev_in.items()}
        static_in["bev_query"].requires_grad_(do_bwd)
        static_in["feat"].requires_grad_(do_bwd)

        def graph_body():
            with torch.set_grad_enabled(do_bwd):
                out = enc(static_in["bev_query"], static_in["feat"], static_in["feat"], bev_h=w.bev_h,
                          bev_w=w.bev_w, bev_pos=static_in["bev_pos"], spatial_shapes=ss,
                          level_start_index=lsi, prev_bev=static_in["prev_bev"], shift=shift,
                          img_metas=host.img_metas, lidar2img=l2i_dev)
                loss = (out * proj).sum()
            if do_bwd:
                loss.backward()
            last.update(out=out.detach(), loss=loss.detach(), bev_query=static_in["bev_query"], feat=static_in["feat"],
                        grads=[p.grad for p in enc.parameters()])
            return loss

        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(3):
                for t in list(enc.parameters()) + [static_in["bev_query"], static_in["feat"]]:
                    t.grad = None
                graph_body()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        for t in list(enc.parameters()) + [static_in["bev_query"], static_in["feat"]]:
            t.grad = None
        def capture(with_timers):
            for t in list(enc.parameters()) + [static_in["bev_query"], static_in["feat"]]:
                t.grad = None
            ops.KERNEL_TIMERS.clear()
            if with_timers:
                ops.KERNEL_TIMERS["msda_rows_backward"] = []
                ops.KERNEL_TIMERS["msda_rows_forward"] = []
            g = torch.cuda.CUDAGraph()
            before = _lib.launch_count()
            with torch.cuda.graph(g):
                loss = graph_body()
            timers = {k: list(v) for k, v in ops.KERNEL_TIMERS.items()}
            ops.KERNEL_TIMERS.clear()
            return g, loss, _lib.launch_count() - before, timers

        try:
            graph, static_loss, launches_per_replay, graph_timers = capture(True)
            graph.replay()
            torch.cuda.synchronize()
            _ = [a.elapsed_time(b) for a, b, _t in graph_timers["msda_rows_backward"]]
        except Exception:  # noqa: BLE001 - event nodes unsupported here: capture again without them
            torch.cuda.synchronize()
            graph, static_loss, launches_per_replay, graph_timers = capture(False)
        graph_outputs = dict(last)               # the graph's static tensors: every replay rewrites them

        def step_resident():                       # noqa: F811 - graph replay replaces the eager step
            graph.replay()
            if world > 1:
                allreduce_grads()
            return static_loss

    # e2e: every step copies its inputs from pinned host memory and reads the loss back.  The copy of
    # step i+1's inputs is issued on a side stream while step i computes (what a training input
    # pipeline does); two device buffer sets alternate.
    copy_stream = torch.cuda.Stream(dev)
    bufs = [{k: torch.empty_like(t, device=dev) for k, t in pin.items()} for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    state = {"i": 0, "primed": False}

    l2i_bufs = [torch.empty_like(l2i_dev), torch.empty_like(l2i_dev)]

    def issue_copy(slot):
        copy_stream.wait_stream(torch.cuda.current_stream(dev))      # the buffers' previous use is done
        with torch.cuda.stream(copy_stream):
            for k, t in pin.items():
                bufs[slot][k].copy_(t, non_blocking=True)
            l2i_bufs[slot].copy_(pin_l2i, non_blocking=True)         # this frame's projection matrices
            ready[slot].record(copy_stream)

    def step_e2e():
        if not state["primed"]:
            issue_copy(0)
            state["primed"] = True
        cur = state["i"] % 2
        issue_copy(1 - cur)                                          # next step's inputs, overlapped
        torch.cuda.current_stream(dev).wait_event(ready[cur])
        with torch.no_grad():
            l2i_dev.copy_(l2i_bufs[cur])
        if graph is not None:
            with torch.no_grad():                                    # staged inputs -> the graph's buffers
                for k in static_in:
                    static_in[k].copy_(bufs[cur][k])
            graph.replay()
            if world > 1:
                allreduce_grads()
            loss = static_loss
        else:
            loss = step({k: v.detach() for k, v in bufs[cur].items()})
        state["i"] += 1
        return float(loss.detach())   # device -> host read of the step's result

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    flush_l2 = args.config != "base"     # tiny / small: the step's working set can sit in the 126 MB L2
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if flush_l2 else None

    def timed(fn, steps):
        """K steps bracketed by barrier+synchronize, CUDA events on the launching stream; ms/step
        as the max over ranks.  With flush_l2 every step is bracketed on its own and a 256 MB buffer is
        written between steps (outside the brackets)."""
        barrier()
        if flush_l2:
            evs = [(torch.cuda.Event(True), torch.cuda.Event(True)) for _ in range(steps)]
            for a, b in evs:
                flush_buf.zero_()
                a.record(); fn(); b.record()
            barrier()
            ms = torch.tensor([sum(a.elapsed_time(b) for a, b in evs) / steps], device=dev)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return float(ms)
        s, e = torch.cuda.Event(True), torch.cuda.Event(True)
        s.record()
        for _ in range(steps):
            fn()
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e) / steps], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    def read_timers(timers):
        """elapsed ms of the SCA launches only (tag = (rows, levels): SCA samples 4 levels over the
        pair list, the interleaved TSA one level over 2*Nq rows)."""
        return {k: [a.elapsed_time(b) for a, b, tag in v if tag is None or tag[1] == len(w.levels)]
                for k, v in timers.items()}

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_resident()
    sampler.mark_begin()
    if graph is None:
        ops.KERNEL_TIMERS["msda_rows_backward"] = []
        ops.KERNEL_TIMERS["msda_rows_forward"] = []
    launches0 = _lib.launch_count()
    ms = timed(step_resident, args.steps)
    launches = _lib.launch_count() - launches0
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    if graph is None:
        kt = read_timers(ops.KERNEL_TIMERS)
        timer_note = "CUDA events around every launch of the kernel inside the timed region"
    else:
        # the event pairs were captured as nodes of the graph: after the timed replays they hold the
        # kernel's duration in the LAST timed step (one sample per launch site)
        launches = launches_per_replay * args.steps
        try:
            kt = read_timers(graph_timers)
            timer_note = ("CUDA event nodes captured around each launch site in the step's CUDA graph; "
                          "values are from the last timed replay")
        except Exception as exc:  # noqa: BLE001
            kt, timer_note = {}, f"event nodes could not be read ({exc})"
        if not kt.get("msda_rows_backward"):
            ops.KERNEL_TIMERS["msda_rows_backward"] = []
            ops.KERNEL_TIMERS["msda_rows_forward"] = []
            for _ in range(3):
                step({k: v.detach() for k, v in dev_in.items()})
            torch.cuda.synchronize()
            kt = read_timers(ops.KERNEL_TIMERS)
            timer_note = ("CUDA events around each launch in 3 eager replays of the same step, run right "
                          "after the timed graph replays (kernels inside a CUDA graph cannot be bracketed)")
    ops.KERNEL_TIMERS.clear()

    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, graph_outputs)

    if args.breakdown and rank == 0:
        # development aid, after both timed loops: CUPTI kernel records of 3 more replays of the same step
        # (warm caches, real overlap with the side stream) grouped by kernel name
        import collections
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                step_resident()
            torch.cuda.synchronize()
        agg = collections.defaultdict(lambda: [0.0, 0])
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                a = agg[ev.name[:150]]
                a[0] += ev.device_time
                a[1] += 1
        rows = sorted(agg.items(), key=lambda kv: -kv[1][0])
        with open(args.breakdown, "w") as f:
            f.write(f"sum of kernel durations per step: {sum(v[0] for _, v in rows) / 3e3:.3f} ms over "
                    f"{sum(v[1] for _, v in rows) // 3} launches (step wall time {ms:.3f} ms; side-stream "
                    f"kernels overlap)\n")
            for name, (us, n) in rows:
                f.write(f"{us / 3e3:8.3f} ms {n // 3:5d}x {us / n:8.1f} us  {name}\n")

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    total_q = w.num_query * world
    enc.check_plan()                                  # raises if any step overflowed the pair-list capacity
    pairs = enc.check_plan(enc.prepare(host.img_metas, w.bev_h, w.bev_w, dev, l2i_dev))   # in-view pairs of this rig
    peak, peak_src = measured_peaks()
    t_bwd = float(np.mean(kt["msda_rows_backward"])) if kt.get("msda_rows_backward") else None
    t_fwd = float(np.mean(kt["msda_rows_forward"])) if kt.get("msda_rows_forward") else None
    roof = None
    if t_bwd and args.config == "base":
        ab = sca_alg_bytes(w, pairs, True)
        kname = "msda_bwd_d32<bf16,bf16> (SCA sampler backward)"
        gv_f16 = os.environ.get("BEVF_GV_ACC", "f16") == "f16" and not dense_mode
        if gv_f16:
            kname = ("SCA sampler backward: bevf_abs_max + zero-fill of the accumulators + msda_bwd_d32<bf16,bf16> with mixed "
                     "accumulation (levels 0-1 scaled fp16, levels 2-3 fp32); timed as one op")
        if dense_mode:
            kname = ("SCA sampler backward = msda_bwd_dense_tc (grad_value of levels 1-3: coefficient scatter into UMMA slabs + "
                     "tcgen05.mma into TMEM bins" + (", on the library's second stream" if dense_mode == 2 else "") +
                     ") + msda_bwd_d32<bf16,bf16> (grad_loc, grad_attn, level-0 reductions); timed as one op")
        roof = {"bound": "hbm", "kernel": kname,
                "achieved": ab / t_bwd / 1e6, "peak": peak, "unit": "GB/s",
                "frac": ab / t_bwd / 1e6 / peak, "peak_source": peak_src,
                # dram__bytes_read.sum + dram__bytes_write.sum of this kernel, one launch, from the
                # `ncu --set full` capture named in traffic_source (ncu cannot run inside a bench run)
                "traffic": (329728512 + 179571712) if gv_f16 else (396693504 + 245205504),
                "traffic_source": (
                    "profiles/r2C_ncu_full_msda_bwd_mixed_raw.csv (msda_bwd_d32<bf16,bf16> with levels 0-1 accumulated in scaled fp16, "
                    "SCA real geometry: 119.5 M L2 reduction sectors instead of 163.3 M)" if gv_f16 else
                    "profiles/r1p_ncu_full_msda_bwd_raw.csv (msda_bwd_d32<bf16,bf16> with every level on the fp32 reduction path, "
                    "SCA real geometry)" + ("; the dense path moves the same compulsory bytes (value, grad_out, loc/attn read "
                                           "twice: +137 MB)" if dense_mode else "")),
                "dense_backward_mode": dense_mode,
                "in_view_pairs": pairs,
                "alg_bytes_per_launch": ab, "avg_launch_ms": t_bwd,
                "launches_timed": len(kt["msda_rows_backward"]), "timing": timer_note,
                "sca_forward": {"avg_launch_ms": t_fwd,
                                "achieved": sca_alg_bytes(w, pairs, False) / t_fwd / 1e6 if t_fwd else None}}
    standin = None
    if world == 1 and args.config == "base" and not args.no_standin:
        # the north-star's ">= 10x the reference CUDA op": mmcv's kernel cannot be built here, so the
        # yardstick is the reference's own grid_sample composition run on this B200 (fp32, as the
        # reference runs the op) -- tools/bench_standin.py; baseline leg, nothing of it is on the product path
        try:
            from tools import bench_standin
            torch.backends.cuda.matmul.allow_tf32 = True
            st = {}
            bench_standin.op_level(dev, st)
            bench_standin.encoder_level(dev, st, w.num_layers)
            standin = {"what": "reference arithmetic (grid_sample composition / restated modules, fp32, TF32 matmuls) "
                               "on the same B200 through PyTorch CUDA kernels; stands in for the mmcv CUDA op",
                       "msda_qps": st["msda_qps_standin_fp32"], "msda_qps_ours": st["msda_qps_ours_bf16"],
                       "msda_ratio": st["msda_ratio_ours_bf16_over_standin"],
                       "msda_ratio_fp32": st["msda_ratio_ours_fp32_over_standin"],
                       "encoder_qps": st["encoder_qps_standin_fp32"],
                       "encoder_ratio": total_q / (ms * 1e-3) / st["encoder_qps_standin_fp32"],
                       "detail_ms": {k: round(v, 4) for k, v in st.items() if k.endswith("_ms")}}
        except Exception as exc:  # noqa: BLE001
            standin = {"error": repr(exc)[:300]}
    cpu = None
    if world == 1 and not args.no_cpu_baseline and args.config == "base":
        cstep, q_per_step, _ = cpu_reference_step_factory(1, 1)
        cstep()                                       # warm-up
        t0 = time.perf_counter(); cstep(); cdt = time.perf_counter() - t0
        cpu = {"value": q_per_step / cdt, "unit": UNIT, "cores": cpu_threads(), "host_cores": os.cpu_count(),
               "kind": "port",
               "sample": "1 of 6 encoder layers fwd+bwd on the base inputs (fp32, pure-PyTorch "
                         "restatement of the reference modules, grid_sample fallback), 1 warm-up + 1 timed; "
                         "q/s = 40000 / (6 x sample time)"}
    lv = "x".join(f"{h}*{ww}" for h, ww in w.levels)
    line = {
        "metric": cfg["metric"], "value": total_q / (ms * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic",
        "config": {"workload": f"bevformer_{args.config} encoder: {w.num_layers} layers, {w.bev_h}x{w.bev_w} BEV queries, "
                               f"{w.num_cams} cams, {len(w.levels)} level(s) ({lv}), D=4 pillar points, TSA with prev_bev, "
                               + ("fwd+bwd, train mode (dropout 0.1)" if do_bwd else "forward only, eval mode")
                               + ", 1 sample per GPU; every step includes the pillar projection (point sampling) and the "
                                 "device-side construction of the in-view (camera, query) pair list"
                               + (", gradient all-reduce over NCCL (one flat bucket per step: the 19.8 MB fp32 accumulator of the gradient arena, averaged in fp32)" if world > 1 else ""),
                   "execution": ("whole step (point sampling + pair list + forward" + (" + backward" if do_bwd else "")
                                 + ") captured in one CUDA graph, replayed per step"
                                 if graph is not None else "eager launches"),
                   "l2": ("a 256 MB buffer is written between timed steps (each step bracketed by its own CUDA events)"
                          if flush_l2 else
                          "per-step working set (>1 GB of activations + 95 MB features) exceeds the 126 MB L2; no explicit flush"),
                   "gradients": ("flat fp32 gradient arena: one memset + one conversion per step (bevformer_b200/arena.py)"
                                 + ("" if args.no_overlap else "; weight-gradient GEMMs on a side stream, joined at the end of the backward pass")
                                 if arena is not None else "one fp32 buffer + conversion per parameter"),
                   "sampler_grad_value": (
                       "fp32 accumulation on every level (BEVF_GV_ACC=fp32)" if os.environ.get("BEVF_GV_ACC", "f16") != "f16"
                       else "scaled-fp16 accumulation (f16x2 vector reductions, scale from max|grad_out|) on the levels with <= "
                            + os.environ.get("BEVF_GV_MAXCONTRIB", "64") + " contributions per (pixel, head) on average -- TSA's BEV "
                            "maps, SCA levels 0-1 at base --, fp32 on the coarse levels; 3.0e-3 / 6.1e-3 of max|grad_value| against "
                            "the fp32 oracle on these launches (bar 1e-2; tests/test_msda_gpu.py)"),
                   "gemm_backend": ("cuBLASLt via torch (library GEMM; BEVF_GEMM=cublas)"
                                    if os.environ.get("BEVF_GEMM", "tc") == "cublas" else
                                    "hand-written tcgen05 kernels (csrc/gemm.cu): forward, dX and split-M dW")},
        "e2e": {"value": total_q / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
        "standin": standin,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-standin", action="store_true", help="skip the grid_sample-on-GPU stand-in leg")
    ap.add_argument("--breakdown", default=None, metavar="PATH",
                    help="after the timed loops, write a per-kernel table (CUPTI) of 3 more steps to PATH")
    ap.add_argument("--no-arena", action="store_true", help="per-parameter gradient buffers instead of the flat arena")
    ap.add_argument("--no-overlap", action="store_true", help="weight-gradient GEMMs on the main stream")
    ap.add_argument("--config", default="base", choices=sorted(CONFIGS),
                    help="BASELINE.json config to run (default: base = the headline metric)")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of a CUDA graph")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last step computed (output, loss, gradients; "
                         "large arrays as a fixed seeded sample) as DIR/<name>.npy")
    ap.add_argument("--dense", type=int, default=None, choices=[0, 1, 2],
                    help="SCA sampler backward: 0 = every level on the L2-reduction kernel, 1 = coarse levels through the "
                         "tensor-core kernel (csrc/msda_dense.cu) on the same stream, 2 = on the library's second stream "
                         "(default: the library's setting / BEVF_MSDA_DENSE)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
