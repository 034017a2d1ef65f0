#!/usr/bin/env python
"""Benchmark: Dreamer-V3 train-steps/sec (BASELINE.json metric) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
    python bench.py --impl reference --steps K --warmup W    # reference algorithm on the host cores (oracle port)
    python bench.py --steps K --dump-outputs DIR             # also write the outputs of the last timed step (.npy)

One "step" = one call of the Dreamer-V3 update (`train()`, reference dreamer_v3.py:48-357) on one per-rank
replay batch of the BASELINE config: size S, B=16, T=64, 64x64x3 uint8 observations, horizon 15, discrete A=2.
Prints ONE JSON line (see the task contract): `value` = device-resident throughput (CUDA-graph replay of the
step, inputs in HBM), `e2e` = the same metric through the public `train()` call with pinned-host inputs
(H2D copy + metric D2H inside the timed region), `roofline` for the dominant kernel family measured live with
CUDA events, `cpu_baseline` = the oracle port of the reference on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "train-steps/s"


def metric_name(args):
    return f"Dreamer-V3 train-steps/sec ({args.size}, bs{args.batch} seq{args.seq} horizon{args.horizon}, 64x64x3 obs)"


def workload_name(args):
    which = {"S": "BASELINE.json configs[1]", "XL": "BASELINE.json configs[4]"}.get(args.size, "")
    return f"dreamer_v3_{args.size} bs{args.batch} seq{args.seq} h{args.horizon} 64x64x3 discreteA2 ({which})"


def workload_config(args):
    """identical in both arms (`--impl b200` / `--impl reference`)"""
    return {"workload": workload_name(args), "size": args.size, "per_rank_batch": args.batch, "seq_len": args.seq,
            "horizon": args.horizon,
            "l2": "per-step working set (activations + optimiser state, GBs) >> 126 MB L2: no flush needed between steps"}


def make_cfg(args, **over):
    from sheeprl_b200.configs import make_dv3_cfg

    kw = dict(per_rank_batch_size=args.batch, per_rank_sequence_length=args.seq, horizon=args.horizon)
    kw.update(over)
    return make_dv3_cfg(args.size, **kw)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.thr = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])

        self.thr = threading.Thread(target=pump, daemon=True)
        self.thr.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.thr.join(timeout=2)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def synthetic_batch(cfg, adim, seed, device=None, pinned=False):
    """SURVEY.md §8d synthetic replay batch (uint8 pixels, one-hot actions, N(0,1) rewards...)."""
    import torch

    g = torch.Generator().manual_seed(seed)
    T, B, sz = cfg.algo.per_rank_sequence_length, cfg.algo.per_rank_batch_size, cfg.env.screen_size
    d = {
        "rgb": torch.randint(0, 256, (T, B, 3, sz, sz), generator=g, dtype=torch.uint8),
        "actions": torch.nn.functional.one_hot(torch.randint(0, adim[0], (T, B), generator=g), adim[0]).float(),
        "rewards": torch.randn(T, B, 1, generator=g),
        "terminated": (torch.rand(T, B, 1, generator=g) < 0.01).float(),
        "truncated": torch.zeros(T, B, 1),
        "is_first": (torch.rand(T, B, 1, generator=g) < 0.02).float(),
    }
    if pinned:
        d = {k: v.pin_memory() for k, v in d.items()}
    if device is not None:
        d = {k: v.to(device) for k, v in d.items()}
    return d


DUMP_CAP = 1 << 21      # elements per dumped array; a larger parameter group is dumped as a fixed, seeded sample


def dump_outputs(eng, directory):
    """Writes what a caller of train() holds after the step: the 13 logged metrics (in METRIC_ORDER), the Moments
    (low, high) and the four parameter groups, as float32 `.npy` files (at most 8 MB per group)."""
    import numpy as np
    import torch

    from sheeprl_b200.algos.dreamer_v3.dreamer_v3 import METRIC_ORDER

    md = eng.metrics_dict()
    out = {"metrics": torch.stack([md[k] for k in METRIC_ORDER]), "moments": eng.moments_state}
    for name, group in (("world_model", eng.wm), ("actor", eng.actor), ("critic", eng.critic), ("target_critic", eng.target)):
        flat = group.flat
        if flat.numel() > DUMP_CAP:
            g = torch.Generator().manual_seed(0)
            idx = torch.randint(0, flat.numel(), (DUMP_CAP,), generator=g).sort().values
            flat = flat[idx.to(flat.device)]
        out[name] = flat
    os.makedirs(directory, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())


# ---------------------------------------------------------------------------------------------------------
# per-op instrumentation (roofline): CUDA events around every C-ABI call of one eager step
# ---------------------------------------------------------------------------------------------------------
class ProfilingOps:
    """Wraps CudaOps; brackets every op with CUDA events on the launching stream and accounts its
    algorithmic FLOPs / bytes (DESIGN.md lists the per-op formulas)."""

    def __init__(self, inner):
        import torch

        self._inner, self._torch = inner, torch
        self.records = []

    def __getattr__(self, name):
        fn = getattr(self._inner, name)
        if not callable(fn):
            return fn
        torch = self._torch

        def wrapped(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            self.records.append((name, e0, e1, self._work(name, a, k)))
            return r

        return wrapped

    @staticmethod
    def _nbytes(*ts):
        return sum(t.numel() * t.element_size() for t in ts if t is not None and hasattr(t, "numel"))

    def _work(self, name, a, k):
        """(flops, bytes) algorithmic work of one call."""
        if name == "gemm":
            A, B, C, tA, tB = a[:5]
            M, N = C.shape
            K = A.shape[0] if tA else A.shape[1]
            return 2.0 * M * N * K, 4.0 * (M * K + K * N + M * N)
        if name in ("conv_down", "conv_up"):
            big, small = (a[0], a[2]) if name == "conv_down" else (a[2], a[0])
            NB, h, w, Cs = small.shape
            Cb = big.shape[-1]
            return 2.0 * NB * h * w * Cs * Cb * 16, 4.0 * (big.numel() + small.numel() + Cs * Cb * 16)
        if name == "conv_wgrad":
            small, big = a[0], a[1]
            NB, h, w, Cs = small.shape
            return 2.0 * NB * h * w * Cs * big.shape[-1] * 16, 4.0 * (big.numel() + small.numel())
        return 0.0, float(self._nbytes(*[x for x in a if hasattr(x, "numel")]))

    def summary(self):
        self._torch.cuda.synchronize()
        agg = {}
        for name, e0, e1, (fl, by) in self.records:
            t = e0.elapsed_time(e1)
            s = agg.setdefault(name, [0.0, 0.0, 0.0, 0])
            s[0] += t
            s[1] += fl
            s[2] += by
            s[3] += 1
        return agg


def run_b200(args):
    import torch
    import torch.distributed as dist

    # Native libraries write banners to fd 1 (NCCL prints "NCCL version ..." at communicator creation): keep stdout
    # for the ONE JSON line of the contract and send everything else to stderr until the result is ready.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    from sheeprl_b200.algos.dreamer_v3.agent import build_agent
    from sheeprl_b200.algos.dreamer_v3.dreamer_v3 import make_optimizers, train
    from sheeprl_b200.algos.dreamer_v3.utils import Moments
    from sheeprl_b200.parallel import init_process_group_from_env

    rank, local, world = init_process_group_from_env("nccl")
    assert world == args.gpus, f"WORLD_SIZE={world} but --gpus {args.gpus}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cfg = make_cfg(args)
    cfg.seed = 5
    cfg.algo.cuda_graph = not args.no_graph
    if args.no_overlap_allreduce or args.overlap_allreduce:
        cfg.algo.overlap_allreduce = bool(args.overlap_allreduce)
    adim = (2,)

    class Fab:  # the three attributes train()/build_agent() read from Fabric
        device, world_size, global_rank = dev, world, rank

    class Space:
        shape = (3, 64, 64)

    # the PUBLIC surface only: build_agent installs the data-parallel hooks when world_size > 1, train() captures the
    # update into a CUDA graph on its third call and replays it afterwards (sheeprl_b200/graph.py)
    wm, actor, critic, target, _ = build_agent(Fab, adim, False, cfg, {"rgb": Space})
    eng = wm._b200_engine
    opts = make_optimizers(eng, cfg)
    mo = cfg.algo.actor.moments
    moments = Moments(mo.decay, mo.max, mo.percentile.low, mo.percentile.high)

    class Agg:
        disabled = False

        def __init__(self):
            self.v = {}

        def update(self, k, v):
            self.v[k] = v

    agg = Agg()
    host = synthetic_batch(cfg, adim, seed=100 + rank, pinned=True)
    static = {k: v.to(dev) for k, v in host.items()}            # device-resident inputs for `value`
    in_bytes = sum(v.numel() * v.element_size() for v in host.values())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_public(data):
        eng.update_target(cfg.algo.critic.tau)                  # main() does this before each train() (:674-680)
        train(Fab, wm, actor, critic, target, *opts, data, agg, cfg, False, adim, moments)

    # ---- warm-up: W >= 3 public calls (the first two run eagerly, the third captures the graph)
    launches0 = eng.ops.launches
    step_public(static)
    launches_per_step = eng.ops.launches - launches0
    for _ in range(max(args.warmup, 3) - 1):
        step_public(static)
    barrier()
    graphed = eng.use_cuda_graph() and eng.step_graph().captured(static, eng.graph_key())

    # ---- per-op breakdown of ONE eager step (roofline evidence).  Every rank runs it: the step contains the
    # data-parallel collectives, so a rank-0-only step would leave the other ranks' NCCL queues one step short.
    breakdown = {}
    if args.breakdown:
        prof = ProfilingOps(eng.ops)
        eng.ops = prof                                          # not a CudaOps instance -> train() runs eagerly
        for m in (eng.reward_wm, eng.cont_wm, eng.actor_mlp, eng.critic_mlp, eng.target_mlp, eng.rew_img, eng.cont_img):
            m.eng = eng
        step_public(static)
        breakdown = prof.summary()
        eng.ops = prof._inner
        barrier()

    # ---- timed region 1: `value` (inputs resident in HBM; train() copies them into the graph's static inputs)
    clocks = ClockSampler(local)
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step_public(static)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs)
    # ---- timed region 2: `e2e`: the same public call with the batch in pinned HOST memory (H2D inside train()) and
    # a device->host read of the step's 13 metrics
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out_host = torch.empty(13, dtype=torch.float32).pin_memory()
    step_public(host)                                           # same signature as `static`: reuses the captured graph
    barrier()
    e2.record()
    for _ in range(args.steps):
        step_public(host)
        out_host[:10].copy_(eng.metrics[:10], non_blocking=True)
        out_host[10:].copy_(eng.norms, non_blocking=True)
        torch.cuda.current_stream().synchronize()               # D2H read of the step's losses
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    clk = clocks.stop()

    # ---- secondary: the same step with single-pass TF32 products (torch's float32_matmul_precision "high", the
    # reference's default on GPUs, configs/config.yaml:18).  NOT the headline: the 1e-4 parity contract is fp32.
    ms_tf32 = 0.0
    if args.tf32_also and hasattr(eng.ops, "set_matmul_precision"):
        eng.ops.set_matmul_precision("high")
        for _ in range(3):
            step_public(static)                                 # new graph key: two eager calls + capture
        e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e4.record()
        for _ in range(args.steps):
            step_public(static)
        e5.record()
        barrier()
        ms_tf32 = e4.elapsed_time(e5)
        eng.ops.set_matmul_precision("highest")

    t = torch.tensor([ms, ms_e2e, ms_tf32], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e, ms_tf32 = float(t[0]), float(t[1]), float(t[2])
    if rank != 0:
        return
    assert all(torch.isfinite(eng.metrics).tolist()), "non-finite metrics"
    value = world * args.steps / (ms / 1e3)
    e2e_v = world * args.steps / (ms_e2e / 1e3)
    hbm, tf, src = measured_peaks()
    # Dominant kernel: gemm_tc_kernel (tcgen05 3xTF32; serves every large Linear / conv forward, input-gradient
    # and weight-gradient product).  `achieved` = algorithmic FLOPs of its largest launch in the step (an MLP
    # GEMM over the imagined trajectories: M=(H+1)*T*B, N=dense_units, K=latent) / its mean launch duration, measured
    # here with CUDA events on the launching stream; operands exceed the 126 MB L2.
    tot_ms = sum(v[0] for v in breakdown.values()) or 1.0
    tc_ops = ("gemm", "gemm_ln_act", "gemm_ln_gru", "conv_down", "conv_up", "conv_wgrad")
    share = sum(breakdown[k][0] for k in tc_ops if k in breakdown) / tot_ms
    gm, gn, gk = (eng.H + 1) * eng.N, eng.du, eng.L
    ga = torch.randn(gm, gk, device=dev)
    gb = torch.randn(gn, gk, device=dev)
    gc = torch.empty(gm, gn, device=dev)
    for _ in range(3):
        eng.ops.gemm(ga, gb, gc, False, True)
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    g0.record()
    for _ in range(20):
        eng.ops.gemm(ga, gb, gc, False, True)
    g1.record()
    torch.cuda.synchronize()
    g_ms = g0.elapsed_time(g1) / 20
    g_tf = 2.0 * gm * gn * gk / (g_ms * 1e-3) / 1e12
    traffic, tsrc = None, None
    for name in ("r2_gemm_tc_traffic.json", "r1_gemm_tc_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath) and args.size == "S":
            traffic, tsrc = json.load(open(tpath)).get("dram_bytes_per_launch"), name
            break
    flops_step = {"S": 0.904e12, "XL": 37.6e12}.get(args.size) if (args.batch, args.seq, args.horizon) in ((16, 64, 15), (64, 64, 15)) else None
    roof = {"kernel": "gemm_tc_kernel<128> (tcgen05.mma kind::tf32, 3xTF32 split, TMA, TMEM)", "bound": "tensor",
            "achieved": g_tf, "peak": tf, "unit": "TFLOP/s", "frac": g_tf / tf, "traffic": traffic,
            "traffic_source": tsrc, "peak_source": f"{src} bf16 cuBLAS",
            "shape": {"M": gm, "N": gn, "K": gk}, "us_per_launch": g_ms * 1e3,
            "step_tflops": (flops_step * world / (ms / args.steps * 1e-3) / 1e12 / world) if flops_step else None,
            "step_frac_of_peak": (flops_step / (ms / args.steps * 1e-3) / 1e12 / tf) if flops_step else None,
            "note": "fp32-equivalent FLOP/s: every product costs 3 TF32 MMAs and TF32 runs at half the bf16 rate, so the "
                    f"scheme's ceiling is peak/6 = {tf / 6:.0f} TFLOP/s (frac of that: {g_tf / (tf / 6):.2f}); tensor-core "
                    f"ops (gemm+conv) take {share:.2f} of the eager step; step_tflops = SURVEY 8(d) algorithmic FLOPs per "
                    "train() call / measured step time"}
    cpu = cpu_baseline(args, steps=3, warmup=1) if (args.cpu_baseline and world == 1) else None
    eager = gpu_eager_baseline(args, dev) if (args.gpu_eager and world == 1) else None
    out = {
        "metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "arm": {"parallelism": f"dp{world}", "cuda_graph": bool(graphed), "api": "sheeprl_b200.algos.dreamer_v3: build_agent() + train()",
                "overlap_allreduce": bool(world > 1 and cfg.algo.get("overlap_allreduce", not eng.fused_scan))},
        "clocks": clk,
        "e2e": {"value": e2e_v, "unit": UNIT, "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": 13 * 4,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": roof,
        "cpu_baseline": cpu,
        "gpu_eager_baseline": eager,
        "matmul_precision_high": ({"value": world * args.steps / (ms_tf32 / 1e3), "unit": UNIT, "ms_per_step": ms_tf32 / args.steps,
                                   "note": "single-pass TF32 products (float32_matmul_precision=high, the reference's GPU default); "
                                           "informational, the headline `value` is fp32-accurate 3xTF32"} if ms_tf32 > 0 else None),
        "breakdown_ms": {k: round(v[0], 3) for k, v in sorted(breakdown.items(), key=lambda kv: -kv[1][0])[:12]},
    }
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(out), flush=True)


# ---------------------------------------------------------------------------------------------------------
# Baseline arms: the reference algorithm on the host cores / in torch eager on the same GPU.
# `kind: "reference"` = the UNMODIFIED reference train() (package installed into baseline/_ref by __graft_entry__.build(),
# imported through the stub harness oracle/ref_harness.py); `kind: "port"` = oracle/dv3_oracle.py when no reference tree is
# reachable.  Only these arms execute anything under oracle/.
# ---------------------------------------------------------------------------------------------------------
def reference_root():
    for p in (os.environ.get("SHEEPRL_REFERENCE_ROOT"), os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
        if p and os.path.isdir(os.path.join(p, "sheeprl")):
            return p
    return None


def _oracle_runner(cfg, adim, device="cpu"):
    import torch

    from oracle import dv3_oracle as O          # checker / baseline only — never on the product path

    dev = torch.device(device)
    wm, actor, critic, target = ({k: v.to(dev) for k, v in d.items()} for d in O.init_params(cfg, adim, seed=0))
    a, w = cfg.algo, cfg.algo.world_model
    opts = [O.AdamState(wm, w.optimizer.lr, w.optimizer.eps), O.AdamState(actor, a.actor.optimizer.lr, a.actor.optimizer.eps),
            O.AdamState(critic, a.critic.optimizer.lr, a.critic.optimizer.eps)]
    ms = {"low": torch.zeros((), device=dev), "high": torch.zeros((), device=dev)}
    data = {k: v.to(dev) for k, v in O.make_batch(cfg, adim, seed=1).items()}
    state = {"s": 0}

    def step():
        noise = O.draw_noise(a.per_rank_sequence_length, a.per_rank_batch_size, a.horizon, w.stochastic_size,
                             w.discrete_size, adim, seed=10 + state["s"])
        noise = {k: (v.to(dev) if torch.is_tensor(v) else [x.to(dev) for x in v]) for k, v in noise.items()}
        state["s"] += 1
        if dev.type == "cuda":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        O.dv3_train_step(cfg, wm, actor, critic, target, *opts, data, noise, ms, adim)
        if dev.type == "cuda":
            torch.cuda.synchronize()
        return time.perf_counter() - t0

    return step


def _reference_runner(cfg, adim, device="cpu"):
    """the executed reference: its own build_agent() + train() (dreamer_v3.py:48-357) with torch.optim.Adam"""
    import torch

    os.environ["SHEEPRL_REFERENCE_ROOT"] = reference_root()
    from oracle import ref_harness, ref_run     # baseline arm only

    ref_harness.install()
    from sheeprl.algos.dreamer_v3 import dreamer_v3 as D
    from sheeprl.algos.dreamer_v3.agent import build_agent
    from sheeprl.algos.dreamer_v3.utils import Moments

    dev = torch.device(device)
    fab = ref_harness.FakeFabric(dev)
    rcfg = ref_run.to_ref_cfg(cfg)
    torch.manual_seed(0)
    sz = cfg.env.screen_size
    wm, actor, critic, target, _ = build_agent(fab, tuple(adim), False, rcfg, {"rgb": ref_harness.Shape((3, sz, sz))})
    a = cfg.algo

    def adam(params, o):
        return torch.optim.Adam(params, lr=o.lr, eps=o.eps, weight_decay=o.weight_decay, betas=tuple(o.betas))

    wo, ao, co = adam(wm.parameters(), a.world_model.optimizer), adam(actor.parameters(), a.actor.optimizer), adam(critic.parameters(), a.critic.optimizer)
    mo = a.actor.moments
    moments = Moments(mo.decay, mo.max, mo.percentile.low, mo.percentile.high).to(dev)
    data = {k: v.to(dev).float() for k, v in synthetic_batch(cfg, adim, seed=1).items()}

    class Agg:                                   # keeps tensors, never synchronises (like torchmetrics' MeanMetric.update)
        disabled = False

        def update(self, k, v):
            self.last = v

    agg = Agg()

    def step():
        batch = {k: v.clone() for k, v in data.items()}
        if dev.type == "cuda":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        D.train(fab, wm, actor, critic, target, wo, ao, co, batch, agg, rcfg, False, tuple(adim), moments)
        if dev.type == "cuda":
            torch.cuda.synchronize()
        return time.perf_counter() - t0

    return step


def _runner(cfg, adim, device):
    if reference_root() is not None:
        try:
            return _reference_runner(cfg, adim, device), "reference"
        except Exception as e:  # harness could not import the reference on this host: fall back to the port, say so
            print(f"[bench] executed reference unavailable ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)
    return _oracle_runner(cfg, adim, device), "port"


def cpu_baseline(args, steps: int, warmup: int):
    """Reference train() on the host cores.  torch's intra-op pool is sized by a short probe on a 1/4-length workload
    (more threads than ~32 make the thousands of tiny RSSM ops slower, not faster; the reference itself defaults to
    num_threads=1, sheeprl/configs/config.yaml)."""
    import torch

    cores = os.cpu_count() or 1
    adim = (2,)
    best_k, best_t = None, None
    if args.size == "S":
        for k in [c for c in (8, 16, 32) if c <= cores] or [cores]:
            torch.set_num_threads(k)
            probe, _ = _runner(make_cfg(args, per_rank_sequence_length=max(8, args.seq // 4)), adim, "cpu")
            probe()
            t = probe()
            if best_t is None or t < best_t:
                best_k, best_t = k, t
    else:
        best_k = min(cores, 32)
    torch.set_num_threads(best_k)
    run, kind = _runner(make_cfg(args), adim, "cpu")
    times = [run() for _ in range(warmup + steps)]
    tt = times[warmup:]
    return {"value": len(tt) / sum(tt), "unit": UNIT, "cores": best_k, "kind": kind,
            "sample": f"{len(tt)} full train() step(s) of the same workload after {warmup} warm-up, torch fp32 CPU, "
                      f"{best_k} of {cores} host threads; s/step={sum(tt) / len(tt):.2f}; "
                      + ("the UNMODIFIED reference (baseline/_ref) through the stub-import harness" if kind == "reference"
                         else "oracle port of the reference (no reference tree on this host)")}


def gpu_eager_baseline(args, dev):
    """The same-box bar (BASELINE.md section 3, SURVEY 2.2): the reference train() in torch eager on THIS GPU, with
    float32_matmul_precision "high" (the reference's default, configs/config.yaml:18: TF32 products) and "highest"."""
    import torch

    adim = (2,)
    out = {"unit": UNIT}
    steps, warm = (10, 3) if args.size == "S" else (3, 2)
    for prec in ("high", "highest"):
        torch.set_float32_matmul_precision(prec)
        torch.backends.cudnn.allow_tf32 = prec != "highest"
        try:
            run, kind = _runner(make_cfg(args), adim, str(dev))
            times = [run() for _ in range(warm + steps)]
            tt = times[warm:]
            out[prec] = {"value": len(tt) / sum(tt), "ms_per_step": 1e3 * sum(tt) / len(tt), "steps": len(tt), "kind": kind}
        except Exception as e:
            out[prec] = {"error": f"{type(e).__name__}: {e}"[:300]}
        finally:
            torch.set_float32_matmul_precision("highest")
            torch.backends.cudnn.allow_tf32 = True
        torch.cuda.empty_cache()
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 30 if args.size == "S" else 2))
    warm = max(args.warmup, 3) if args.size == "S" else 1
    cb = cpu_baseline(args, steps=steps, warmup=warm)
    out = {
        "impl": "reference", "metric": metric_name(args), "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 / cb["value"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "arm": {"parallelism": "host cpu threads", "cuda_graph": False, "api": "sheeprl.algos.dreamer_v3: build_agent() + train()"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-graph", action="store_true", help="keep train() eager (cfg.algo.cuda_graph=False)")
    ap.add_argument("--size", default="S", choices=["S", "XL"], help="S = BASELINE configs[1]; XL = configs[4]")
    ap.add_argument("--batch", type=int, default=None, help="per-rank batch (default 16 for S, 64 for XL)")
    ap.add_argument("--seq", type=int, default=64)
    ap.add_argument("--horizon", type=int, default=15)
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-gpu-eager", dest="gpu_eager", action="store_false")
    ap.add_argument("--no-breakdown", dest="breakdown", action="store_false")
    ap.add_argument("--no-tf32", dest="tf32_also", action="store_false", help="skip the secondary single-pass-TF32 measurement")
    ap.add_argument("--no-overlap-allreduce", action="store_true", help="one all-reduce of the whole world-model gradient "
                    "before the optimizer instead of three overlapped buckets (the default when the persistent scan runs)")
    ap.add_argument("--overlap-allreduce", action="store_true", help="force the three overlapped bucket reductions")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of `value`, write what the last of them computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    if args.batch is None:
        args.batch = 16 if args.size == "S" else 64
    if args.size != "S" and "--cpu-baseline" not in sys.argv:
        args.cpu_baseline = False          # minutes per step on the host at XL: only the explicit reference arm times it
    if args.impl == "reference":
        run_reference(args)
    else:
        try:
            run_b200(args)
        finally:
            import gc

            import torch.distributed as dist

            from sheeprl_b200.graph import release_all

            # captured graphs hold NCCL kernels: they must be gone before the communicator is torn down, or
            # destroy_process_group() blocks (the engine sits in a reference cycle, so drop the graphs explicitly)
            release_all()
            gc.collect()
            if dist.is_available() and dist.is_initialized():
                dist.destroy_process_group()


if __name__ == "__main__":
    main()
