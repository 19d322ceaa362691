"""bench.py — image-text pairs/sec, forward+backward, VisualBERT-base (BASELINE.json metric).

    python bench.py --gpus 1 --steps 10 --warmup 3                    # this build (CUDA, sm_100a)
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1    # the reference's CPU arithmetic (oracle port)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --gpus 1 --steps 10 --warmup 3 --dump-outputs DIR  # + what the last timed step computed, as .npy

Workload at N=1: BASELINE.json configs[1] ("cfg2"): VisualBERT-base 12L/768H, COCO masked-LM pretrain step
(MLM + NSP heads), batch 256, 36 regions (2048-d) + 128 tokens, bf16, train mode (dropout active).
N>1: weak scaling — the same 256 pairs per GPU, one process per GPU, a single NCCL all-reduce of the flat
fp32 gradient buffer inside the timed step.
One step = zero grads -> forward -> loss.backward() (+ all-reduce); the optimizer is excluded on both the GPU
and the CPU side, as BASELINE.md §2 specifies for this metric.

Printed JSON (one line, rank 0): the driver contract plus
  roofline      dominant kernel family (gemm_tcgen05_kernel): algorithmic FLOPs / CUDA-event kernel time measured
                live inside the timed steps (vb_profile_*), against MEASURED_PEAKS.json bf16_tflops_sustained
  step_roofline the whole step: hot-path algorithmic FLOPs per pair (SURVEY.md §8d, heads excluded) x pairs/s
  cpu_baseline  the oracle (CPU restatement of the reference, oracle/vb_oracle.py) on a bounded sample
  e2e           same step through the public API with inputs in pinned HOST memory (H2D + loss D2H inside)
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

import numpy as np  # noqa: E402
import torch  # noqa: E402

from visualbert_b200 import synthetic  # noqa: E402

METRIC = "image-text pairs/sec fwd+bwd VisualBERT-base"
UNIT = "pairs/s"


def hot_path_flops_per_pair(c):
    """SURVEY.md §8d: F = 3 * [2 V Dv H + L (24 S H^2 + 4 S^2 H)] (encoder + visual projection, heads excluded)."""
    S = c["T"] + c["V"]
    H, L = c["hidden"], c["layers"]
    return 3.0 * (2.0 * c["V"] * c["Dv"] * H + L * (24.0 * S * H * H + 4.0 * S * S * H))


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(bf16_sustained=p.get("bf16_tflops_sustained", 1400.0), bf16_burst=p.get("bf16_tflops", 1590.0),
                    hbm=p.get("hbm_gbs", 6650.0), source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_sustained=1400.0, bf16_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def mark(self):
        """Start of the timed window: earlier samples (nvidia-smi spin-up during warm-up) are dropped."""
        self.t0 = time.time()

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        t0 = getattr(self, "t0", 0.0)
        for t, r in self.rows:
            if t < t0:
                continue
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def build_cfg(name, batch_override=None):
    c = dict(synthetic.CONFIGS[name])
    c["index"] = int(name[3:]) - 1
    c["B"] = c["B"] // c.pop("dp", 1)  # per-GPU batch: BASELINE.json quotes configs[2..4] as global batches over 8 GPUs
    if batch_override:
        c["B"] = batch_override
    return c


def cpu_oracle_step_time(c, sample_b, steps, warmup, threads=None):
    """Time the oracle (reference arithmetic, fp32, CPU) fwd+bwd on `sample_b` pairs of the same workload."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vb_oracle
    if threads:
        torch.set_num_threads(threads)
    cfg = synthetic.bert_config_dict(c["layers"], c["hidden"], c["heads"], c["inter"])
    sd = synthetic.init_state_dict(cfg, c["head"], c["Dv"], seed=0)
    sd = {k: v.requires_grad_(True) for k, v in sd.items()}
    batch = synthetic.make_batch(sample_b, c["T"], c["V"], c["Dv"], head=c["head"], seed=1234,
                                 nlvr_types=(c["head"] == "nlvr"))
    kw = {k: v for k, v in batch.items() if k != "position_embeddings_visual"}

    def step():
        for v in sd.values():
            v.grad = None
        out = vb_oracle.objective(sd, cfg, c["head"], **kw)
        out["loss"].backward()
        return out["loss"].item()

    for _ in range(warmup):
        step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    times.sort()
    dt = sum(times) / max(len(times), 1)
    spread = {"min_ms": 1e3 * times[0], "median_ms": 1e3 * times[len(times) // 2], "max_ms": 1e3 * times[-1], "steps": len(times)}
    return dt, torch.get_num_threads(), spread


def cpu_threads():
    """Threads for the CPU arm: one per physical core (the box exposes 2 hardware threads per core), set EXPLICITLY —
    under torch.distributed.run OMP_NUM_THREADS defaults to 1, which made the N>1 reference lines incomparable."""
    n = os.cpu_count() or 2
    return max(1, min(64, n // 2))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    c = build_cfg(args.config)
    sample_b = args.cpu_sample
    dt, threads, spread = cpu_oracle_step_time(c, sample_b, args.steps, args.warmup, threads=cpu_threads())
    value = sample_b / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic (seeded region features / token ids; random-init weights)",
        "config": {"workload": workload_name(c), "global_batch": sample_b,
                   "note": "reference arithmetic on host cores: oracle port of modeling.py (the Python reference itself "
                           "is not present on the GPU box); each step is a bounded sample of the workload"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "spread": spread,
                         "sample": f"{sample_b} pairs/step fwd+bwd, fp32, {os.cpu_count()} logical CPUs, {threads} torch threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, outputs, model):
    """Write what one step handed back as float32 .npy files under `out_dir`: every output tensor of the forward pass
    (`<key>.npy`, in full) and every parameter's gradient (`grad.<parameter name>.npy`), the latter at positions drawn
    from a fixed seed wherever a gradient is too large to fit its share of the 64 MB the whole dump may take."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in outputs.items()}
    named = [(n, p.grad.detach().reshape(-1)) for n, p in model.named_parameters() if p.grad is not None]
    header = 4096   # per file: the .npy header, with room to spare
    per_grad = ((DUMP_BYTES - sum(a.nbytes + header for a in arrays.values())) // len(named) - header) // 4
    gen = torch.Generator().manual_seed(0)
    for name, g in named:
        if g.numel() > per_grad:
            idx = torch.randint(g.numel(), (per_grad,), generator=gen).sort().values
            g = g[idx.to(g.device)]
        arrays["grad." + name] = g.float().cpu().numpy()
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    total = sum(os.path.getsize(os.path.join(out_dir, k + ".npy")) for k in arrays)
    assert total <= DUMP_BYTES, total
    return len(arrays), total


def workload_name(c):
    return (f"VisualBERT L{c['layers']}/H{c['hidden']} {c['head']} step, {c['V']} regions x {c['Dv']}-d + {c['T']} tokens "
            f"(BASELINE.json configs[{c.get('index', 1)}])")


def run_ours(args):
    import torch.distributed as dist
    from visualbert_b200 import BertConfig, TrainVisualBERTObjective, _lib
    from visualbert_b200.parallel import FlatGradSync

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this build has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    c = build_cfg(args.config, args.batch)
    B = c["B"]
    cfg = synthetic.bert_config_dict(c["layers"], c["hidden"], c["heads"], c["inter"])
    torch.manual_seed(0)
    model = TrainVisualBERTObjective(BertConfig.from_dict(cfg), c["head"], visual_embedding_dim=c["Dv"])
    model.bert.embeddings.special_intialize()
    model.to(dev).train()
    sync = FlatGradSync(model)
    opt = None
    if args.optimizer:  # parameter groups of the reference's wrapper (model_wrapper.py:100-111): no pooler, two decay groups
        from visualbert_b200 import BertAdam
        named = [(n, p) for n, p in model.named_parameters() if "pooler" not in n]
        nd = ("bias", "LayerNorm.bias", "LayerNorm.weight")
        opt = BertAdam([{"params": [p for n, p in named if not any(x in n for x in nd)], "weight_decay": 0.01},
                        {"params": [p for n, p in named if any(x in n for x in nd)], "weight_decay": 0.0}],
                       lr=1e-5, warmup=0.1, t_total=100000)

    host = synthetic.make_batch(B, c["T"], c["V"], c["Dv"], head=c["head"], seed=1234 + rank,
                                nlvr_types=(c["head"] == "nlvr"))
    host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in host.items()}
    from visualbert_b200.parallel import BatchPrefetcher
    pf = BatchPrefetcher(dev)  # also ships the indices of the MLM targets (found on the host): no host sync in forward
    resident = pf.take(pf.stage(host))
    torch.cuda.synchronize()
    h2d_bytes = sum(v.numel() * v.element_size() for v in resident.values() if torch.is_tensor(v))

    lscale = sync.loss_scale()   # 1 / world: the mean over ranks is folded into the loss, no divide pass over the buffer
    last = {}   # --dump-outputs: the output tensors of the latest step

    def step(batch):
        sync.zero()
        out = model(**batch)
        (out["loss"] * lscale if world > 1 else out["loss"]).backward()
        sync.allreduce(prescaled=True)
        if args.dump_outputs:
            # dict.items: the entries as stored; a lazy one the step never read (the MLM logits) is None, not computed
            last.clear()
            last.update((k, v) for k, v in dict.items(out) if torch.is_tensor(v))
        if opt is not None:
            opt.step()
        return out["loss"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    with ClockSampler(local) as clk:  # nvidia-smi needs ~0.5 s to start streaming: launch it before the warm-up
        for _ in range(max(args.warmup, 3)):
            step(resident)
        barrier()
        # ---- timed region: inputs resident in HBM (no per-launch events: they cost ~2 % of the step) ----
        n0 = _lib.launch_count()
        clk.mark()
        ms_total = timed(lambda: step(resident), args.steps)
        launches = _lib.launch_count() - n0
        if args.dump_outputs and rank == 0:   # before the passes below overwrite the gradients
            dumped = dump_outputs(args.dump_outputs, last, model)
        # ---- roofline pass: the SAME K steps again with a CUDA-event pair around every launch of the library ----
        _lib.profile_read()
        _lib.profile_enable(True)
        ms_profiled = timed(lambda: step(resident), args.steps) / args.steps
        prof = _lib.profile_read()
        _lib.profile_enable(False)
    ms_step = ms_total / args.steps
    value = world * B / (ms_step * 1e-3)

    # ---- end to end: host (pinned) inputs, H2D + loss D2H inside the timed region ----
    # every step copies ITS inputs from pinned host memory (BatchPrefetcher: on a copy stream, overlapping the previous
    # step) and reads ITS loss back (asynchronously into pinned memory; the value is consumed one step later, the way a
    # training loop logs it, so the host never drains the GPU queue). K input copies and K loss reads per K steps, all
    # inside the timed region.
    loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()

    diag = os.environ.get("VB_BENCH_E2E_DIAG", "")  # "nocopy" / "noloss": diagnostics only, never a reported number
    enq = [0.0, 0]

    def e2e_loop(steps):
        staged = pf.stage(host)                      # step 0's inputs: not overlapped with anything
        pending, seen = None, 0.0
        for i in range(steps):
            t0 = time.perf_counter()
            batch = pf.take(staged) if diag != "nocopy" else resident
            if i + 1 < steps and diag != "nocopy":
                staged = pf.stage(host)              # step i+1's inputs, in flight while step i computes
            loss = step(batch)
            enq[0] += time.perf_counter() - t0; enq[1] += 1
            if diag == "noloss":
                continue
            if pending is not None:
                pending.synchronize()                # step i-1's loss has long arrived
                seen += float(loss_host[(i - 1) & 1])
            loss_host[i & 1].copy_(loss.detach().float(), non_blocking=True)
            pending = torch.cuda.Event()
            pending.record()
        if pending is not None:
            pending.synchronize()
            seen += float(loss_host[(steps - 1) & 1])
        return seen

    e2e_loop(2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    e2e_loop(args.steps)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
    ms_e2e /= args.steps
    e2e_value = world * B / (ms_e2e * 1e-3)

    opt_info = None
    if opt is not None:  # the optimizer alone: K steps on the gradients left by the last backward
        n_params = sum(p.numel() for g in opt.param_groups for p in g["params"])
        for _ in range(2):
            opt.step()
        ms_opt = timed(opt.step, args.steps) / args.steps
        opt_bytes = 32.0 * n_params  # 4 (grad norm pass) + 28 (p, g, m, v read; p, m, v written) bytes per parameter
        opt_info = {"ms_per_step": ms_opt, "params": n_params, "launches_per_step": 2,
                    "roofline": {"bound": "hbm", "achieved": opt_bytes / (ms_opt * 1e-3) / 1e9, "unit": "GB/s",
                                 "bytes_per_param": 32}}

    # ---- the other BASELINE.json configs at their per-GPU batch (global batch / 8), same step, same all-reduce ----
    others = None
    had_opt = opt is not None
    if (world > 1 or args.other_configs) and args.config == "cfg2" and not args.batch:
        model = sync = opt = resident = pf = None   # release the cfg2 replica (weights, flat gradients, optimizer state)
        torch.cuda.empty_cache()
        others = {}
        for name in ("cfg3", "cfg4", "cfg5"):
            oc = build_cfg(name)
            ocfg = synthetic.bert_config_dict(oc["layers"], oc["hidden"], oc["heads"], oc["inter"])
            torch.manual_seed(0)
            m2 = TrainVisualBERTObjective(BertConfig.from_dict(ocfg), oc["head"], visual_embedding_dim=oc["Dv"])
            m2.bert.embeddings.special_intialize()
            m2.to(dev).train()
            s2 = FlatGradSync(m2)
            hb = synthetic.make_batch(oc["B"], oc["T"], oc["V"], oc["Dv"], head=oc["head"], seed=1234 + rank,
                                      nlvr_types=(oc["head"] == "nlvr"))
            pf2 = BatchPrefetcher(dev)
            res2 = pf2.take(pf2.stage({k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in hb.items()}))

            def step2():
                s2.zero()
                out = m2(**res2)
                (out["loss"] * lscale if world > 1 else out["loss"]).backward()
                s2.allreduce(prescaled=True)

            for _ in range(3):
                step2()
            k2 = max(3, min(args.steps, 10))
            ms2 = timed(step2, k2) / k2
            others[name] = {"workload": workload_name(oc), "per_gpu_batch": oc["B"], "global_batch": world * oc["B"],
                            "seq_len": oc["T"] + oc["V"], "ms_per_step": ms2, "value": world * oc["B"] / (ms2 * 1e-3), "unit": UNIT,
                            "step_roofline_frac": (oc["B"] / (ms2 * 1e-3)) * hot_path_flops_per_pair(oc) / 1e12 / load_peaks()["bf16_sustained"],
                            "steps": k2}
            del m2, s2, res2, pf2
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peaks = load_peaks()
    if opt_info is not None:
        opt_info["roofline"]["peak"] = peaks["hbm"]
        opt_info["roofline"]["frac"] = opt_info["roofline"]["achieved"] / peaks["hbm"]
    g = {k: sum(prof[c][k] for c in ("gemm_fwd", "gemm_dgrad", "gemm_wgrad")) for k in ("ms", "work", "launches")}
    gemm_tf = (g["work"] / (g["ms"] * 1e-3) / 1e12) if g["ms"] > 0 else 0.0
    F = hot_path_flops_per_pair(c)
    step_tf = (value / world) * F / 1e12
    kern_ms = {k: round(v["ms"] / args.steps, 3) for k, v in prof.items()}
    traffic, traffic_src = None, None
    for tname in ("r02b_traffic.json", "r02_traffic.json"):   # newest committed capture first
        tj = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", tname)
        if os.path.exists(tj) and args.config == "cfg2" and B == 256:  # the ncu capture is of this workload only
            tr = json.load(open(tj))
            traffic, traffic_src = tr["gemm_dram_bytes_per_launch_avg"], f"profiles/{tname} ({tr['source']})"
            break
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic (seeded region features / token ids; random-init weights; no network for COCO features or BERT checkpoints)",
        "config": {"workload": workload_name(c), "global_batch": world * B, "per_gpu_batch": B, "seq_len": c["T"] + c["V"],
                   "parallelism": f"dp{world}", "mode": "train (dropout 0.1 active)",
                   "step": "zero_grad + forward (MLM+NSP heads) + backward" + (" + 1 NCCL all-reduce (flat fp32 grads)" if world > 1 else "")
                           + ("; + fused BertAdam step (--optimizer; NOT the BASELINE metric)" if had_opt
                              else "; optimizer excluded (BASELINE.md §2)"),
                   "l2": "per-step working set (>12 GB of activations) is >> the 126 MB L2; no explicit flush needed"},
        "clocks": clk.summary(),
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "kernel": "gemm_tcgen05_2cta_kernel (all 12 GEMMs/layer fwd+dgrad+wgrad, projection, MLM decoder)",
                     "achieved": gemm_tf, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                     "frac": gemm_tf / peaks["bf16_sustained"], "traffic": traffic,
                     "traffic_note": ("NOT measured in this run: DRAM read+write bytes per GEMM launch from the committed ncu capture "
                                      "(ncu --set full, mean over one layer's 12 GEMM launches), "
                                      + traffic_src) if traffic else "no ncu capture for this workload",
                     "flops_per_launch": g["work"] / max(1, g["launches"]),
                     "of": peaks["source"] + " bf16_tflops_sustained", "launches_per_step": g["launches"] / args.steps,
                     "kernel_ms_per_step": round(g["ms"] / args.steps, 3),
                     "measured": f"per-launch CUDA events over a second pass of the same {args.steps} steps "
                                 f"({ms_profiled:.2f} ms/step with the events enabled)"},
        "step_roofline": {"flops_per_pair": F, "achieved": step_tf, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                          "frac": step_tf / peaks["bf16_sustained"],
                          "note": "hot-path algorithmic FLOPs (SURVEY.md §8d, heads and recompute not credited) over the whole step"},
        "kernel_ms_per_step": kern_ms,
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": int(h2d_bytes),
                "d2h_bytes_per_step": 4, "host_enqueue_ms_per_step": round(1e3 * enq[0] / max(1, enq[1]), 3)},
    }
    if args.dump_outputs:
        line["dump_outputs"] = {"dir": args.dump_outputs, "files": dumped[0], "bytes": dumped[1],
                                "of": f"the last of the {args.steps} timed steps"}
    if opt_info is not None:
        line["optimizer"] = opt_info
    if others is not None:
        line["other_configs"] = others
    if world == 1 and not args.no_cpu_baseline:
        dt, threads, spread = cpu_oracle_step_time(c, args.cpu_sample, 5, 1, threads=cpu_threads())
        line["cpu_baseline"] = {"value": args.cpu_sample / dt, "unit": UNIT, "cores": threads, "kind": "port", "spread": spread,
                                "sample": f"{args.cpu_sample} pairs/step x 5 steps fwd+bwd of the same workload, fp32 oracle, "
                                          f"{os.cpu_count()} logical CPUs, {threads} torch threads"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(synthetic.CONFIGS))
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch override (parity/debug only)")
    ap.add_argument("--cpu-sample", type=int, default=8, help="pairs per CPU step (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--other-configs", action="store_true",
                    help="also time BASELINE.json configs[2..4] at their per-GPU batch (always on for N > 1)")
    ap.add_argument("--optimizer", action="store_true",
                    help="also run the fused BertAdam step every step (SURVEY §8f rank 2; the BASELINE metric excludes it)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (outputs, sampled gradients) as "
                         "DIR/<name>.npy, float32, 64 MB at most")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
