#!/usr/bin/env python
"""bench.py -- headline benchmark: tokens/sec (device-timed) of the Llama training step.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c1|c2|c3|c4|c5] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workloads = BASELINE.json `configs` (YAMLs under configs/, reference schema), default C2, the configuration
the metric is quoted on at one GPU:
  c1  Llama 2M    AdamW    fp32   B16 x S1024                     (plumbing / loss parity config)
  c2  Llama "80M" Muon     bf16   B16 x S1024   V = 32003         <- default, `value`
  c3  Llama 400M  Muon     bf16   B16 x S2048 x 8 accumulation micro-batches, clip 1.0
  c4  Llama 256M  Shampoo  bf16   B64 x S2048   roots every 100 steps (the timed region contains one recompute)
  c5  Llama 1B    AdamW    bf16   B32 x S2048   D = 128
A "step" = ONE OPTIMIZER UPDATE: `gradient_accumulation_steps` x (fwd + bwd + clamp/accumulate) + gradient
all-reduce (N > 1) + the full optimizer update.  Weak scaling: per-GPU batch fixed.  One JSON line (rank 0).

Keys beyond the base contract:
  roofline      dominant hand-written kernel family of the config (Muon configs: the Newton-Schulz GEMM chain;
                others: attention backward), timed live with CUDA events on the launching stream
  kernels       every hand-written tensor-core family timed the same way
  cpu_baseline  CPU restatement of the reference step (oracle/) on the host cores: for c1/c2 ONE FULL measured
                step, for c3-c5 a bounded sample (stated in `sample`)
  e2e           same step through the public Trainer.train_step with per-step pinned H2D + loss D2H
  configs       (default run only) C3 -- the 400M + Muon config the >= 100x target is quoted on -- on one GPU,
                with its own CPU baseline sample
  dp_check      (N > 1) replicas bit-identical after the timed loop; one update through every exchange
                implementation (peer-store unicast / NVSwitch multicast / NCCL all-gather) compared
--impl reference times the reference's CPU path (the oracle port: MLX is not installable here).
--dump-outputs DIR writes what the last timed step returned (see dump_outputs) so two builds can be compared.
Trainer run directories go to a temporary directory: the benchmark writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402
import yaml  # noqa: E402

CONFIG_FILES = {"c1": "c1-llama2m-adamw.yaml", "c2": "c2-llama80m-muon.yaml", "c3": "c3-llama400m-muon-dp8.yaml",
                "c4": "c4-llama256m-shampoo-dp4.yaml", "c5": "c5-llama1b-adamw-dp8.yaml"}


def load_config(tag: str, distributed: bool) -> dict:
    d = yaml.safe_load((ROOT / "configs" / CONFIG_FILES[tag]).read_text())
    d["name"] = f"bench-{tag}"
    d["overwrite"] = True
    d["system"]["distributed"] = bool(distributed)
    d["logging"]["steps"] = {"logging_interval": 10 ** 9, "checkpoint_interval": 0, "validation_interval": 0}
    return d


def dims_of(d: dict) -> dict:
    m, hp = d["model"], d["training"]["hyperparameters"]
    hidden = m["dimensions"]["hidden_size"]
    heads = m["attention"]["num_heads"]
    return dict(hidden=hidden, inter=m["dimensions"]["intermediate_size"], layers=m["dimensions"]["num_layers"],
                heads=heads, kv_heads=m["attention"].get("num_kv_heads") or heads,
                head_dim=m["attention"].get("head_dim") or hidden // heads,
                vocab_normal=d["data"]["tokenizer"]["normal_vocab_size"],
                vocab=d["data"]["tokenizer"]["normal_vocab_size"] + 3,
                batch=hp["batch_size"], seq=d["data"]["preprocessing"]["max_context_size"],
                accum=int(hp.get("gradient_accumulation_steps") or 1),
                optimizer=d["training"]["optimization"]["optimizer"],
                mixed=bool(d["system"].get("mixed_precision")))


def workload_name(tag: str, c: dict) -> str:
    opt = {"muon": "Muon NS5", "adamw": "AdamW", "shampoo": "Shampoo"}.get(c["optimizer"], c["optimizer"])
    acc = f" x {c['accum']} accumulation micro-batches" if c["accum"] > 1 else ""
    return (f"{tag.upper()}: Llama (h{c['hidden']} i{c['inter']} L{c['layers']} H{c['heads']}/{c['kv_heads']} "
            f"D{c['head_dim']} V{c['vocab']}) {opt}, batch {c['batch']} x seq {c['seq']}{acc} per GPU")


def matrix_shapes(c: dict):
    mats = [(c["vocab"], c["hidden"])]
    for _ in range(c["layers"]):
        mats += [(c["heads"] * c["head_dim"], c["hidden"]), (c["kv_heads"] * c["head_dim"], c["hidden"]),
                 (c["kv_heads"] * c["head_dim"], c["hidden"]), (c["hidden"], c["heads"] * c["head_dim"]),
                 (c["inter"], c["hidden"]), (c["inter"], c["hidden"]), (c["hidden"], c["inter"])]
    return mats


def ns_flops(shape) -> float:
    m, n = min(shape), max(shape)
    return 5.0 * (4.0 * m * m * n + 2.0 * m ** 3)


def ns_flops_per_step(c: dict) -> float:
    """5*(4 m^2 n + 2 m^3) over every 2-D parameter (SURVEY 8d): 4.129 TF for C2, 6.566 TF for C3."""
    return sum(ns_flops(s) for s in matrix_shapes(c))


def attn_flops_fwd_per_step(c: dict) -> float:
    """4 B H S^2 D per layer, full (non-causal-discounted) count, all micro-batches of one update."""
    return 4.0 * c["batch"] * c["heads"] * c["seq"] ** 2 * c["head_dim"] * c["layers"] * c["accum"]


def attn_bytes_per_step(c: dict):
    """Algorithmic HBM bytes of attention fwd / bwd (bf16 I/O, fp32 LSE/delta), SURVEY 8d formulas."""
    B, S, H, Hk, D, L = c["batch"], c["seq"], c["heads"], c["kv_heads"], c["head_dim"], c["layers"] * c["accum"]
    fwd = L * (B * S * (2 * H * D + 2 * Hk * D) * 2 + 4 * B * H * S)
    bwd = L * (B * S * (3 * H * D + 2 * Hk * D) * 2 + B * S * (H * D + 2 * Hk * D) * 2 + 8 * B * H * S)
    return float(fwd), float(bwd)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = time.perf_counter() + 0.5
        while not self.rows and time.perf_counter() < t_end:   # timed region shorter than one 100 ms sample (C1):
            time.sleep(0.02)                                   # take the first sample that arrives right after it
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:  # noqa: BLE001
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def load_peaks() -> dict:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"bf16_tflops": d.get("bf16_tflops", 1590.0), "bf16_tflops_sustained": d.get("bf16_tflops_sustained", 1400.0),
                "hbm_gbs": d.get("hbm_gbs", 6650.0), "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference step on the host cores
# ------------------------------------------------------------------------------------------------
def pick_cpu_threads(c: dict) -> int:
    """Thread count for the CPU arm: the fastest of n, n/2, n/4, n/8 host threads on a probe of the workload itself
    -- fwd+bwd of ONE sequence through a 2-layer cut of the config's model (same widths, seq <= 1024) -- because the
    oracle's step mixes GEMMs with memory-bound elementwise work and a plain matmul probe picked 64 threads on a box
    where 32 ran the real step 1.4x faster (profiles/r03_bench_c2.json vs r03_bench_reference.json).  The choice is
    reported in cpu_baseline.cores."""
    from oracle import reference_math as R
    n = os.cpu_count() or 1
    cand = sorted({n, max(1, n // 2), max(1, n // 4), max(1, n // 8)}, reverse=True)
    dims = R.LlamaDims(c["hidden"], c["inter"], 2, c["heads"], c["kv_heads"], c["head_dim"], c["vocab"])
    params = R.init_params(dims, seed=1)
    batch = R.synthetic_batch(0, 0, 1, min(c["seq"], 1024), c["vocab_normal"])
    best, best_t = n, float("inf")
    for th in cand:
        torch.set_num_threads(th)
        R.loss_and_grads(params, batch, dims, pad_token=c["vocab_normal"])       # warm the pool at this width
        t0 = time.perf_counter()
        R.loss_and_grads(params, batch, dims, pad_token=c["vocab_normal"])
        t = time.perf_counter() - t0
        if t < best_t:
            best, best_t = th, t
    torch.set_num_threads(best)
    return best


def cpu_reference_step(tag: str, threads: int, full: bool) -> dict:
    """Times the CPU restatement of the reference optimizer step (oracle/reference_math.py, fp32; the oracle is
    test infrastructure and only ever the thing TIMED here, never the product path).

    full=True  : every micro-batch sequence goes through fwd+bwd (in chunks of 4 sequences, gradients averaged:
                 same arithmetic as one big batch, bounded memory for the oracle's dense [B,H,S,S] scores) and
                 the optimizer updates every parameter -> a measured step, nothing extrapolated.
    full=False : bounded sample for the big configs: fwd+bwd on ONE sequence (scaled by batch x accumulation)
                 + the full optimizer update on every parameter (measured, not scaled)."""
    from oracle import reference_math as R
    d = load_config(tag, False)
    c = dims_of(d)
    dims = R.LlamaDims(c["hidden"], c["inter"], c["layers"], c["heads"], c["kv_heads"], c["head_dim"], c["vocab"])
    params = R.init_params(dims, seed=42)
    hp, oc = d["training"]["hyperparameters"], d["training"]["optimization"]
    lr = hp["learning_rate"]
    if c["optimizer"] == "muon":
        opt = R.MuonOracle(lr)
    elif c["optimizer"] == "shampoo":
        opt = R.ShampooOracle(lr, R.ShampooParams(beta2=oc.get("beta2", 0.95), update_period=oc.get("update_period", 100),
                                                 start_preconditioning_step=oc.get("start_preconditioning_step", 1000)))
    else:
        opt = R.AdamWOracle(lr, betas=tuple(oc.get("betas", (0.9, 0.999))), eps=oc.get("eps", 1e-8),
                            weight_decay=hp.get("weight_decay", 0.01))
    n_seq_total = c["batch"] * c["accum"]
    chunk = 4 if full else 1
    n_chunks = (c["batch"] // chunk) * c["accum"] if full else 1
    grads = None
    t0 = time.perf_counter()
    loss = None
    for i in range(n_chunks):
        batch = R.synthetic_batch(i, 0, chunk, c["seq"], c["vocab_normal"])
        loss, ntoks, g = R.loss_and_grads(params, batch, dims, pad_token=c["vocab_normal"])
        if grads is None:
            grads = g
        else:
            for k in grads:
                grads[k] += g[k]
    if n_chunks > 1:
        for k in grads:
            grads[k] /= n_chunks
    t_fb = time.perf_counter() - t0
    t0 = time.perf_counter()
    opt.update(params, grads)
    t_opt = time.perf_counter() - t0
    scale = 1.0 if full else n_seq_total / chunk
    step_s = t_fb * scale + t_opt
    tokens = c["batch"] * c["seq"] * c["accum"]
    if full:
        sample = (f"oracle fp32 CPU, ONE FULL measured step: fwd+bwd on all {n_seq_total} sequences "
                  f"({n_chunks} chunks of {chunk}, {t_fb:.1f}s) + {c['optimizer']} update of all parameters "
                  f"({t_opt:.1f}s); nothing extrapolated")
    else:
        sample = (f"oracle fp32 CPU, bounded sample: fwd+bwd on 1 of {n_seq_total} sequences ({t_fb:.1f}s, scaled x"
                  f"{int(scale)}) + the full {c['optimizer']} update of all parameters ({t_opt:.1f}s, measured); "
                  f"est. step {step_s:.0f}s")
    return {"value": tokens / step_s, "unit": "tokens/s", "cores": threads, "kind": "port",
            "sample": sample + "; MLX (the reference runtime) is not installable here",
            "step_s": step_s, "measured_s": t_fb + t_opt, "fwd_bwd_s": t_fb, "optimizer_s": t_opt,
            "full_step": bool(full), "loss": float(loss)}


def run_reference(args) -> None:
    """Reference arm: rank 0 only.  Each "step" is one cpu_reference_step (a FULL step for c1/c2), and exactly
    `--steps` of them are timed (a C2 step takes tens of seconds on the host cores)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    tag = args.config
    c = dims_of(load_config(tag, False))
    full = tag in ("c1", "c2")
    threads = pick_cpu_threads(c)
    rows = [cpu_reference_step(tag, threads, full) for _ in range(args.steps)]
    v = statistics.median(r["value"] for r in rows)
    last = rows[-1]
    tokens = c["batch"] * c["seq"] * c["accum"]
    line = {"impl": "reference", "metric": "tokens/sec (device-timed) Llama training step", "value": v, "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": len(rows), "steps_requested": args.steps, "warmup": 0,
            "ms_per_step": 1e3 * tokens / v, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(tag, c)},
            "cpu_baseline": {**{k: last[k] for k in ("unit", "cores", "kind", "sample", "full_step")}, "value": v,
                             "host_threads_available": os.cpu_count(),
                             "note": "wall-clock of whole steps; no warm-up steps are discarded (the first step "
                                     "includes thread-pool start-up, < 1 % of a step)"},
            "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def master_fingerprint(store) -> torch.Tensor:
    """Order-independent but bit-sensitive checksum of the fp32 masters: sum of the raw bit patterns (int64)."""
    return store.master.view(torch.int32).to(torch.int64).sum().reshape(1)


DUMP_BYTES = 60 << 20      # data bytes of all dumped arrays; with the .npy headers the dump stays under 64 MiB


def dump_outputs(out_dir: Path, loss: torch.Tensor, store) -> None:
    """What a caller of the timed step receives after its last step: `loss.npy` (the loss of the last micro-batch)
    and `param.<name>.npy` for every parameter (the fp32 master weights after the update), flattened.  A tensor
    larger than its share of DUMP_BYTES is sampled at distinct indices drawn from a generator seeded with 0 that
    depend only on its size, so two builds dump the same elements of the same parameter."""
    import numpy as np
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "loss.npy", loss.float().reshape(1).cpu().numpy())
    named = store.named_master()
    cap = DUMP_BYTES // 4 // len(named)
    index_of_size = {}
    for name, t in named.items():
        flat = t.detach().reshape(-1)
        n = flat.numel()
        if n > cap:
            if n not in index_of_size:
                index_of_size[n] = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:cap].sort().values
            flat = flat[index_of_size[n].to(flat.device)]
        np.save(out_dir / f"param.{name}.npy", flat.float().cpu().numpy())


def run_workload(tag: str, K: int, W: int, with_e2e: bool = True, with_dp_check: bool = True,
                 dump_dir: Path | None = None) -> dict:
    from mlx_cuda_distributed_pretraining_b200 import ops
    from mlx_cuda_distributed_pretraining_b200._lib import lib
    from mlx_cuda_distributed_pretraining_b200.core.training import Config, Trainer
    from mlx_cuda_distributed_pretraining_b200.distributed import dp

    rank, world, local_rank = dp.env_rank_world()
    d = load_config(tag, distributed=world > 1)
    c = dims_of(d)
    k = c["accum"]
    d["training"]["hyperparameters"]["iters"] = max(d["training"]["hyperparameters"].get("iters", 0), (2 * (K + W) + 8) * k)
    run_root = tempfile.TemporaryDirectory(prefix="bench-runs-")
    tr = Trainer(Config.from_dict(d), synthetic=True, quiet=True, run_root=run_root.name)
    tr._accum_step, tr._accum_tokens = 0, 0
    dev = tr.device
    tokens_per_step = c["batch"] * c["seq"] * k * world
    shampoo_t0 = None
    if c["optimizer"] == "shampoo":
        # BASELINE configs[3]: "preconditioner recompute every 100 steps".  Steady state = preconditioners
        # present on every step and one recompute per `update_period`: the first warm-up step lands on a
        # recompute (t0 = first multiple of the period at/after start_preconditioning_step), and after the warm-up
        # the counter is moved so that the NEXT recompute (t0 + period) falls in the middle of the timed region.
        hpp = tr.optimizer.params
        shampoo_t0 = -(-hpp.start_preconditioning_step // hpp.update_period) * hpp.update_period
        tr.optimizer.init(tr.model)
        tr.optimizer.count = shampoo_t0 - 1

    def sync_all():
        if world > 1:
            dp.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    # ---------------- leg 1: device-resident inputs (the `value`) --------------------------------
    n_micro = (K + W) * k
    dev_batches = [tr.data_manager.generate_batch(s).to(dev) for s in range(n_micro)]

    def update_resident(u: int):
        for j in range(k):
            loss, _, _ = tr.micro_step(u * k + j, dev_batches[u * k + j])
        return loss

    for u in range(W):
        update_resident(u)
    if shampoo_t0 is not None:
        tr.optimizer.count = shampoo_t0 + tr.optimizer.params.update_period - 1 - K // 2
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ops.TIMER = ops.KernelTimer()
    launches0 = lib().b200_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    h0 = time.perf_counter()
    for u in range(W, W + K):
        loss = update_resident(u)
    host_issue_ms = 1e3 * (time.perf_counter() - h0) / K     # CPU time to ISSUE a step (no sync inside): << ms_per_step
    e1.record()                                              # means the device, not the host, sets the pace
    sync_all()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = int(lib().b200_launch_count() - launches0)
    kt = ops.TIMER.totals_ms()
    ops.TIMER = None
    clocks = sampler.stop() if rank == 0 else {}
    final_loss = float(loss.item())
    if dump_dir is not None and rank == 0:      # before the e2e leg below trains on
        dump_outputs(dump_dir, loss, tr.store)
    ms_per_step = ms_total / K
    value = tokens_per_step / (ms_per_step / 1e3)

    # ---------------- leg 2: end to end through the public API (pinned H2D + loss D2H) -----------
    e2e = None
    if with_e2e:
        host_batches = [tr.data_manager.generate_batch(s) for s in range((K + 1) * k)]
        base = n_micro
        for j in range(k):      # one untimed update on this path
            l, _, _ = tr.train_step(base + j, host_batches[j])
        float(l.item())
        sync_all()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for u in range(K):
            for j in range(k):
                l, _, _ = tr.train_step(base + (u + 1) * k + j, host_batches[(u + 1) * k + j])
            float(l.item())  # device -> host read of the update's loss
        f1.record()
        sync_all()
        e2e_ms = max_over_ranks(f0.elapsed_time(f1)) / K
        e2e = {"value": tokens_per_step / (e2e_ms / 1e3), "unit": "tokens/s", "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": host_batches[0].numel() * host_batches[0].element_size() * k,
               "d2h_bytes_per_step": 4}

    # ---------------- data-parallel cross-checks (N > 1) ------------------------------------------
    dp_check = None
    if world > 1 and with_dp_check:
        fp = master_fingerprint(tr.store)
        lo, hi = fp.clone(), fp.clone()
        torch.distributed.all_reduce(lo, op=torch.distributed.ReduceOp.MIN)
        torch.distributed.all_reduce(hi, op=torch.distributed.ReduceOp.MAX)
        dp_check = {"replicas_bit_identical": bool(int(lo.item()) == int(hi.item())),
                    "after_updates": 2 * K + W + 1, "exchange_in_timed_region": getattr(tr.optimizer, "exchange_mode", None)}
        # gradient exchange precision: the flat gradient buffer is reduced in its storage type (bf16 unless the
        # config accumulates micro-batches in fp32); measure what that costs against an fp32 reduction of the same
        # per-rank gradients (the reference averages fp32 arrays, hybrid_distributed.py:352)
        if not tr.use_acc and tr.store.grad.dtype == torch.bfloat16:
            tr.store.zero_grad()
            fb = tr.data_manager.generate_batch(10 ** 6 + 7).to(dev)
            l_, _ = tr.compute_loss(tr.model, fb[:, :-1], fb[:, 1:])
            l_.backward()
            g32 = tr.store.grad.float()
            g16 = tr.store.grad.clone()
            torch.distributed.all_reduce(g32)
            torch.distributed.all_reduce(g16)
            dp_check["grad_allreduce"] = {"dtype": "bf16", "ranks": world,
                                          "rel_err_vs_fp32_reduce": float((g16.float() - g32).norm() / (g32.norm() + 1e-30)),
                                          "bf16_storage_rounding_alone": float((g32.to(torch.bfloat16).float() - g32).norm() / (g32.norm() + 1e-30))}
            del g32, g16
            tr.store.zero_grad()
        elif tr.use_acc:
            dp_check["grad_allreduce"] = {"dtype": "f32", "ranks": world, "note": "fp32 accumulation buffer is reduced"}
        opt = getattr(tr.optimizer, "matrix_optimizer", tr.optimizer)
        if hasattr(opt, "set_exchange") and getattr(opt, "shard_ns", False):
            # ONE update from identical state through every exchange implementation: the fused GEMM -> all-gather
            # peer stores (unicast, NVSwitch multicast) must reproduce the plain NCCL all-gather's parameters
            store = tr.store
            # gradients of one fixed batch, computed and all-reduced ONCE (the backward's fp32 dQ atomics are not
            # bit-reproducible, and Newton-Schulz amplifies such noise): every mode starts from the same bits
            store.zero_grad()
            tr._accum_step = 0
            for j in range(k):
                fb = tr.data_manager.generate_batch(10 ** 6 + j).to(dev)
                l_, _ = tr.compute_loss(tr.model, fb[:, :-1], fb[:, 1:])
                l_.backward()
                if tr.use_acc:
                    ops.clip_accum(store.grad, store.acc, tr.clip_value, 1.0 / k, init=(j == 0))
                    store.zero_grad()
            gsrc = store.acc if tr.use_acc else store.grad
            dp.all_reduce_sum_(gsrc)
            snap = (store.master.clone(), opt._buf.clone(), opt.count, gsrc.clone())
            alt = getattr(opt, "alternate_optimizer", None)
            alt_snap = (alt._m.clone(), alt._v.clone(), alt.count) if alt is not None and hasattr(alt, "_m") else None
            results = {}
            for mode in ("nccl", "unicast", "multicast"):
                eff = opt.set_exchange(mode)
                if (mode == "multicast") != ("multicast" in eff) or (mode == "nccl") != ("NCCL" in eff):
                    results[mode] = {"available": False, "effective": eff}
                    continue
                store.master.copy_(snap[0]); store.refresh_shadow(); opt._buf.copy_(snap[1]); opt.count = snap[2]
                gsrc.copy_(snap[3])
                if alt_snap is not None:
                    alt._m.copy_(alt_snap[0]); alt._v.copy_(alt_snap[1]); alt.count = alt_snap[2]
                tr.optimizer.update(tr.model)
                torch.cuda.synchronize()
                upd = store.master - snap[0]
                fpm = master_fingerprint(store)
                lo, hi = fpm.clone(), fpm.clone()
                torch.distributed.all_reduce(lo, op=torch.distributed.ReduceOp.MIN)
                torch.distributed.all_reduce(hi, op=torch.distributed.ReduceOp.MAX)
                results[mode] = {"available": True, "effective": eff, "replicas_bit_identical": bool(int(lo.item()) == int(hi.item())),
                                 "_upd": upd}
            ref = results.get("nccl", {}).get("_upd")
            for mode, r in results.items():
                u = r.pop("_upd", None)
                if u is not None and ref is not None and mode != "nccl":
                    # same gradients, same momentum: ownership (flop-balanced vs equal chunks) only changes which rank
                    # computes a matrix and, through the batch size of a launch, the split-K choice of a few GEMMs
                    r["max_rel_update_diff_vs_nccl"] = float((u - ref).norm() / (ref.norm() + 1e-30))
                    r["bit_identical_to_nccl"] = bool(torch.equal(u, ref))
            opt.set_exchange("auto")
            dp_check["exchange"] = results

    if world > 1:
        dp.barrier()
    out = {"tag": tag, "c": c, "rank": rank, "world": world, "value": value, "ms_per_step": ms_per_step,
           "tokens_per_step": tokens_per_step, "launches": launches, "host_issue_ms": host_issue_ms, "kt": kt, "clocks": clocks, "final_loss": final_loss,
           "e2e": e2e, "dp_check": dp_check, "K": K, "W": W}
    # flops of the matrices THIS rank orthogonalised (all of them unless the owner-computes mode is on)
    optm = getattr(tr.optimizer, "matrix_optimizer", tr.optimizer)
    if c["optimizer"] in ("muon", "hybrid"):
        sharded = bool(getattr(optm, "shard_ns", False)) and world > 1
        fl = 0.0
        for gi, g in enumerate(tr.store.mat_groups):
            owned = sum(hi_ - lo_ for lo_, hi_ in optm.owned_ranges_of(gi, world if sharded else 1, rank))
            fl += owned * ns_flops((g.rows, g.cols))
        out.update(ns_flops_rank=fl, ns_sharded=sharded, ns_exchange=getattr(optm, "exchange_mode", None))
        if sharded:
            # every rank's Newton-Schulz bracket and flops: the slowest rank sets the step (the others wait at the
            # exchange barrier), so the JSON line can name the limiter
            mine = torch.tensor([kt.get("newton_schulz", (0.0, 0))[0] / K, fl / 1e12], device=dev, dtype=torch.float64)
            allr = [torch.zeros_like(mine) for _ in range(world)]
            torch.distributed.all_gather(allr, mine)
            ms_r, tf_r = [float(t[0]) for t in allr], [float(t[1]) for t in allr]
            slow = max(range(world), key=lambda i: ms_r[i])
            share = sum(tf_r) / world
            why = ("flop-balanced ownership; the spread is the last GEMM's peer stores sharing NVLink with the all-gather "
                   "of every rank's updates (2 bytes x all matrix parameters into each rank per step)")
            if tf_r[slow] > 1.15 * share:
                why = (f"this rank's largest matrix is one indivisible chain above the per-rank share of {share:.2f} TFLOP "
                       "(C2 at 8 ranks: the 32003 x 1024 embedding, 0.68 TFLOP, 0.65 ms when timed alone on an idle GPU: "
                       "tools/ns_single_probe.py), and its last GEMM's peer stores share NVLink with the all-gather of "
                       "every rank's updates (2 bytes x all matrix parameters into each rank per step)")
            out["ns_ranks"] = {
                "ns_ms_per_rank": [round(x, 3) for x in ms_r], "ns_tflop_per_rank": [round(x, 3) for x in tf_r],
                "slowest_rank": slow,
                "limiter": (f"rank {slow}: {ms_r[slow]:.2f} ms for {tf_r[slow]:.2f} TFLOP (mean of the others "
                            f"{(sum(ms_r) - ms_r[slow]) / max(1, world - 1):.2f} ms); " + why)}
    del tr
    torch.cuda.empty_cache()
    run_root.cleanup()
    return out


def summarize(r: dict, peaks: dict) -> dict:
    """JSON line pieces (roofline / kernels) from a run_workload result."""
    c, kt, K = r["c"], r["kt"], r["K"]
    peak_tf, peak_burst = peaks["bf16_tflops_sustained"], peaks["bf16_tflops"]
    kernels = {}
    afl = attn_flops_fwd_per_step(c)
    ab_f, ab_b = attn_bytes_per_step(c)
    for nm, fl, by in (("attn_fwd", afl, ab_f), ("attn_bwd", 2.5 * afl, ab_b)):
        ms, calls = kt.get(nm, (0.0, 0))
        if ms > 0:
            tf = fl / (ms / K * 1e-3) / 1e12
            kernels[nm] = {"ms_per_step": ms / K, "calls_per_step": calls / K, "tflops_full_count": tf,
                           "frac_of_tensor_peak": tf / peak_tf, "frac_of_tensor_peak_burst": tf / peak_burst,
                           "algorithmic_gb_per_step": by / 1e9,
                           "frac_of_hbm_peak": by / (ms / K * 1e-3) / 1e9 / peaks["hbm_gbs"]}
    for nm in ("shampoo_stats", "shampoo_root", "shampoo_precond"):
        ms, calls = kt.get(nm, (0.0, 0))
        if calls:
            kernels[nm] = {"ms_total_in_timed_region": ms, "calls": calls, "ms_per_call": ms / calls}
    ns_ms, _ = kt.get("newton_schulz", (0.0, 0))
    roofline = None
    if ns_ms > 0 and "ns_flops_rank" in r:
        ns_step = ns_ms / K
        tf = r["ns_flops_rank"] / (ns_step * 1e-3) / 1e12
        traffic, traffic_src = None, None
        for tf_path in sorted(ROOT.glob("profiles/*_gemm_traffic.json")):   # written by tools/summarize_profiles.py
            try:
                traffic = float(json.loads(tf_path.read_text())["mean_dram_bytes_per_launch"])
                traffic_src = f"{tf_path.relative_to(ROOT)} (ncu --set full, mean DRAM read+write bytes per launch)"
            except Exception:  # noqa: BLE001
                pass
        roofline = {"kernel": "gemm2_bf16_tc_kernel (Newton-Schulz chain: batched tcgen05 cta_group::2 GEMMs)",
                    "bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf,
                    "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
                    "frac_of_burst": tf / peak_burst, "algorithmic_flops_per_step": r["ns_flops_rank"],
                    "algorithmic_flops_all_ranks": ns_flops_per_step(c), "ns_sharded_over_ranks": r["ns_sharded"],
                    "ns_exchange": r["ns_exchange"], "ms_per_step": ns_step, "share_of_step": ns_step / r["ms_per_step"]}
        if r.get("ns_ranks"):
            roofline.update(r["ns_ranks"])
    elif "attn_bwd" in kernels:
        kb = kernels["attn_bwd"]
        roofline = {"kernel": "attn_bwd (fused causal/GQA attention backward, tcgen05; 2.5 x 4BHS^2D flops, full count)",
                    "bound": "tensor", "achieved": kb["tflops_full_count"], "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": kb["frac_of_tensor_peak"], "frac_of_burst": kb["frac_of_tensor_peak_burst"], "traffic": None,
                    "peak_source": peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
                    "hbm_frac": kb["frac_of_hbm_peak"], "ms_per_step": kb["ms_per_step"],
                    "share_of_step": kb["ms_per_step"] / r["ms_per_step"]}
    return {"roofline": roofline, "kernels": kernels}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=str, default="c2", choices=sorted(CONFIG_FILES))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs-block", action="store_true", help="skip the extra C3 single-GPU leg of the default run")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs: only the device-resident leg")
    ap.add_argument("--dump-outputs", type=Path, metavar="DIR",
                    help="b200 arm: write the loss and (sampled) parameters after the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return
    args.warmup = max(args.warmup, 3)

    from mlx_cuda_distributed_pretraining_b200.distributed import dp
    rank, world, _ = dp.env_rank_world()
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    tag = args.config
    r = run_workload(tag, args.steps, args.warmup, with_e2e=not args.no_e2e, dump_dir=args.dump_outputs)
    extra = None
    if world == 1 and tag == "c2" and not args.no_configs_block:
        extra = run_workload("c3", args.steps, 3, with_e2e=False)
    if rank != 0:
        dp.destroy()
        return

    peaks = load_peaks()
    c = r["c"]
    s = summarize(r, peaks)
    line = {
        "metric": "tokens/sec (device-timed) Llama training step", "value": r["value"], "unit": "tokens/s",
        "n_gpus": world, "steps": r["K"], "warmup": r["W"], "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if c["mixed"] else "f32", "data": "synthetic",
        "config": {"workload": workload_name(tag, c), "global_batch": c["batch"] * world, "seq_len": c["seq"],
                   "micro_batches_per_step": c["accum"], "parallelism": f"dp{world}",
                   "l2": "working set (params+grads+activations, GBs) >> 126 MB L2"},
        "e2e": r["e2e"], "gpu_launches": r["launches"], "host_issue_ms_per_step": r["host_issue_ms"], "clocks": r["clocks"], "roofline": s["roofline"],
        "kernels": s["kernels"], "final_loss": r["final_loss"],
    }
    if r["dp_check"] is not None:
        line["dp_check"] = r["dp_check"]
        modes = r["dp_check"].get("exchange") or {}
        ok = r["dp_check"]["replicas_bit_identical"] and all(m.get("replicas_bit_identical", True) for m in modes.values())
        line["dp_check"]["passed"] = bool(ok)
        if not ok:   # the number below is still printed, but a diverged replica set must not pass unnoticed
            print("[bench] DATA-PARALLEL CHECK FAILED: replicas are not bit-identical: "
                  + json.dumps(r["dp_check"]), file=sys.stderr, flush=True)
    if world == 1 and not args.no_cpu_baseline:
        try:
            threads = pick_cpu_threads(dims_of(load_config(tag, False)))
            line["cpu_baseline"] = cpu_reference_step(tag, threads, full=tag in ("c1", "c2"))
            line["cpu_baseline"]["host_threads_available"] = os.cpu_count()
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"error": repr(e)}
    if extra is not None:
        s3 = summarize(extra, peaks)
        blk = {"workload": workload_name("c3", extra["c"]), "n_gpus": 1, "value": extra["value"], "unit": "tokens/s",
               "ms_per_step": extra["ms_per_step"], "steps": extra["K"], "warmup": extra["W"],
               "roofline": s3["roofline"], "kernels": s3["kernels"], "final_loss": extra["final_loss"]}
        if not args.no_cpu_baseline:
            try:
                blk["cpu_baseline"] = cpu_reference_step("c3", torch.get_num_threads(), full=False)
                blk["speedup_vs_cpu_baseline"] = extra["value"] / blk["cpu_baseline"]["value"]
            except Exception as e:  # noqa: BLE001
                blk["cpu_baseline"] = {"error": repr(e)}
        line["configs"] = {"c3": blk}
    print(json.dumps(line), flush=True)
    if world > 1:
        dp.destroy()


if __name__ == "__main__":
    main()
