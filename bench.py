#!/usr/bin/env python
"""bench.py -- MoE-layer forward tokens/s on B200 (BASELINE.json metric), one fused persistent kernel per step.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--sweeps a,b,..]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload (default `--config B`): BASELINE.json configs[1] (8 experts, top-2, S=4096 tokens per rank, d_model 1024, ffn 4096,
bf16, capacity_factor 1, drop_tokens 1, ReLU, zero bias), synthetic N(0,1) activations/weights seeded per rank like the
reference harness (flashmoe/worker.py:56-58); at N > 1 the experts are sharded over the N ranks and every rank keeps its
own S tokens (weak scaling, per-GPU FLOPs fixed).  `--config C | D1k | D4k | D16k | D64k | E8 .. E128` selects the other
BASELINE.json shapes (flashmoe_b200/config.py); `--sweeps` appends reduced-step measurements of further configs to the
same JSON line (`"sweeps": [...]`).

Prints ONE JSON line (rank 0).  `value` = N*S / (max over ranks of the device time per step), inputs resident in HBM;
`e2e` = the same metric through the public host-buffer entry point (pinned host activations in, host output back, every
step's copies inside the timed region; steps are pipelined three deep so the copies overlap the kernels).  `roofline`
describes the dominant work (the two expert GEMMs on tcgen05) against the measured cuBLAS bf16 throughput of this pool
(MEASURED_PEAKS.json: burst peak when the timed region is shorter than a second, else sustained; both fractions are
printed); `parity_check` is one extra forward on seeded, scaled inputs after the timed loops, every rank's output and
top-k checked against the CPU oracle on a sample of its tokens (outside any timed region; a failure exits non-zero);
`cpu_baseline` is a plain torch CPU forward of the same layer on the host cores (a reported baseline, not a target).
`--impl reference` times that CPU implementation as the reference arm: the reference itself has no CPU path and cannot
be built here (SURVEY.md section 8c), so the oracle port is the stated stand-in.

`--steps K` is the number of steps of every timed loop of the headline configuration (device-resident and end to end).
`--dump-outputs DIR` writes what the last device-resident timed step returned to its caller, the layer output, as
float32 `DIR/out.npy` (`DIR/out_rank<r>.npy` per rank at N > 1); the inputs are seeded, so two builds run with the same
arguments can be compared output for output.  Above 64 MB for all ranks together a fixed, seeded sample of token rows
is written instead (`dump_outputs`).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def _configs():
    # flashmoe_b200.config is pure Python; imported by file path so that the reference arm never runs the package's
    # __init__ (which maps the product's native library into the process)
    import importlib.util

    spec = importlib.util.spec_from_file_location("_fm_config", os.path.join(ROOT, "flashmoe_b200", "config.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["_fm_config"] = mod
    spec.loader.exec_module(mod)
    return mod


_CFG = _configs()
BASELINE_CONFIGS, CONFIG_DESCRIPTIONS = _CFG.BASELINE_CONFIGS, _CFG.CONFIG_DESCRIPTIONS


def env_int(name, default):
    return int(os.environ.get(name, default))


def config_dict(name, cfg, world):
    """The `config` object of the JSON line; identical in both arms (the driver compares them)."""
    return {"workload": CONFIG_DESCRIPTIONS[name], "name": name, "experts": cfg.E, "top_k": cfg.k, "tokens_per_rank": cfg.S,
            "d_model": cfg.H, "ffn": cfg.P, "capacity_factor": cfg.capacity_factor, "drop_tokens": cfg.drop_tokens,
            "hidden_act": "relu", "parallelism": f"ep{world}"}


def make_inputs(cfg, nlx, rank):
    """Reference-harness style synthetic data (N(0,1), unscaled), seeded: x and local experts per rank, the gate
    weights identical on all ranks."""
    g = torch.Generator().manual_seed(0x5EED + rank)
    gw = torch.Generator().manual_seed(0x5EED)
    x = torch.randn(cfg.mini_batch, cfg.sequence_len, cfg.H, generator=g).bfloat16()
    wg = torch.randn(cfg.H, cfg.E, generator=gw).bfloat16()
    we = torch.empty(nlx, 2, cfg.P, cfg.H, dtype=torch.bfloat16)
    for i in range(nlx):  # per expert: keeps the fp32 temporary small at ffn 14336
        we[i] = torch.randn(2, cfg.P, cfg.H, generator=g).bfloat16()
    return x, wg, we


DUMP_BUDGET_BYTES = 64 * 10 ** 6 - (1 << 16)   # all ranks' files together, .npy headers included


def dump_outputs(directory, out, rank, world):
    """This rank's layer output (a CPU tensor in the caller's [mini_batch, seq, d_model] shape) as float32
    `out.npy` (`out_rank<r>.npy` at N > 1).  When the ranks' outputs together would exceed 64 MB, a fixed, seeded sample
    of token rows (the same rows on every rank and in every run, in ascending order) is written as [rows, d_model]."""
    import numpy as np

    a = out.float().numpy()
    flat = a.reshape(-1, a.shape[-1])
    rows = DUMP_BUDGET_BYTES // world // (flat.shape[1] * flat.itemsize)
    if rows < flat.shape[0]:
        a = flat[np.sort(np.random.default_rng(0).choice(flat.shape[0], rows, replace=False))]
    os.makedirs(directory, exist_ok=True)
    path = os.path.join(directory, "out.npy" if world == 1 else f"out_rank{rank}.npy")
    np.save(path, a)
    return path


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"bf16_burst": float(p["bf16_tflops"]), "bf16_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "hbm_gbs": float(p["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json)"}
    # /opt/skills/guides/B200_PROFILING.md fallback figures
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """Samples SM clock / power / throttle reasons through NVML from a host thread while the timed regions run."""

    REASONS = ("SwPowerCap", "HwSlowdown", "HwThermalSlowdown", "SwThermalSlowdown", "HwPowerBrakeSlowdown",
               "ApplicationsClocksSetting")
    NAMES = ("sw_power_cap", "hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "hw_power_brake", "app_clocks")

    def __init__(self, index: int):
        self.samples, self.stop_flag, self.thread, self.ok, self.errors = [], False, None, False, 0
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max_mhz = None

    def _reasons(self):
        nv = self.nv
        for fn in ("nvmlDeviceGetCurrentClocksEventReasons", "nvmlDeviceGetCurrentClocksThrottleReasons"):
            try:
                return int(getattr(nv, fn)(self.h))
            except Exception:
                continue
        return None

    def sample_once(self):
        nv = self.nv
        try:
            mhz = int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        except Exception:
            self.errors += 1
            return
        try:
            watts = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
        except Exception:
            watts = None
        self.samples.append((time.perf_counter(), mhz, self._reasons(), watts))

    def _loop(self):
        while not self.stop_flag:
            self.sample_once()
            time.sleep(0.001)

    def start(self):
        if self.ok:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=1.0)

    def summary(self, windows):
        """`windows`: list of (t0, t1) host-time intervals during which the GPU was running timed work."""
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml_unavailable"], "samples": 0}
        inside = [s for s in self.samples if any(a <= s[0] <= b for a, b in windows)]
        mhz = sorted(s[1] for s in inside)
        nv, bits, known = self.nv, 0, False
        for s in inside:
            if s[2] is not None:
                bits |= s[2]
                known = True
        reasons = []
        for attr, name in zip(self.REASONS, self.NAMES):
            for prefix in ("nvmlClocksEventReason", "nvmlClocksThrottleReason"):
                b = getattr(nv, prefix + attr, None)
                if b is not None:
                    if bits & b:
                        reasons.append(name)
                    break
        if not known:
            reasons.append("reasons_unavailable")
        watts = [s[3] for s in inside if s[3] is not None]
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_mhz_min": mhz[0] if mhz else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(reasons), "samples": len(inside), "power_w_max": max(watts) if watts else None,
                "sampler_errors": self.errors}


def in_tree_native_libs():
    """In-tree shared objects mapped into this process (what the driver records as `native_so_loaded`)."""
    libs = set()
    try:
        for line in open("/proc/self/maps"):
            path = line.rsplit(" ", 1)[-1].strip()
            if path.startswith(ROOT) and ".so" in os.path.basename(path):
                libs.add(os.path.relpath(path, ROOT))
    except OSError:
        pass
    return sorted(libs)


def usable_cpus() -> int:
    """Host threads this process may really use: CPU affinity capped by the cgroup CPU quota (the GPU box shows 128
    CPUs but grants a quota of ~24; running MKL with 128 threads there is 5x slower than with 24-32)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, -(-int(quota) // int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def cpu_forward_sample(cfg, budget_s, steps_hint=3):
    """Prepare the plain torch CPU MoE forward (oracle/torch_moe.py) of the bench workload on the host cores: one
    warm-up forward on a probe of the workload sizes a bounded per-step sample (about `budget_s` seconds in total).
    Returns (torch_moe module, x sample [tokens,H], gate weights, expert weights, EC of the sample, tokens per step)."""
    from oracle import torch_moe

    torch.set_num_threads(usable_cpus())
    x, wg, we = make_inputs(cfg, cfg.E, 0)
    S = cfg.S
    xs = x.reshape(S, cfg.H)
    probe = min(S, 512)
    ec_of = lambda n: cfg.replace(sequence_len=n, mini_batch=1).EC  # noqa: E731
    t0 = time.perf_counter()
    torch_moe.moe_forward_cpu(xs[:probe].contiguous(), wg, we, k=cfg.k, EC=ec_of(probe), act=cfg.hidden_act)
    t_probe = time.perf_counter() - t0
    per_tok = t_probe / probe
    tokens = int(budget_s / ((steps_hint + 1) * per_tok)) // 128 * 128
    tokens = max(128, min(S, tokens))
    return torch_moe, xs[:tokens].contiguous(), wg, we, ec_of(tokens), tokens


def run_reference_arm(args, rank, world):
    """The reference arm: the CPU implementation of the path (oracle port: plain torch CPU MoE forward), all host threads."""
    if rank != 0:
        return 0
    cfg = BASELINE_CONFIGS[args.config]
    budget = float(os.environ.get("FM_BENCH_CPU_BUDGET_S", "120"))
    torch_moe, xsub, wg, we, ec, tokens = cpu_forward_sample(cfg, budget, steps_hint=args.steps + args.warmup)
    for _ in range(max(0, args.warmup)):
        torch_moe.moe_forward_cpu(xsub, wg, we, k=cfg.k, EC=ec, act=cfg.hidden_act)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        torch_moe.moe_forward_cpu(xsub, wg, we, k=cfg.k, EC=ec, act=cfg.hidden_act)
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    tps = tokens / dt
    cores = torch.get_num_threads()
    sample = f"{tokens} of {cfg.S} tokens per step through all {cfg.E} experts (capacity scaled), plain torch CPU forward"
    line = {"impl": "reference", "metric": "moe_layer_fwd_tokens_per_s", "value": tps, "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": config_dict(args.config, cfg, args.gpus),
            "note": "the reference has no CPU path and cannot be built here; this arm is the oracle port "
                    "(oracle/torch_moe.py) on the host cores",
            "cpu_baseline": {"value": tps, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": tps, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "native_so_mapped": in_tree_native_libs()}
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------------------------
class Env:
    def __init__(self, rank, world, dev):
        self.rank, self.world, self.dev = rank, world, dev

    def barrier(self):
        import torch.distributed as dist

        torch.cuda.synchronize(self.dev)
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, v):
        import torch.distributed as dist

        if self.world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v):
        import torch.distributed as dist

        if self.world == 1:
            return v
        t = torch.tensor([v], dtype=torch.int64, device=self.dev)
        dist.all_reduce(t)
        return int(t.item())


def parity_check(env, ctx, cfg, xd, wgd, wed, n_tokens):
    """One extra forward on SCALED weights (non-degenerate softmax, O(1) activations), every rank's output and top-k
    indices against the CPU oracle on a seeded sample of its tokens.  All experts' weights are all-gathered (the oracle's
    world composition, SURVEY.md Appendix A.8); the oracle's cost is per sampled token, so full-size shapes stay cheap."""
    import numpy as np
    import torch.distributed as dist

    from oracle import moe_oracle as mo

    scale = cfg.H ** -0.5
    wgd.mul_(scale)
    wed.mul_(scale)
    out = ctx.forward(xd, wgd, wed)
    ctx.synchronize()
    topk = ctx.read("topk_idx")
    if env.world > 1:
        wes = [torch.empty_like(wed) for _ in range(env.world)]
        dist.all_gather(wes, wed)
        full = torch.cat([w.cpu() for w in wes], dim=0)
        del wes
    else:
        full = wed.cpu()
    up, down = mo.split_expert_weights(mo.to_bits(full))
    del full
    rng = np.random.default_rng(1234 + env.rank)
    sample = np.sort(rng.choice(cfg.S, size=min(n_tokens, cfg.S), replace=False)).astype(np.int32)
    xb = mo.to_bits(xd.cpu().reshape(cfg.S, cfg.H))
    wg_eff = mo.gate_weights_effective(mo.to_bits(wgd.cpu()), cfg.E, cfg.H)
    ref = mo.forward_sample(xb, wg_eff, up, down, sample, k=cfg.k, EC=cfg.EC, act=cfg.hidden_act)
    mism = (topk != ref.topk_idx).any(axis=1)
    hard = int((mism & ~ref.ambiguous).sum())
    got = mo.bits_to_f32(mo.to_bits(out.cpu().reshape(cfg.S, cfg.H))[sample]).astype(np.float64)
    ok_rows = ~mism[sample]
    finite = bool(np.isfinite(got).all())

    def rel_frobenius(want_bits):
        want = mo.bits_to_f32(want_bits).astype(np.float64)
        if not finite:
            return float("inf")
        return float(np.linalg.norm(got[ok_rows] - want[ok_rows]) / max(np.linalg.norm(want[ok_rows]), 1e-30))

    relf_plain = rel_frobenius(ref.out)
    # Router weights: the bf16 rounding of a gate probability hangs on the last bits of its fp32 logit, i.e. on the
    # summation order of the router GEMM (sequential in the oracle, tensor-core tiles on the device from 17 experts, as in
    # the reference).  They must agree to <= 1 bf16 ulp; where some differ, the FFN + combine arithmetic is judged with
    # the oracle evaluated on the DEVICE's router weights, and the plain end-to-end figure is reported next to it.
    dev_w = np.ascontiguousarray(ctx.read("topk_w")).view(np.uint16).reshape(cfg.S, cfg.k)[sample]
    dev_mcw = np.ascontiguousarray(ctx.read("mcw"), dtype=np.float32).reshape(cfg.S)[sample]
    ulps = mo.router_weight_ulps(dev_w, ref, sample)[ok_rows]
    flips = int((ulps > 0).sum())
    max_ulp = int(ulps.max()) if ulps.size else 0
    relf = relf_plain
    if flips and finite:
        ref_w = mo.forward_sample(xb, wg_eff, up, down, sample, k=cfg.k, EC=cfg.EC, act=cfg.hidden_act,
                                  topk_w_given=dev_w, mcw_given=dev_mcw)
        relf = rel_frobenius(ref_w.out)
    ok = finite and hard == 0 and max_ulp <= 1 and relf <= 1e-3
    res = torch.tensor([relf if finite else 1e30, float(hard), float(int(mism.sum())), 0.0 if ok else 1.0,
                        relf_plain if finite else 1e30, float(flips), float(max_ulp)], dtype=torch.float64, device=env.dev)
    if env.world > 1:
        allr = [torch.empty_like(res) for _ in range(env.world)]
        dist.all_gather(allr, res)
        allr = torch.stack(allr).cpu()
    else:
        allr = res.cpu().unsqueeze(0)
    return {"n_ranks": env.world, "tokens_checked": int(len(sample)) * env.world, "tokens_routed_per_rank": cfg.S,
            "relF_max": float(allr[:, 0].max()), "topk_mismatch_unambiguous": int(allr[:, 1].sum()),
            "topk_mismatch_ambiguous": int(allr[:, 2].sum() - allr[:, 1].sum()), "tolerance_relF": 1e-3,
            "router_weights_off_by_one_bf16_ulp": int(allr[:, 5].sum()), "router_weight_max_ulp": int(allr[:, 6].max()),
            "relF_max_with_oracle_router_weights": float(allr[:, 4].max()),
            "rule": "top-k indices exact on unambiguous tokens; router weights within 1 bf16 ulp of the oracle's; "
                    "relF <= tolerance against the oracle's FFN + combine on the device's router weights (the plain "
                    "end-to-end relF, which includes the 0.4 % steps of those ulps, is reported next to it)",
            "inputs": "x N(0,1), gate/expert weights N(0,1)*d_model^-0.5, seeded; checked against oracle/moe_oracle.c",
            "ok": bool(allr[:, 3].sum() == 0)}


def run_config(env, name, steps, warmup, sampler, *, e2e=True, parity_tokens=0, out_in_slab=True, keep_output=False):
    """Measure one configuration; returns a dict with the device-resident and end-to-end numbers (and, with
    `keep_output`, a CPU copy of the last timed step's output as "output")."""
    from flashmoe_b200.runtime import MoEContext

    rank, world, dev = env.rank, env.world, env.dev
    cfg = BASELINE_CONFIGS[name]
    nlx = cfg.num_local_experts(world)
    ctx = MoEContext(cfg, rank=rank, world=world, device=dev.index, timeout_ms=30000)
    x, wg, we = make_inputs(cfg, nlx, rank)
    xd, wgd, wed = x.to(dev), wg.to(dev), we.to(dev)
    del we
    # at N > 1 peers add their expert outputs into this rank's symmetric accumulator; asking for the output THERE
    # (ctx.output_buffer()) saves the final copy into a caller tensor.  N == 1 accumulates straight into `out`.
    out = ctx.output_buffer() if (out_in_slab and world > 1) else torch.empty_like(xd)

    for _ in range(warmup):
        ctx.forward(xd, wgd, wed, out=out)
    env.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = ctx.launch_count
    t_host0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        ctx.forward(xd, wgd, wed, out=out)
    e1.record()
    env.barrier()
    t_host1 = time.perf_counter()
    ctx.check()
    launches = ctx.launch_count - launches0
    ms = env.max_over_ranks(e0.elapsed_time(e1) / steps)
    windows = [(t_host0, t_host1)]
    rows_exec = int(ctx.read("recv_cnt").sum())  # token-expert pairs this rank's experts executed (after drops)
    rows_total = env.sum_over_ranks(rows_exec)
    res = {"name": name, "ms": ms, "launches": launches, "rows_total": rows_total, "cfg": cfg, "nlx": nlx,
           "out_buffer": "symmetric accumulator (MoEContext.output_buffer)" if (out_in_slab and world > 1) else "caller tensor"}
    if keep_output:  # copied now: the end-to-end arm and the parity forward below overwrite `out` at N > 1
        res["output"] = out.cpu()

    if e2e:
        # end-to-end arm: host activations in, host output back, EVERY step; three steps in flight (public API:
        # MoEContext.submit_host / wait_host -> fm_host_submit / fm_host_wait), so copies overlap kernels
        depth = 3
        x_pins = [x.clone().pin_memory() for _ in range(depth)]
        out_pins = [torch.empty_like(x).pin_memory() for _ in range(depth)]
        e2e_steps = steps

        def run_e2e(n):
            tickets = []
            for i in range(n):
                if len(tickets) == depth:
                    ctx.wait_host(tickets.pop(0))
                tickets.append(ctx.submit_host(x_pins[i % depth], wgd, wed, out_pins[i % depth]))
            for t in tickets:
                ctx.wait_host(t)

        run_e2e(depth + 2)
        env.barrier()
        t0 = time.perf_counter()
        run_e2e(e2e_steps)
        t1 = time.perf_counter()
        env.barrier()
        res["e2e_ms"] = env.max_over_ranks((t1 - t0) / e2e_steps * 1e3)
        windows.append((t0, t1))
        # the blocking single call (H2D -> kernel -> D2H -> wait), for context
        ctx.forward_host(x_pins[0], wgd, wed, out_pins[0])
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(5):
            ctx.forward_host(x_pins[0], wgd, wed, out_pins[0])
        res["e2e_blocking_ms"] = env.max_over_ranks((time.perf_counter() - t0) / 5 * 1e3)
        res["e2e_steps"], res["e2e_depth"] = e2e_steps, depth
        del x_pins, out_pins
    res["clocks"] = sampler.summary(windows)
    if parity_tokens > 0:
        res["parity"] = parity_check(env, ctx, cfg, xd, wgd, wed, parity_tokens)
    env.barrier()
    ctx.close()
    del xd, wgd, wed, out
    torch.cuda.empty_cache()
    env.barrier()
    return res


def derived(res, world, peaks, steps):
    """Roofline figures of one measured configuration (SURVEY.md section 8d)."""
    cfg, ms, rows_total, nlx = res["cfg"], res["ms"], res["rows_total"], res["nlx"]
    S, H, P, E = cfg.S, cfg.H, cfg.P, cfg.E
    flops_rank = 4.0 * (rows_total / world) * H * P + 2.0 * S * H * E  # 4*R*H*P + 2*S*H*E per rank
    achieved = flops_rank / (ms * 1e-3) / 1e12
    timed_s = steps * ms * 1e-3
    kind = "burst" if timed_s < 1.0 else "sustained"
    peak = peaks["bf16_burst"] if kind == "burst" else peaks["bf16_sustained"]
    hbm_alg = S * H * 2 * 2 + E * H * 2 + nlx * 2 * H * P * 2 + (rows_total / world) * (2 * H + 2 * P) * 2
    nvl_bytes = 2.0 * (rows_total / world) * (1.0 - 1.0 / world) * H * 2  # per GPU per direction: rows out + outputs back
    nvl_floor_ms = nvl_bytes / 770e9 * 1e3   # measured peer-copy bandwidth of this pool (B200_PROFILING.md)
    flop_floor_ms = flops_rank / (peak * 1e12) * 1e3
    return {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "peak_kind": f"{kind} cuBLAS bf16 ({'timed region %.3f s' % timed_s}), {peaks['source']}",
            "frac_of_burst": achieved / peaks["bf16_burst"], "frac_of_sustained": achieved / peaks["bf16_sustained"],
            "algorithmic_flops_per_launch": flops_rank, "algorithmic_hbm_bytes_per_launch": hbm_alg,
            "hbm_frac_of_measured_copy": hbm_alg / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
            "nvlink_bytes_per_dir_per_gpu": nvl_bytes, "nvlink_floor_ms_at_770GBs": nvl_floor_ms,
            "flop_floor_ms": flop_floor_ms, "frac_of_slower_floor": max(nvl_floor_ms, flop_floor_ms) / ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=32)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="B", choices=sorted(BASELINE_CONFIGS))
    ap.add_argument("--sweeps", default=os.environ.get("FM_BENCH_SWEEPS"),
                    help="comma-separated extra configs measured with reduced steps and appended as \"sweeps\" (default: the "
                         "BASELINE.json multi-GPU configs at 8 GPUs -- C, the token sweep, the expert sweep -- the expert sweep "
                         "at 4 GPUs, none otherwise; 'none' disables)")
    ap.add_argument("--sweep-steps", type=int, default=20)
    ap.add_argument("--parity-tokens", type=int, default=int(os.environ.get("FM_BENCH_PARITY_TOKENS", "256")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's layer output as float32 .npy files into DIR (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path; the reference arm times a CPU sample whose size is set by timing")
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            print(f"bench.py: --gpus {args.gpus} needs a torchrun launch with {args.gpus} ranks", file=sys.stderr)
            return 2
        args.gpus = world
    if args.impl == "reference":
        return run_reference_arm(args, rank, world)
    if args.warmup < 3:
        args.warmup = 3

    if not torch.cuda.is_available():
        print("bench.py: no CUDA device; the MoE forward path has no CPU fallback", file=sys.stderr)
        return 3
    torch.cuda.set_device(local % torch.cuda.device_count())
    dev = torch.device("cuda", torch.cuda.current_device())
    import torch.distributed as dist

    if world > 1:
        dist.init_process_group(backend="cpu:gloo,cuda:nccl", rank=rank, world_size=world, device_id=dev)
    env = Env(rank, world, dev)
    peaks = load_peaks()
    sampler = ClockSampler(dev.index)
    sampler.start()

    name = args.config
    cfg = BASELINE_CONFIGS[name]
    res = run_config(env, name, args.steps, args.warmup, sampler, e2e=not args.no_e2e, parity_tokens=args.parity_tokens,
                     keep_output=bool(args.dump_outputs))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res.pop("output"), rank, world)
    S, ms = cfg.S, res["ms"]
    roof = derived(res, world, peaks, args.steps)
    # DRAM traffic per launch comes from a committed `ncu --set full` capture; it describes one configuration at one N only
    roof["traffic"] = None
    prof = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if os.path.exists(prof):
        try:
            pj = json.load(open(prof))
            if pj.get("config", "B") == name and int(pj.get("n_gpus", 1)) == world:
                roof["traffic"] = pj.get("dram_bytes_per_launch")
                roof["traffic_source"] = pj.get("source")
        except Exception:
            pass
    cd = config_dict(name, cfg, world)
    line = {
        "metric": "moe_layer_fwd_tokens_per_s", "value": world * S / (ms * 1e-3), "unit": "tokens/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": cd,
        "run": {"token_expert_pairs_executed": res["rows_total"], "output_buffer": res["out_buffer"],
                "l2": "no explicit flush: the per-step working set (expert weights + activations/staging, >= 250 MB per "
                      "rank for config B) exceeds the 126 MB L2"},
        "roofline": roof, "gpu_launches": res["launches"], "clocks": res["clocks"], "native_so_mapped": in_tree_native_libs(),
    }
    if "e2e_ms" in res:
        line["e2e"] = {"value": world * S / (res["e2e_ms"] * 1e-3), "unit": "tokens/s", "h2d_bytes_per_step": S * cfg.H * 2,
                       "d2h_bytes_per_step": S * cfg.H * 2, "ms_per_step": res["e2e_ms"], "steps": res["e2e_steps"],
                       "pipeline_depth": res["e2e_depth"], "blocking_call_ms": res["e2e_blocking_ms"],
                       "api": "MoEContext.submit_host/wait_host -> fm_host_submit/fm_host_wait (pinned host activations in, "
                              "pinned host output back every step, device-resident weights; copies overlap kernels)"}
    if "parity" in res:
        line["parity_check"] = res["parity"]

    if args.sweeps is None:   # BASELINE.json: configs[2..4] are quoted on 8 (and 4) GPUs
        args.sweeps = {8: "C,D1k,D4k,D16k,D64k,E8,E16,E32,E64,E128", 4: "E8,E16,E32,E64,E128"}.get(world, "")
    sweeps = [s for s in args.sweeps.split(",") if s and s != "none"]
    if sweeps:
        line["sweeps"] = []
        t_sweeps0, sweep_budget = time.perf_counter(), float(os.environ.get("FM_BENCH_SWEEP_BUDGET_S", "240"))
        for sname in sweeps:
            if sname not in BASELINE_CONFIGS or BASELINE_CONFIGS[sname].E % world:
                line["sweeps"].append({"config": sname, "skipped": "num_experts not divisible by the world size"})
                continue
            # (a collective decision: ranks that disagreed about skipping would wait for each other forever)
            if env.max_over_ranks(time.perf_counter() - t_sweeps0) > sweep_budget:
                line["sweeps"].append({"config": sname, "skipped": "sweep time budget exhausted"})
                continue
            try:
                r = run_config(env, sname, args.sweep_steps, max(3, args.sweep_steps // 4), sampler, e2e=False,
                               parity_tokens=int(os.environ.get("FM_BENCH_SWEEP_PARITY_TOKENS", "0")))
                rf = derived(r, world, peaks, args.sweep_steps)
                c = r["cfg"]
                entry = {"config": sname, "workload": CONFIG_DESCRIPTIONS[sname], "tokens_per_s": world * c.S / (r["ms"] * 1e-3),
                         "ms_per_step": r["ms"], "steps": args.sweep_steps, "tflops_per_gpu": rf["achieved"],
                         "frac_of_burst": rf["frac_of_burst"], "frac_of_sustained": rf["frac_of_sustained"],
                         "nvlink_floor_ms_at_770GBs": rf["nvlink_floor_ms_at_770GBs"], "flop_floor_ms_burst": rf["algorithmic_flops_per_launch"] / (peaks["bf16_burst"] * 1e12) * 1e3,
                         "token_expert_pairs_executed": r["rows_total"], "clocks": r["clocks"]}
                if "parity" in r:
                    entry["parity_check"] = r["parity"]
                line["sweeps"].append(entry)
            except Exception as exc:  # keep the headline line even if a sweep point fails
                line["sweeps"].append({"config": sname, "error": str(exc)[:300]})
                break
    sampler.stop()

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        budget = float(os.environ.get("FM_BENCH_CPU_BUDGET_S", "20"))
        torch_moe, xsub, wg_c, we_c, ec, tokens = cpu_forward_sample(cfg, budget)
        iters = 3
        t0 = time.perf_counter()
        for _ in range(iters):
            torch_moe.moe_forward_cpu(xsub, wg_c, we_c, k=cfg.k, EC=ec, act=cfg.hidden_act)
        dt = (time.perf_counter() - t0) / iters
        line["cpu_baseline"] = {"value": tokens / dt, "unit": "tokens/s", "cores": torch.get_num_threads(), "kind": "port",
                                "sample": f"{iters} forwards of {tokens} of {S} tokens (plain torch CPU MoE forward, "
                                          f"oracle/torch_moe.py; {os.cpu_count()} host CPUs visible, {usable_cpus()} usable under the cgroup quota)"}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line), flush=True)
    pc = line.get("parity_check")
    return 0 if (pc is None or pc["ok"]) else 4


if __name__ == "__main__":
    sys.exit(main())
