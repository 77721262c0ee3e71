"""bench.py's output contract: on the CPU-only legs the reference arm prints one JSON line with the agreed keys, and the
multi-rank convention (only rank 0 works and prints) holds; on the GPU, `--steps` sets the timed steps and
`--dump-outputs` writes the layer output the timed path computed."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, args=()):
    env = dict(os.environ)
    env.update({"FM_BENCH_CPU_BUDGET_S": "2"})  # shrink the per-step sample so the test stays at seconds
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                           *args], capture_output=True, text=True, env=env, cwd=ROOT, timeout=300)


def test_reference_arm_json_line():
    res = _run()
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "moe_layer_fwd_tokens_per_s" and d["unit"] == "tokens/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["dtype"] == "bf16" and d["data"] == "synthetic"
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "tokens" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    # the same `config` object as the GPU arm prints (the driver compares the two arms' configs) ...
    sys.path.insert(0, ROOT)
    import bench

    assert d["config"] == bench.config_dict("B", bench.BASELINE_CONFIGS["B"], 1)
    # ... and the product's native library is never mapped into the reference arm's process
    assert d["native_so_mapped"] == [] or all("flashmoe" not in s for s in d["native_so_mapped"]), d["native_so_mapped"]


def test_every_baseline_config_is_selectable():
    sys.path.insert(0, ROOT)
    import bench

    assert set(bench.BASELINE_CONFIGS) >= {"A", "B", "C", "D1k", "D4k", "D16k", "D64k", "E8", "E16", "E32", "E64", "E128"}
    for name, cfg in bench.BASELINE_CONFIGS.items():
        assert bench.config_dict(name, cfg, 8)["workload"].startswith("configs[")


def test_reference_arm_non_zero_ranks_exit_quietly():
    res = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, args=("--gpus", "2"))
    assert res.returncode == 0 and not [l for l in res.stdout.splitlines() if l.startswith("{")]


def test_usable_cpus_respects_affinity():
    sys.path.insert(0, ROOT)
    import bench

    n = bench.usable_cpus()
    assert 1 <= n <= (os.cpu_count() or 1)


class _FakeEnv:
    world, rank = 1, 0

    def __init__(self):
        import torch

        self.dev = torch.device("cpu")


class _OracleBackedContext:
    """Stands in for MoEContext in bench.parity_check: `forward` is the oracle itself, optionally with some router weights
    moved by `ulp` bf16 ulps (and the output recomputed with them), the way a different summation order of the router GEMM
    would."""

    def __init__(self, cfg, flip_tokens=(), ulp=1):
        self.cfg, self.flip_tokens, self.ulp, self.bufs = cfg, list(flip_tokens), ulp, {}

    def forward(self, xd, wgd, wed):
        import numpy as np
        import torch

        from oracle import moe_oracle as mo

        cfg = self.cfg
        xb = mo.to_bits(xd.reshape(cfg.S, cfg.H))
        wg_eff = mo.gate_weights_effective(mo.to_bits(wgd), cfg.E, cfg.H)
        up, down = mo.split_expert_weights(mo.to_bits(wed))
        ref = mo.forward(xb, wg_eff, up, down, k=cfg.k, EC=cfg.EC, act=cfg.hidden_act)
        topk_w = ref.gate_out[np.arange(cfg.S)[:, None], ref.topk_idx].astype(np.uint16)
        out = ref.out.copy()
        if self.flip_tokens:
            topk_w[self.flip_tokens, 0] += self.ulp
            smp = np.asarray(sorted(self.flip_tokens), dtype=np.int32)
            alt = mo.forward_sample(xb, wg_eff, up, down, smp, k=cfg.k, EC=cfg.EC, act=cfg.hidden_act,
                                    topk_w_given=topk_w[smp], mcw_given=ref.mcw[smp])
            out[smp] = alt.out
        self.bufs = {"topk_idx": ref.topk_idx, "topk_w": topk_w, "mcw": ref.mcw}
        return torch.from_numpy(out.view(np.int16)).view(torch.bfloat16).reshape(1, cfg.S, cfg.H)

    def synchronize(self):
        pass

    def read(self, name):
        return self.bufs[name]


def _parity_case(flip_tokens, ulp):
    import torch

    sys.path.insert(0, ROOT)
    import bench
    from flashmoe_b200.config import MoEConfig

    cfg = MoEConfig(num_experts=8, expert_top_k=2, sequence_len=128, hidden_size=64, intermediate_size=128)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(1, cfg.S, cfg.H, generator=g).bfloat16()
    wg = torch.randn(cfg.H, cfg.E, generator=g).bfloat16()
    we = torch.randn(cfg.E, 2, cfg.P, cfg.H, generator=g).bfloat16()
    ctx = _OracleBackedContext(cfg, flip_tokens, ulp)
    return bench.parity_check(_FakeEnv(), ctx, cfg, x, wg, we, cfg.S)


def test_parity_check_rule_on_router_weight_ulps():
    """bench.parity_check: identical router weights -> plain comparison; weights one bf16 ulp off -> still ok, judged on
    the device's weights, flips counted, plain relF reported next to it; two ulps off -> not ok."""
    same = _parity_case([], 1)
    assert same["ok"] and same["router_weights_off_by_one_bf16_ulp"] == 0 and same["relF_max"] == 0.0
    one = _parity_case([5, 17, 99], 1)
    assert one["ok"] and one["router_weights_off_by_one_bf16_ulp"] == 3 and one["router_weight_max_ulp"] == 1
    assert one["relF_max"] == 0.0 and one["relF_max_with_oracle_router_weights"] > 0.0
    two = _parity_case([5], 2)
    assert not two["ok"] and two["router_weight_max_ulp"] == 2


def test_roofline_block_arithmetic():
    """bench.derived: achieved = algorithmic FLOPs per launch / step time; burst peak for timed regions under a second,
    sustained above; the NVLink figure is zero on one GPU."""
    sys.path.insert(0, ROOT)
    import bench

    cfg = bench.BASELINE_CONFIGS["B"]
    peaks = {"bf16_burst": 1696.0, "bf16_sustained": 1429.2, "hbm_gbs": 6584.5, "source": "test"}
    res = {"cfg": cfg, "ms": 0.14, "rows_total": 8192, "nlx": 8}
    r = bench.derived(res, 1, peaks, 200)
    flops = 4.0 * 8192 * cfg.H * cfg.P + 2.0 * cfg.S * cfg.H * cfg.E
    assert abs(r["algorithmic_flops_per_launch"] - flops) < 1
    assert abs(r["achieved"] - flops / 0.14e-3 / 1e12) < 1e-6
    assert r["peak"] == 1696.0 and abs(r["frac"] - r["achieved"] / 1696.0) < 1e-12 and "burst" in r["peak_kind"]
    assert r["nvlink_bytes_per_dir_per_gpu"] == 0.0
    long = bench.derived(res, 1, peaks, 20000)   # 2.8 s of timed region
    assert long["peak"] == 1429.2 and "sustained" in long["peak_kind"]
    r8 = bench.derived({"cfg": cfg, "ms": 0.18, "rows_total": 8 * 8192, "nlx": 1}, 8, peaks, 20)
    assert abs(r8["nvlink_bytes_per_dir_per_gpu"] - 2.0 * 8192 * (7 / 8) * cfg.H * 2) < 1
    assert abs(r8["algorithmic_flops_per_launch"] - flops) < 1   # weak scaling: per-GPU work fixed


def test_dump_outputs_whole_and_sampled(tmp_path):
    """bench.dump_outputs: float32 in the caller's shape while all ranks' files fit in 64 MB; above that the same seeded
    rows on every rank and in every run, within the budget."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    g = torch.Generator().manual_seed(0)
    small = torch.randn(1, 256, 64, generator=g).bfloat16()
    path = bench.dump_outputs(str(tmp_path / "a"), small, 0, 1)
    assert os.path.basename(path) == "out.npy"
    a = np.load(path)
    assert a.dtype == np.float32 and a.shape == (1, 256, 64) and (a == small.float().numpy()).all()

    big = torch.randn(2, 8192, 1024, generator=g).bfloat16()   # 4 ranks x 64 MiB of float32 > 64 MB
    paths = [bench.dump_outputs(str(tmp_path / "b"), big, r, 4) for r in range(4)]
    assert [os.path.basename(p) for p in paths] == [f"out_rank{r}.npy" for r in range(4)]
    assert sum(os.path.getsize(p) for p in paths) <= 64 * 10 ** 6
    rows = bench.DUMP_BUDGET_BYTES // 4 // (1024 * 4)
    idx = np.sort(np.random.default_rng(0).choice(2 * 8192, rows, replace=False))
    b = np.load(paths[0])
    assert b.dtype == np.float32 and b.shape == (rows, 1024)
    assert (b == big.float().numpy().reshape(-1, 1024)[idx]).all()
    again = bench.dump_outputs(str(tmp_path / "c"), big, 0, 4)
    assert (np.load(again) == b).all()


@pytest.mark.parametrize("args", [("--steps", "0"), ("--impl", "reference", "--dump-outputs", "unused")])
def test_bench_rejects_arguments_it_cannot_honour(args, tmp_path):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         cwd=tmp_path, timeout=300)
    assert res.returncode == 2 and "error" in res.stderr and not os.listdir(tmp_path)


@pytest.mark.gpu
def test_gpu_arm_steps_and_dumped_output(tmp_path):
    """`--steps 3` runs three timed launches and three end-to-end steps; `--dump-outputs` writes config B's layer output
    of the last timed step, which matches the CPU oracle on bench.py's own seeded inputs."""
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench
    from oracle import moe_oracle as mo
    from tests.util import check_output, run_oracle

    out_dir = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3",
                          "--no-cpu-baseline", "--parity-tokens", "0", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert res.returncode == 0, res.stderr[-4000:]
    d = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 3 and d["gpu_launches"] == 3 and d["e2e"]["steps"] == 3
    assert sorted(os.listdir(out_dir)) == ["out.npy"]
    got = np.load(out_dir / "out.npy")
    cfg = bench.BASELINE_CONFIGS["B"]
    assert got.dtype == np.float32 and got.shape == (cfg.mini_batch, cfg.sequence_len, cfg.H)
    x, wg, we = bench.make_inputs(cfg, cfg.E, 0)
    ref = run_oracle(cfg, x, wg, we)
    got_bits = mo.f32_to_bits(got.reshape(cfg.S, cfg.H))   # exact: the values are bf16
    # the dump carries no routing tables: compare all rows the oracle does not flag as ambiguous
    check_output(got_bits, ref.out, rows_ok=~ref.ambiguous, what="dumped output vs oracle")
