"""CPU-side checks of the measurement harness (no GPU): the nvidia-smi clock / throttle parser of bench.py, the
reference arm's JSON line (contract keys, bounded per-step sample, every host thread even under torchrun's
OMP_NUM_THREADS=1), the --dump-outputs sample, and the bucket schedule of the data-parallel gradient exchange as a
property over random tapes."""
import json
import os
import random
import subprocess
import sys

import numpy as np

import icap_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pkg = icap_loader.load()


def _bench():
    import importlib
    return importlib.import_module("bench")


def test_clock_sampler_parses_nvidia_smi_lines():
    b = _bench()
    s = b.ClockSampler(0)
    s.proc, s.t = _FakeProc(), _FakeThread()
    s.lines = [
        "0, 1965, 1965, 412.3, 0x0000000000000000, Not Active, Not Active, Not Active, Not Active\n",
        "0, 1950, 1965, 998.1, 0x0000000000000004, Not Active, Not Active, Not Active, Active\n",
        "0, 1965, 1965, 640.0, 0x0000000000000000, Not Active, Not Active, Not Active, Not Active\n",
        "garbage line\n",
        "0, [N/A], 1965, 1.0, 0x0, Not Active, Not Active, Not Active, Not Active\n",
    ]
    out = s.stop()
    assert out == {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": ["sw_power_cap"], "samples": 3}
    s.lines = ["0, 1200, 1965, 300.0, 0x8, Active, Active, Not Active, Not Active\n"]
    out = s.stop()
    assert out["reasons"] == ["hw_slowdown", "hw_thermal_slowdown"] and out["sm_mhz"] == 1200.0


def test_clock_sampler_without_nvidia_smi():
    b = _bench()
    s = b.ClockSampler(0)            # never started: no process
    assert s.stop()["reasons"] == ["nvidia-smi unavailable"]


class _FakeProc:
    def terminate(self):
        pass


class _FakeThread:
    def join(self, timeout=None):
        pass


def test_workload_table_matches_baseline_json():
    """bench.py's workloads are BASELINE.json's configs (metric name and the model dimensions they are quoted on)."""
    b = _bench()
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "train samples/sec" in base["metric"] and "beam-5 captions/sec" in base["metric"] and len(base["configs"]) == 5
    assert "batch 256" in base["configs"][1] and b.WORKLOADS["modelA"]["per_gpu"] == 256
    assert "batch 512" in base["configs"][2] and b.DECODE_BATCH == 512
    assert "global batch 2048" in base["configs"][3] and "2048" in b.WORKLOADS["global2048"]["text"]
    assert "d_model=1024" in base["configs"][4] and b.MODEL_C["encode_input_size"] == 1024 and b.MODEL_C["num_vocab"] == 30000
    assert set(b.WORKLOADS) == {"modelA", "global2048", "modelC"}
    for name, wl in b.WORKLOADS.items():
        assert wl["scaling"] in ("weak", "strong")
        assert wl["kw"]["encode_dim_features"] == 2048 and wl["kw"]["encode_dim_positions"] == 84
        # model FLOPs per sample: 3 x forward matmul FLOPs; sanity bound against the parameter count (6 * params * tokens
        # counts every weight once per token; region rows and caption rows differ, so only an order-of-magnitude check)
        assert 1.0 < wl["gflop_train"] < 200.0 and wl["gflop_beam5"] < wl["gflop_train"]
    assert b.MODEL_B["encode_num_heads"] == 32 and b.MODEL_B["decode_num_blocks"] == 5      # core/config.py:87-129


def test_reference_arm_line_contract():
    """`bench.py --impl reference`: one JSON line with the contract's keys; all host threads although torchrun-style
    OMP_NUM_THREADS=1 is exported; non-zero ranks print nothing and exit 0."""
    env = dict(os.environ, OMP_NUM_THREADS="1")
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
           "--ref-batch", "4"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "train_samples_per_sec" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["gpu_launches"] == 0
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["value"] == d["value"]
    assert cb["cores"] == len(os.sched_getaffinity(0))
    assert d["config"]["workload"].startswith("configs[1]") and d["config"]["global_batch"] == 4
    r = subprocess.run(cmd, env=dict(env, RANK="1", WORLD_SIZE="2"), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_bounds_its_sample_by_the_step_count():
    """A large --steps shrinks the batch of each step (about 3 minutes of CPU work in total) instead of running for hours."""
    b = _bench()
    wl = b.WORKLOADS["modelA"]
    rate = 110.0
    for steps, warm in ((20, 5), (100, 5), (1000, 3)):
        fit = int(rate * 180.0 / (steps + max(1, warm)))
        bs = max(4, min(wl["ref_batch"], fit // 4 * 4))
        assert 4 <= bs <= 256 and bs % 4 == 0
        assert bs * (steps + warm) / rate <= 200.0 or bs == 4
    assert max(4, min(256, int(110.0 * 180.0 / 25) // 4 * 4)) == 256       # the driver's --steps 20 --warmup 5: full batch


def test_output_sample_is_seeded_float32_and_bounded(monkeypatch):
    """--dump-outputs: the same model gives the same arrays (fixed sample positions), every array is float32, small
    parameters are kept whole, and every workload's dump stays under 64 MB."""
    import math

    import torch
    b = _bench()
    kw = dict(num_vocab=97, max_length=6, encode_dim_positions=12, encode_dim_features=300, output_name="x",
              encode_input_size=32, encode_q_k_dim=32, encode_v_dim=32, encode_hidden_size=64, encode_num_blocks=1,
              encode_num_heads=4, dim_word_embedding=32, decode_input_size=32, decode_q_k_dim=32, decode_v_dim=32,
              decode_hidden_size=64, decode_num_blocks=1, decode_num_heads=4)
    torch.manual_seed(0)
    m = pkg.Transformer(device=None, **kw)
    with monkeypatch.context() as mp:
        mp.setattr(b, "DUMP_SAMPLE", 1000)         # below the 300 x 32 input projection: exercises the sampled branch
        a1 = b.output_sample(torch.tensor(2.5), m.named_parameters())
        a2 = b.output_sample(torch.tensor(2.5), m.named_parameters())
    params = dict(m.named_parameters())
    assert set(a1) == {"loss"} | {"param." + n for n in params} and float(a1["loss"][0]) == 2.5
    for name, arr in a1.items():
        assert arr.dtype == np.float32 and np.array_equal(arr, a2[name]), name
        if name != "loss":
            q = params[name[len("param."):]]
            assert arr.shape == ((q.numel(),) if q.numel() <= 1000 else (1000,)), name
            if q.numel() <= 1000:
                assert np.array_equal(arr, q.detach().reshape(-1).numpy()), name
            else:
                assert np.isin(arr, q.detach().reshape(-1).numpy()).all(), name
    assert any(q.numel() > 1000 for q in params.values())
    for wl in b.WORKLOADS.values():
        shapes = pkg.param_layout(pkg.ModelConfig(**wl["kw"])).values()
        assert 4 * (1 + sum(min(math.prod(s), b.DUMP_SAMPLE) for s in shapes)) <= 64 << 20


def test_grad_buckets_property_random_tapes():
    """Every element of the flat gradient buffer is handed out exactly once, in descending contiguous slices, whatever
    the closure order / offsets / `None` reports are; no slice is fired before every closure that writes into it (i.e.
    every closure with lo >= slice.lo that reports an offset) has run."""
    rng = random.Random(1234)
    for _ in range(300):
        total = rng.randint(1, 5000)
        bucket = rng.randint(1, 1500)
        tail = rng.choice([None, rng.randint(1, bucket)])
        tail_below = rng.choice([None, rng.randint(0, total)])
        plan = pkg.GradBuckets(total, bucket, tail_elems=tail, tail_below=tail_below)
        # a tape: offsets mostly descending, with repeats, out-of-order (higher) values and None reports
        los, cur = [], total
        for _ in range(rng.randint(0, 40)):
            kind = rng.random()
            if kind < 0.15:
                los.append(None)
            elif kind < 0.25:
                los.append(rng.randint(0, total))          # out of order: must never re-open a fired range
            else:
                cur = max(0, cur - rng.randint(0, 400))
                los.append(cur)
        fired, seen_min = [], total
        for lo in los:
            sl = plan.on_done(lo)
            if lo is not None:
                seen_min = min(seen_min, lo)
            if sl is not None:
                assert sl[0] >= seen_min                       # nothing below the lowest completed offset goes out
                fired.append(sl)
        last = plan.flush()
        if last is not None:
            fired.append(last)
        assert plan.flush() is None
        hi = total
        for lo_, hi_ in fired:
            assert hi_ == hi and 0 <= lo_ < hi_
            hi = lo_
        assert hi == 0
