#!/usr/bin/env python
"""Benchmark of the caption-generator hot path (BASELINE.json metric: train samples/sec, plus beam-5
captions/sec as a secondary figure), contract of the task prompt:

    python bench.py --gpus N --steps K --warmup W            # this repo (B200, CUDA path via the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the UNMODIFIED reference on the host CPU

Prints ONE JSON line.  Default workload = BASELINE.json configs[1]: teacher-forced training step (forward +
backward + Adam, dropout on), bf16, batch 256 per GPU, 36 regions x 2048-d, caption length 22 (T = 21 decoder
positions), vocab 10k, ctor-default Transformer (d512/8h/2048/6+6).  Synthetic data, random-init weights.
`--dump-outputs DIR` writes the loss and the updated parameters of the last timed train step as DIR/<name>.npy; inputs,
weights and dropout streams are seeded, so two builds run with the same arguments can be compared array for array.
Not bit for bit: the step reduces weight gradients with fp32 atomics, so two runs of one build already differ (B200 at
1000 W, --steps 20 --warmup 5: losses by 1e-6 relative, single sampled weights by up to 9e-2 of their tensor's max).
N > 1 = data parallel (weak scaling, 256 samples per rank), gradients summed by bucketed NCCL all-reduces that
overlap the backward.  Other BASELINE configs through `--workload`:
    modelA      configs[1] (+ configs[2] beam-5/3/greedy decode of 512 images, configs[0] model B greedy B=8 as extras)
    global2048  configs[3]: model A, GLOBAL batch 2048 split over the N ranks (strong scaling; N=1 runs 2048 on one GPU)
    modelC      configs[4]: scaled model (d1024 / 16 heads / FFN 4096 / 6+6, 100 regions, vocab 30k), 256 per GPU
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

MODEL_A = dict(num_vocab=10000, max_length=22, encode_dim_positions=84, encode_dim_features=2048,
               output_name="bench", dropout=0.2)
# core/config.py defaults of the reference (config.py:87-129): BASELINE configs[0]
MODEL_B = dict(num_vocab=10000, max_length=51, encode_dim_positions=84, encode_dim_features=2048, output_name="bench",
               dropout=0.3, encode_mask=True, split_image_objects=True, encode_input_size=256, encode_q_k_dim=256,
               encode_v_dim=256, encode_hidden_size=256, encode_num_blocks=2, encode_num_heads=32, dim_word_embedding=256,
               decode_input_size=256, decode_q_k_dim=256, decode_v_dim=256, decode_hidden_size=256, decode_num_blocks=5,
               decode_num_heads=32)
MODEL_C = dict(num_vocab=30000, max_length=22, encode_dim_positions=84, encode_dim_features=2048, output_name="bench",
               dropout=0.2, encode_input_size=1024, encode_q_k_dim=1024, encode_v_dim=1024, encode_hidden_size=4096,
               encode_num_blocks=6, encode_num_heads=16, dim_word_embedding=1024, decode_input_size=1024,
               decode_q_k_dim=1024, decode_v_dim=1024, decode_hidden_size=4096, decode_num_blocks=6, decode_num_heads=16)
CAP_LEN = 22
DECODE_BATCH = 512
DUMP_SAMPLE = 1 << 16      # --dump-outputs: elements kept per parameter tensor (190 tensors of model A / C: < 26 MB)

# SURVEY.md §8(d): algorithmic matmul FLOPs as the reference executes them (fwd+bwd) / KV-cached beam-5, 21 steps
WORKLOADS = {
    "modelA": dict(kw=MODEL_A, regions=36, gflop_train=8.458, gflop_beam5=7.274, per_gpu=256, scaling="weak",
                   ref_batch=256,
                   text="configs[1]: teacher-forced train step fwd+bwd+Adam, model A (d512/8h/ffn2048/6+6), batch 256 per GPU, "
                        "R=36x2048, T=21, V=10k"),
    "global2048": dict(kw=MODEL_A, regions=36, gflop_train=8.458, gflop_beam5=7.274, per_gpu=None, scaling="strong",
                       ref_batch=256,
                       text="configs[3]: teacher-forced train step fwd+bwd+Adam, model A, GLOBAL batch 2048 split over the "
                            "ranks, R=36x2048, T=21, V=10k"),
    "modelC": dict(kw=MODEL_C, regions=100, gflop_train=69.75, gflop_beam5=42.78, per_gpu=256, scaling="weak",
                   ref_batch=16,
                   text="configs[4]: teacher-forced train step fwd+bwd+Adam, model C (d1024/16h/ffn4096/6+6), batch 256 per "
                        "GPU, R=100x2048, T=21, V=30k"),
}


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"tflops": d["bf16_tflops"], "tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "hbm": d["hbm_gbs"], "src": "measured (MEASURED_PEAKS.json)"}
    return {"tflops": 1590.0, "tflops_sustained": 1400.0, "hbm": 6650.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clock / throttle sampling DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def output_sample(loss: torch.Tensor, named_params) -> dict:
    """What a caller of the training step holds after its last step, as float32 host arrays keyed by file name: the
    loss and every updated parameter -- whole up to DUMP_SAMPLE elements, larger ones at DUMP_SAMPLE positions drawn
    from a generator seeded per tensor, so that two runs or two builds sample the same elements."""
    out = {"loss": loss.detach().float().reshape(1).cpu().numpy()}
    for name, q in named_params:
        flat = q.detach().reshape(-1)
        if flat.numel() > DUMP_SAMPLE:
            idx = torch.randint(flat.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            flat = flat[idx.to(flat.device)]
        out["param." + name] = flat.float().cpu().numpy()
    return out


def write_outputs(out_dir: str, arrays: dict) -> None:
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------- the reference on the CPU
class CpuReference:
    """The reference's own classes (staged under baseline/_ref, see baseline/ref_loader.py) on the host cores, with the
    wrapper logic of core/models.py:111-126 (Adam lr 5e-4, zero_grad -> forward -> backward -> step) restated here
    because core/models.py itself needs COCO artefacts to import.  Falls back to the oracle port (same arithmetic,
    functional restatement) when the reference is not staged; `kind` says which one ran."""

    def __init__(self, kw: dict, train: bool):
        from baseline import ref_loader
        torch.set_num_threads(host_threads())          # torchrun exports OMP_NUM_THREADS=1: use every host core anyway
        self.kw = kw
        ref = ref_loader.load()
        if ref is not None:
            self.kind = "reference"
            torch.manual_seed(0)
            self.model = ref[0](device=torch.device("cpu"), **kw)
            self.model.train(train)
            self.opt = torch.optim.Adam((p for p in self.model.parameters() if p.requires_grad), lr=5e-4)
        else:
            from oracle import caption_oracle as O
            self.kind = "port"
            self.O = O
            self.cfg = O.OracleConfig(**{**kw, "dropout": 0.0})
            self.sd = O.init_state_dict(self.cfg, seed=0)
            self.opt = O.AdamState(self.sd)

    def state_dict(self):
        return {k: v.detach().clone() for k, v in self.model.state_dict().items()} if self.kind == "reference" else self.sd

    def train_step(self, f, p, c) -> float:
        if self.kind == "reference":
            self.opt.zero_grad()
            loss = self.model(f, p, c)["loss"]
            loss.backward()
            self.opt.step()
            return float(loss)
        loss, grads = self.O.loss_and_grads(self.sd, self.cfg, f, p, c)
        self.opt.step(self.sd, grads)
        return float(loss)

    @torch.no_grad()
    def greedy(self, f, p):
        if self.kind == "reference":
            return self.model.generate_caption_vector(f, p)[0]
        return self.O.generate_caption_vector(self.sd, self.cfg, f, p)[0]

    @torch.no_grad()
    def beam(self, f, p, k):
        if self.kind == "reference":
            return self.model.beam_search(f, p, beam_size=k)
        return self.O.beam_search(self.sd, self.cfg, f, p, beam_size=k)

    def describe(self) -> str:
        return ("unmodified reference classes (baseline/_ref), train mode, dropout on" if self.kind == "reference"
                else "oracle port of the reference (baseline/_ref not staged), dropout off")


def run_reference(args):
    """bench.py --impl reference: the reference's own CPU implementation of the path, all host threads, on the same
    workload / metric; each step = one train step on a bounded sample (model A: the full batch 256; model C: batch 16)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import caption_oracle as O
    wl = WORKLOADS[args.workload]
    kw = wl["kw"]
    bs = args.ref_batch or wl["ref_batch"]
    if not args.ref_batch:
        # bounded sample: the whole --steps + --warmup run stays near 3 minutes of CPU time (measured on the bench box's 16
        # cores: ~115 samples/s for model A, ~13 for model C), so a large K shrinks the batch of each step instead
        rate = 110.0 if wl["gflop_train"] < 20 else 12.0
        fit = int(rate * 180.0 / (args.steps + max(1, args.warmup)))
        bs = max(4, min(bs, fit // 4 * 4))
    ref = CpuReference(kw, train=True)
    f, p, c = O.synthetic_batch(bs, wl["regions"], 2048, 84, CAP_LEN, kw["num_vocab"], seed=1234)
    for _ in range(max(1, args.warmup)):
        ref.train_step(f, p, c)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ref.train_step(f, p, c)
    dt = time.perf_counter() - t0
    v = bs * args.steps / dt
    sample = f"{args.steps} train steps (fwd+bwd+Adam) at batch {bs}, {ref.describe()}, torch CPU fp32"
    line = {"impl": "reference", "metric": "train_samples_per_sec", "value": v, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["text"], "dropout": "on (0.2 / attention 0.1)" if ref.kind == "reference" else "off",
                       "global_batch": bs, "batch_per_gpu": None, "parallelism": f"cpu, {torch.get_num_threads()} host threads",
                       "sample": f"each step = one train step on batch {bs}"},
            "cpu_baseline": {"value": v, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": ref.kind,
                             "sample": sample},
            "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def cpu_baseline_sample(wl, budget_s: float = 15.0, max_steps: int = 100):
    """`cpu_baseline` of our arm: the reference on the host cores for ~budget_s seconds of train steps of the same
    model / shapes (bounded sample: batch 64 for model A, 8 for model C)."""
    from oracle import caption_oracle as O
    kw = wl["kw"]
    bs = 64 if wl["gflop_train"] < 20 else 8
    ref = CpuReference(kw, train=True)
    f, p, c = O.synthetic_batch(bs, wl["regions"], 2048, 84, CAP_LEN, kw["num_vocab"], seed=1234)
    ref.train_step(f, p, c)
    n, t0 = 0, time.perf_counter()
    while n < max_steps and (n < 2 or time.perf_counter() - t0 < budget_s):
        ref.train_step(f, p, c)
        n += 1
    dt = time.perf_counter() - t0
    return {"value": bs * n / dt, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": ref.kind,
            "sample": f"{n} train steps (fwd+bwd+Adam) at batch {bs} of the same model/shapes in {dt:.1f} s, "
                      f"{ref.describe()}, torch CPU fp32, all host threads"}


def cpu_decode_baselines(extra: dict):
    """CPU anchors for the decode figures: configs[0] (model B, greedy, B=8, 50 steps -- BASELINE.md 5.4 'mandatory')
    and model A beam-5 at B=8 (the reference recomputes the whole prefix per step and beam: no KV cache)."""
    from oracle import caption_oracle as O
    out = {}
    refB = CpuReference(MODEL_B, train=False)
    f, p, _ = O.synthetic_batch(8, 36, 2048, 84, MODEL_B["max_length"], 10000, seed=4321)
    refB.greedy(f, p)
    t0 = time.perf_counter()
    for _ in range(3):
        ids_b = refB.greedy(f, p)
    out["config1_cpu_greedy_captions_per_s"] = 8 * 3 / (time.perf_counter() - t0)
    out["config1_cpu"] = {"kind": refB.kind, "cores": torch.get_num_threads(),
                          "sample": "model B (config.py defaults: d256/32h/2+5, encode_mask, split_image_objects), "
                                    "greedy, batch 8, 50 steps, eval(), 1 warm-up + 3 runs"}
    refA = CpuReference({**MODEL_A}, train=False)
    fa, pa, _ = O.synthetic_batch(8, 36, 2048, 84, CAP_LEN, 10000, seed=4321)
    refA.beam(fa, pa, 5)
    t0 = time.perf_counter()
    for _ in range(2):
        refA.beam(fa, pa, 5)
    out["beam5_cpu_captions_per_s"] = 8 * 2 / (time.perf_counter() - t0)
    out["beam5_cpu"] = {"kind": refA.kind, "cores": torch.get_num_threads(),
                        "sample": "model A, beam_search(beam_size=5), batch 8, 21 steps, eval(), 1 warm-up + 2 runs"}
    extra.update(out)
    return refB, (f, p, ids_b)


# ----------------------------------------------------------------------------------------------- our arm
def dp_parity_check(pkg, dist, dev, rank, world):
    """N-GPU gradient == 1-GPU gradient on the concatenated batch (SURVEY.md §4 item 4), through the REAL path: fp32
    mode, bucketed NCCL all-reduces fired from the backward (2 MB buckets so that several fire), dropout off.
    Returns the relative Frobenius error of the whole flat gradient."""
    kw = dict(MODEL_A, dropout=0.0, encode_num_blocks=2, decode_num_blocks=2)
    from oracle import caption_oracle as O
    torch.manual_seed(0)
    m = pkg.Transformer(device=dev, **kw).to(dev)
    m.set_precision("fp32")
    eng = m._engine()
    dp = pkg.DataParallel(m, dist, bucket_mb=2.0)
    b = 4
    f, p, c = O.synthetic_batch(b, 36, 2048, 84, CAP_LEN, 10000, seed=777 + rank)
    f, p, c = f.to(dev), p.to(dev), c.to(dev)
    dp.begin(eng)
    eng.forward_backward(f, p, c, train_mode=False)
    dp.end(eng)
    torch.cuda.synchronize(dev)
    n = eng.n_flat
    g_dp = (eng.g32[:n] / eng.g32[n]).clone()
    nb = dp.n_buckets
    gf = [torch.empty_like(f) for _ in range(world)]
    gp = [torch.empty_like(p) for _ in range(world)]
    gc = [torch.empty_like(c) for _ in range(world)]
    dist.all_gather(gf, f)
    dist.all_gather(gp, p)
    dist.all_gather(gc, c)
    eng.dp_unnormalized = False
    eng.forward_backward(torch.cat(gf), torch.cat(gp), torch.cat(gc), train_mode=False)
    torch.cuda.synchronize(dev)
    g_1 = eng.g32[:n]
    err = float((g_dp - g_1).norm() / g_1.norm())
    del m, eng, dp
    return err, nb


def run_ours(args):
    import icap_loader
    from oracle import caption_oracle as O      # synthetic input generator (+ CPU baseline fall-back) only
    pkg = icap_loader.load()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    wl = WORKLOADS[args.workload]
    kw, R, V = wl["kw"], wl["regions"], wl["kw"]["num_vocab"]
    BATCH = wl["per_gpu"] if wl["per_gpu"] else 2048 // world
    extra = {}

    if dist is not None:
        err, nb = dp_parity_check(pkg, dist, dev, rank, world)
        extra["dp_parity_rel_err"] = err
        extra["dp_parity"] = (f"fp32, model A with 2+2 blocks, 4 samples per rank: flat gradient of the {world}-rank step "
                              f"({nb} NCCL buckets fired from the backward) vs one rank on the all-gathered batch")

    torch.manual_seed(0)
    model = pkg.Transformer(device=dev, **kw).to(dev).train()
    model.set_precision(args.precision)
    eng = model._engine()

    # a pool of distinct synthetic batches (pool > L2), resident in HBM and mirrored in pinned host memory
    pool = []
    for i in range(4):
        f, p, c = O.synthetic_batch(BATCH, R, 2048, 84, CAP_LEN, V, seed=1234 + 17 * rank + i)
        pool.append((f.pin_memory(), p.pin_memory(), c.pin_memory()))
    dpool = [(f.to(dev), p.to(dev), c.to(dev)) for f, p, c in pool]
    h2d_bytes = sum(t.numel() * t.element_size() for t in pool[0])

    dp = None
    if world > 1:
        dp = pkg.DataParallel(model, dist)
    gs = pkg.GraphedTrainStep(model, BATCH, R, CAP_LEN, lr=5e-4, dp=dp)
    gs.load(*dpool[0])
    gs.capture()
    launches_per_step = gs.launches_per_step

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        t = torch.tensor([ms], device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # ---------------- device-resident timing (value)
    for i in range(max(3, args.warmup)):
        gs.load(*dpool[i % 4])
        gs.step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        gs.load(*dpool[i % 4])
        loss_dev = gs.step()
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    final_loss = float(loss_dev)
    if args.dump_outputs and rank == 0:    # before the end-to-end loops below step the weights further
        write_outputs(args.dump_outputs, output_sample(loss_dev, model.named_parameters()))
    value = world * BATCH * args.steps / (ms / 1e3)

    # ---------------- end-to-end: pinned host inputs -> H2D (copy stream, double buffered) -> step -> D2H loss
    copy_stream = torch.cuda.Stream(device=dev)
    stage = [tuple(torch.empty_like(x) for x in dpool[0]) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    losses_host = torch.zeros(args.steps + 8, dtype=torch.float32).pin_memory()
    main = torch.cuda.current_stream(dev)

    def e2e_loop(n, offset):
        for i in range(n):
            b = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[b])
                for dst, src in zip(stage[b], pool[i % 4]):
                    dst.copy_(src, non_blocking=True)
                ready[b].record(copy_stream)
            main.wait_event(ready[b])
            gs.load(*stage[b])
            consumed[b].record(main)
            out = gs.step()
            losses_host[offset + i:offset + i + 1].copy_(out.reshape(1), non_blocking=True)

    for b in range(2):
        consumed[b].record(main)
    e2e_loop(4, args.steps)
    barrier()
    e0.record()
    e2e_loop(args.steps, 0)
    e1.record()
    barrier()
    e2e_value = world * BATCH * args.steps / (max_over_ranks(e0.elapsed_time(e1)) / 1e3)
    clocks = sampler.stop() if rank == 0 else None      # sampled over both timed regions (device-resident + end to end)

    # ---------------- data feed (SURVEY.md 8f #2): batches named by image number into a device-resident region cache;
    # at N > 1 this is the end-to-end figure that does not saturate the host's PCIe with 8 x 79 MB of fp32 per step
    if not args.no_decode:
        n_img = 2048
        F, P, _ = O.synthetic_batch(n_img, R, 2048, 84, CAP_LEN, V, seed=99 + rank)
        t0 = time.perf_counter()
        cache = pkg.RegionCache(model, F.numpy(), P.numpy())
        torch.cuda.synchronize(dev)
        extra["region_cache_build_images_per_s"] = n_img / (time.perf_counter() - t0)
        extra["region_cache_bytes_per_image"] = cache.nbytes // n_img
        gen = torch.Generator().manual_seed(5 + rank)
        idx_pool = [torch.randint(0, n_img, (BATCH,), generator=gen).pin_memory() for _ in range(4)]
        if world == 1:      # what the reference's DataLoader does on the host for the same batch (dataset.py:12-18 + collate)
            t0 = time.perf_counter()
            torch.stack([F[int(i)] for i in idx_pool[0]])
            extra["reference_host_collate_ms_per_batch"] = 1e3 * (time.perf_counter() - t0)
        del F, P
        gc = pkg.GraphedTrainStep(model, BATCH, R, CAP_LEN, lr=5e-4, cache=cache, dp=dp)
        gc.load(idx_pool[0], None, pool[0][2])
        gc.capture()

        def cached_loop(n, offset):
            for i in range(n):
                gc.load(idx_pool[i % 4], None, pool[i % 4][2])         # 2 KB of image numbers + 22 KB of captions
                out = gc.step()
                losses_host[offset + i:offset + i + 1].copy_(out.reshape(1), non_blocking=True)
        cached_loop(4, args.steps)
        barrier()
        e0.record()
        cached_loop(args.steps, 0)
        e1.record()
        barrier()
        cache.check()
        extra["train_region_cache_e2e_samples_per_s"] = world * BATCH * args.steps / (max_over_ranks(e0.elapsed_time(e1)) / 1e3)
        extra["train_region_cache_h2d_bytes_per_step"] = idx_pool[0].numel() * 8 + pool[0][2].numel() * 4
        extra["train_region_cache_launches_per_step"] = gc.launches_per_step
        del gc, cache

    # ---------------- secondary figures: KV-cached beam-5 / beam-3 / greedy captions/s (configs[2]).  Decode partitions
    # by image with no collective (SURVEY.md 8e): every rank decodes its own 512 images; captions/s = all ranks' images /
    # max-over-ranks device time.
    if not args.no_decode:
        model.eval()
        f, p, _ = O.synthetic_batch(DECODE_BATCH, R, 2048, 84, CAP_LEN, V, seed=4321 + rank)
        f, p = f.to(dev), p.to(dev)
        fh, ph = f.cpu().pin_memory(), p.cpu().pin_memory()
        for k in (5, 3, 1):
            gd = pkg.GraphedDecode(model, DECODE_BATCH, R, k)
            for _ in range(2):
                gd.run(f, p)
            barrier()
            e0.record()
            reps = 5
            for _ in range(reps):
                gd.run(f, p)
            e1.record()
            barrier()
            msd = max_over_ranks(e0.elapsed_time(e1) / reps)
            name = f"beam{k}" if k > 1 else "greedy"
            extra[f"{name}_captions_per_s"] = world * DECODE_BATCH / (msd / 1e3)
            extra[f"{name}_ms_per_batch512"] = msd
            # end to end through the drop-in API: pinned host features in, token ids back on the host
            fn = (lambda: model.beam_search(fh, ph, beam_size=k).cpu()) if k > 1 else \
                (lambda: model.generate_caption_vector(fh, ph)[0].cpu())
            fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(3):
                fn()
            torch.cuda.synchronize(dev)
            t = torch.tensor([time.perf_counter() - t0], device=dev)
            if dist is not None:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            extra[f"{name}_e2e_single_call_captions_per_s"] = world * DECODE_BATCH * 3 / float(t)
            # the evaluation loop of main.py: batches of pinned host features through PrefetchLoader (the copy of batch
            # i + 1 runs on a copy stream while batch i decodes), token ids read back to the host after every batch
            def eval_loop(n):
                ids = None
                for fd, pd_ in pkg.PrefetchLoader([(fh, ph)] * n, dev):
                    ids = (model.beam_search(fd, pd_, beam_size=k) if k > 1 else model.generate_caption_vector(fd, pd_)[0]).cpu()
                return ids
            eval_loop(2)
            barrier()
            t0 = time.perf_counter()
            eval_loop(6)
            torch.cuda.synchronize(dev)
            t = torch.tensor([time.perf_counter() - t0], device=dev)
            if dist is not None:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            extra[f"{name}_e2e_captions_per_s"] = world * DECODE_BATCH * 6 / float(t)
            del gd
        tf5 = extra["beam5_captions_per_s"] / world * wl["gflop_beam5"] * 1e9 / 1e12
        extra["roofline_decode"] = {
            "bound": "tensor", "what": "KV-cached beam-5 decode of 512 images per GPU, whole graph (encoder + cross-K/V + "
                                       "21 steps), algorithmic %.3f GFLOP per image" % wl["gflop_beam5"],
            "achieved": tf5, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": tf5 / pk["tflops"],
            "frac_sustained": tf5 / pk["tflops_sustained"], "ms_per_batch512": extra["beam5_ms_per_batch512"]}
        extra["beam5_frac_of_tensor_peak"] = tf5 / pk["tflops"]
        model.train()

    if rank != 0:
        # No process-group teardown: destroying the NCCL communicator while CUDA graphs that captured its
        # collectives are alive can hang; the timed work is done and rank 0 needs no further collective.
        torch.cuda.synchronize(dev)
        sys.stdout.flush()
        os._exit(0)

    # ---------------- per-kernel roofline: CUDA events around every GEMM launch of one eager step
    if args.ncu_region:       # one eager step bracketed by cudaProfilerStart/Stop for `ncu --profile-from-start off`
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        eng.train_step(*dpool[0], lr=5e-4)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
    # All GEMM launches of one step, re-launched back to back from ONE CUDA graph (no host launch gaps, same
    # operand buffers / shapes / epilogues as the step): average in-situ duration of the dominant kernel.
    keep = []        # keeps the step's activations allocated so that the recorded pointers stay valid
    orig_new = eng.new

    def pinned_new(*a, **k):
        t = orig_new(*a, **k)
        keep.append(t)
        return t
    eng.new = pinned_new
    hook = eng.bucket_hook
    eng.bucket_hook = None
    log = eng.record_gemms(lambda: eng.train_step(*dpool[0], lr=5e-4))
    eng.bucket_hook = hook
    eng.new = orig_new
    torch.cuda.synchronize(dev)
    gg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gg):
        gemm_flops = eng.replay_gemms(log)
    for _ in range(3):
        gg.replay()
    torch.cuda.synchronize(dev)
    reps = 10
    e0.record()
    for _ in range(reps):
        gg.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    gemm_ms = e0.elapsed_time(e1) / reps
    del keep
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tpath) and args.workload in ("modelA", "global2048") and BATCH == 256:   # the capture is of the
        # model-A step at batch 256 only (bytes per launch grow with the batch: no figure for other per-GPU batches)
        tj = json.load(open(tpath))
        traffic = tj.get("dram_bytes_per_launch")
        traffic_src = ("static, NOT measured by this run: dram__bytes_read+write per launch from the ncu capture "
                       + str(tj.get("source", "profiles/r1_gemm_dram_launches.csv")) + " (cold cache, L2 flushed per launch)")
    step_tf = value * wl["gflop_train"] * 1e9 / world / 1e12
    roofline = {"bound": "tensor",
                "kernel": "gemm_tc_kernel (persistent tcgen05/TMA bf16 GEMM): its %d launches in one train step, replayed "
                          "back to back from one CUDA graph%s" % (len(log), (
                              " (the forward's projection+LayerNorm GEMMs run in the fused cluster kernel gemm_ln_kernel "
                              "and are not part of this figure)" if eng.gemm_ln_mode == 2 else "")),
                "achieved": achieved, "peak": pk["tflops"], "unit": "TFLOP/s",
                "frac": achieved / pk["tflops"], "frac_sustained": achieved / pk["tflops_sustained"],
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": pk["src"] + ", BURST figure (the replay is a ~25 ms burst at full clocks); sustained peak "
                               "%.1f" % pk["tflops_sustained"],
                "avg_launch_us": 1e3 * gemm_ms / max(1, len(log)),
                "gemm_ms_per_step": gemm_ms, "gemm_gflop_per_step": gemm_flops / 1e9,
                "gemm_share_of_step": gemm_ms / (ms / args.steps),
                "step_model_tflops": step_tf, "step_model_flops_frac": step_tf / pk["tflops"],
                "step_model_flops_frac_of_sustained": step_tf / pk["tflops_sustained"]}

    cpu = None
    if not args.no_cpu_baseline and world == 1:       # CPU baselines: rank 0 at N = 1 only (the reference arm covers N > 1)
        cpu = cpu_baseline_sample(wl)
        if args.workload == "modelA" and not args.no_decode:
            # configs[0]: model B greedy B=8 on the CPU (reference) and on the GPU (bf16 timing + fp32 id parity)
            refB, (fb, pb, ids_cpu) = cpu_decode_baselines(extra)
            mB = pkg.Transformer(device=dev, **MODEL_B)
            mB.load_state_dict(refB.state_dict())
            mB = mB.to(dev).eval()
            mB.set_precision("fp32")
            ids32, _ = mB.generate_caption_vector(fb, pb)
            ids32 = ids32.cpu()
            same = ids32.shape == ids_cpu.shape and bool((ids32 == ids_cpu).all())
            extra["config1_gpu_fp32_ids_identical_to_cpu_reference"] = same
            if not same:
                extra["config1_gpu_fp32_min_gap"] = float(mB.last_gaps.min())
            mB.set_precision("bf16")
            mB.generate_caption_vector(fb, pb)
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for _ in range(5):
                mB.generate_caption_vector(fb, pb)[0].cpu()
            extra["config1_gpu_greedy_captions_per_s"] = 8 * 5 / (time.perf_counter() - t0)
            extra["config1_gpu"] = "model B, greedy, batch 8, 50 steps, bf16, through generate_caption_vector with host inputs"
            extra["beam5_gpu_over_cpu"] = extra["beam5_e2e_captions_per_s"] / extra["beam5_cpu_captions_per_s"]
    line = {"metric": "train_samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": wl["text"], "dropout": "on (0.2 / attention 0.1)",
                       "global_batch": world * BATCH, "batch_per_gpu": BATCH, "parallelism": f"dp{world}",
                       "l2": "4 rotating input batches (%d MB) + parameter/optimizer state per step >> 126 MB L2"
                             % (4 * h2d_bytes >> 20),
                       "cuda_graph": True},
            "final_loss": final_loss,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "note": "pinned host inputs, H2D double-buffered on a copy stream, loss read back every step"},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline, "cpu_baseline": cpu, "extra": extra}
    print(json.dumps(line))
    sys.stdout.flush()
    if dist is not None:
        torch.cuda.synchronize(dev)
        os._exit(0)          # see the note at the non-zero ranks' exit above


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 100 on the GPU, 20 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="modelA", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--ref-batch", type=int, default=0, help="reference arm: batch of each step (0 = the workload's)")
    ap.add_argument("--no-decode", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ncu-region", action="store_true", help="wrap one eager step in cudaProfilerStart/Stop")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and the updated parameters of the last timed train step as DIR/<name>.npy "
                         "(float32; parameters above %d elements as a fixed seeded sample)" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (--impl ours)")
    if args.steps is None:
        args.steps = 20 if args.impl == "reference" else 100
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
