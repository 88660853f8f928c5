"""Sampled decoding timings on one GPU -> one JSON line.

  decode        model A (6 + 6 blocks, V = 10,000, max_length 22), bf16, 512 images x 36 regions, every decode replayed
                from its CUDA graph: greedy, beam-5, sampled n = 1 and n = 5 at temperature 1.  CUDA-event time per call
                (median of `--reps` timed calls after warm-up) and captions/s (images x captions per image / time).
  kernels       a separate torch.profiler pass: sample_kernel (icap_sample_tokens) against argmax_kernel (icap_argmax)
                over the same 2560 x 10,000 bf16 logits rows (ldl 10,000), mean GPU time per launch.

Card name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import icap_loader  # noqa: E402
from oracle import caption_oracle as O  # noqa: E402

pkg = icap_loader.load()
N = pkg._native
DEV = torch.device("cuda:0")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as exc:                    # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({exc})"}


def time_calls(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms.sort()
    return ms[len(ms) // 2]


def decode_times(reps):
    kw = dict(num_vocab=10000, max_length=22, encode_dim_positions=84, encode_dim_features=2048, output_name="x",
              dropout=0.0)
    torch.manual_seed(0)
    m = pkg.Transformer(device=DEV, **kw).to(DEV).eval()
    B = 512
    f, p, _ = O.synthetic_batch(B, 36, 2048, 84, 22, 10000, seed=4321)
    f, p = f.to(DEV), p.to(DEV)
    runs = {
        "greedy": (lambda: m.generate_caption_vector(f, p), 1),
        "beam5": (lambda: m.beam_search(f, p, beam_size=5), 1),
        "sample_n1": (lambda: m.sample_captions(f, p, num_samples=1), 1),
        "sample_n5": (lambda: m.sample_captions(f, p, num_samples=5), 5),
    }
    out = {}
    for name, (fn, per_image) in runs.items():
        ms = time_calls(fn, reps)
        out[name] = {"ms_per_call": round(ms, 3), "captions_per_s": round(B * per_image / ms * 1e3, 1)}
    return out


def kernel_times(iters):
    M, V = 2560, 10000
    g = torch.Generator(device=DEV).manual_seed(0)
    logits = (torch.randn(M, V, device=DEV, generator=g) * 2).to(torch.bfloat16)
    tokens = torch.ones(M, 22, dtype=torch.int32, device=DEV)
    logp = torch.zeros(M, 21, device=DEV)
    counter = torch.zeros(1, dtype=torch.int32, device=DEV)
    st = torch.cuda.current_stream().cuda_stream

    def sample():
        N.call("icap_sample_tokens", N.BF16, M, V, logits.data_ptr(), V, 1.0, 0x243F6A8885A308D3, counter.data_ptr(), 0,
               22, tokens.data_ptr(), logp.data_ptr(), 21, 2, 0, st)

    def argmax():
        N.call("icap_argmax", N.BF16, M, V, logits.data_ptr(), V, tokens.data_ptr() + 4, 22, None, st)

    for fn in (sample, argmax):
        fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            sample()
            argmax()
        torch.cuda.synchronize()
    tot = {"sample_kernel": [0.0, 0], "argmax_kernel": [0.0, 0]}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        for k in tot:
            if k in e.name:
                tot[k][0] += e.device_time
                tot[k][1] += 1
    return {k: {"us_per_launch": round(t / max(n, 1), 2), "launches": n, "rows": M, "V": V} for k, (t, n) in tot.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--kernel-iters", type=int, default=200)
    a = ap.parse_args()
    res = {"tool": "sample_bench", **gpu_info(), "decode_512_images_bf16": decode_times(a.reps),
           "kernels_2560x10000_bf16": kernel_times(a.kernel_iters)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
