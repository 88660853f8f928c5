"""Caption-metric timings on one GPU -> one JSON line.

  reward_ms      CaptionReward.on_device (clear table, cook targets, df, ref norms, score) replayed from a CUDA graph,
                 CUDA-event time per call, at B in {32, 256} x T in {22, 50}
  host_ms        the same batches through the host rewards: ngram_precision_reward (the default reward_fn) and the
                 fp64 reference scorer (tests/caption_metrics_oracle.py), wall time per call
  scorer         CaptionScorer build (cook, count, df table, norms) and score of one caption per image, wall time
                 around device-synchronised work, for a 5,000-image and a COCO-train-size (113,287-image) split with
                 5 references per image, and the df table's size in bytes

Captions draw Zipf-distributed ids (vocabulary 10,000) from a fixed seed: uniform ids would make nearly every 4-gram
unique and size the table unrealistically.  Card name and power limit are read in the same run."""
import importlib.util
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import icap_loader  # noqa: E402
import caption_metrics_oracle as ref_scorer  # noqa: E402

pkg = icap_loader.load()
DEV = torch.device("cuda:0")
VOCAB = 10000


def _loss_module():
    spec = importlib.util.spec_from_file_location(
        "icap_rl_loss", os.path.join(ROOT, "image-caption_b200", "core", "TRANSFORMER", "loss.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def captions(rng, n, width, start=True):
    """n id rows of `width`: [<START>] words <END> <NULL>..., 8..20 Zipf-distributed words."""
    x = np.zeros((n, width), dtype=np.int64)
    lens = rng.integers(8, 21, size=n)
    words = 3 + (rng.zipf(1.2, size=(n, width)) % (VOCAB - 3))
    off = 1 if start else 0
    if start:
        x[:, 0] = 1
    pos = np.arange(width)[None, :]
    lens = np.minimum(lens, width - 1 - off)
    x = np.where((pos >= off) & (pos < off + lens[:, None]), words, x)
    x[np.arange(n), off + lens] = 2
    return x


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as exc:                    # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({exc})"}


def reward_times(rng, iters=1000):
    loss = _loss_module()
    out = {}
    for B in (32, 256):
        for T in (22, 50):
            t = captions(rng, B, T + 1)[:, 1:]
            s = np.where(rng.random((B, T)) < 0.5, t, captions(rng, B, T, start=False))
            ts, ss = torch.as_tensor(t).to(DEV), torch.as_tensor(s).to(DEV)
            rw = pkg.CaptionReward(1.0, 1.0)
            rw.on_device(ts, ss)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            from image_caption_b200.transformer import _graph_capture
            with _graph_capture(g):
                rw.on_device(ts, ss)
            for _ in range(20):
                g.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(iters):
                g.replay()
            e1.record()
            torch.cuda.synchronize()
            dev_ms = e0.elapsed_time(e1) / iters
            n_host = 20 if B == 32 else 5
            t0 = time.perf_counter()
            for _ in range(n_host):
                loss.ngram_precision_reward(t, s)
            ngram_ms = (time.perf_counter() - t0) / n_host * 1e3
            t0 = time.perf_counter()
            for _ in range(n_host):
                ref_scorer.reward(t, s)
            fp64_ms = (time.perf_counter() - t0) / n_host * 1e3
            out[f"B{B}_T{T}"] = {"reward_graph_ms": round(dev_ms, 4), "iters": iters,
                                 "host_ngram_precision_ms": round(ngram_ms, 3), "host_fp64_reference_ms": round(fp64_ms, 3)}
    return out


def scorer_times(rng):
    out = {}
    for n_img in (5000, 113287):
        refs = captions(rng, 5 * n_img, 52)
        ref_imgs = np.repeat(np.arange(n_img), 5)
        cands = np.where(rng.random((n_img, 52)) < 0.5, refs[::5], captions(rng, n_img, 52))
        cand_t = torch.as_tensor(cands).to(DEV)
        cand_i = torch.arange(n_img, device=DEV)
        pkg.CaptionScorer(refs[:50], ref_imgs[:50], VOCAB, DEV).score(cand_t[:10], cand_i[:10])   # load the kernels
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sc = pkg.CaptionScorer(refs, ref_imgs, VOCAB, DEV)
        torch.cuda.synchronize()
        build_ms = (time.perf_counter() - t0) * 1e3
        times = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, corpus = sc.score(cand_t, cand_i)
            torch.cuda.synchronize()
            times.append((time.perf_counter() - t0) * 1e3)
        out[f"{n_img}x5"] = {"build_ms": round(build_ms, 2), "score_ms_median": round(float(np.median(times)), 2),
                             "table_bytes": sc.table_bytes, "table_slots": sc.table.cap,
                             "ref_rows": int(len(refs)), "CIDEr-D": round(corpus["CIDEr-D"], 4)}
        del sc
        torch.cuda.empty_cache()
    return out


def main():
    rng = np.random.default_rng(1234)
    res = {"tool": "score_bench", **gpu_info(), "reward": reward_times(rng), "scorer": scorer_times(rng)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
