"""Cost of the beam search that stops at <END> -> one JSON line.

Model A (6 + 6 blocks, V = 10,000, max_length 22) in bf16, 512 images x 36 regions, beam 5: Transformer.beam_search
(the reference's search) against Transformer.beam_search_nbest (length penalty 0.6, all 5 hypotheses returned), both
replayed from their CUDA graphs.  The two are timed in alternating rounds of `--reps` calls (CUDA events around each
call, median per round, median over rounds) so that drift of a shared machine hits both alike.  The model is at
initialisation with the <END> bias raised by each of `--end-bias` in turn: 0 lets no hypothesis finish (the full
per-step cost), larger values make hypotheses finish earlier (finished fraction and mean length of the best caption
reported).  Card name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import icap_loader  # noqa: E402
from oracle import caption_oracle as O  # noqa: E402
from sample_bench import gpu_info, time_calls  # noqa: E402

pkg = icap_loader.load()
DEV = torch.device("cuda:0")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--end-bias", default="0,1.2,3", help="comma-separated <END> bias offsets")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    kw = dict(num_vocab=10000, max_length=22, encode_dim_positions=84, encode_dim_features=2048, output_name="x",
              dropout=0.0)
    B, k = 512, 5
    f, p, _ = O.synthetic_batch(B, 36, 2048, 84, 22, 10000, seed=4321)
    f, p = f.to(DEV), p.to(DEV)
    cases = []
    for bias in (float(x) for x in a.end_bias.split(",")):
        torch.manual_seed(0)
        m = pkg.Transformer(device=DEV, **kw)
        with torch.no_grad():
            m.classifer.bias[2] += bias
        m = m.to(DEV).eval()
        runs = {"beam_search": lambda: m.beam_search(f, p, beam_size=k),
                "beam_search_nbest": lambda: m.beam_search_nbest(f, p, beam_size=k, length_penalty=0.6)}
        times = {name: [] for name in runs}
        for _ in range(a.rounds):
            for name, fn in runs.items():
                times[name].append(time_calls(fn, a.reps))
        _, _, lens = m.beam_search_nbest(f, p, beam_size=k, length_penalty=0.6)
        res = {name: round(statistics.median(v), 3) for name, v in times.items()}
        cases.append({"end_bias": bias, "ms_per_call": res,
                      "rounds_ms": {n: [round(x, 3) for x in v] for n, v in times.items()},
                      "nbest_over_beam": round(res["beam_search_nbest"] / res["beam_search"], 4),
                      "mean_len_best": round(float(lens[:, 0].float().mean()), 2),
                      "finished_fraction": round(float((lens < 21).float().mean()), 3)})
        del m
    out = {"workload": "model A bf16, 512 images x 36 regions, beam 5, graph replay", "cases": cases, **gpu_info()}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
