"""Time of CIDEr-D on the device (CiderCorpus.score, one kernel launch) against the fp64 Python oracle, and of one self-critical
training step with the CIDEr-D reward against the synthetic reward of tools/bench_sample.py.

Corpus: seeded and MSVD-shaped (data.synthetic_captions): 1200 videos x 40 references, 3-30 words, Zipf ids over V 9000.
Candidates: seeded Zipf captions of 3-30 words ended by <EOS>, padded to 31 steps, time-major, each scored against a random video.

    score        : rows 500 (5 samples x 100 videos) and 1024; CUDA events around `--calls` back-to-back calls after a warm-up,
                   median per call over `--rounds` rounds; the oracle (tests/cider_oracle.py) once on the same rows, host clock;
                   the largest |device - oracle| / max(1, |oracle|) on those rows
    scst_step    : tools/bench_sample.py's SCST step (forward_decoder_self_critical at 5 x 100 + backward + ClipAdam step) with
                   CiderCorpus.reward_fn against a corpus of the same shape over the decoder's V 4188, next to the synthetic reward,
                   arms alternated round by round in one process

Writes one JSON record with the GPU's name and power limit read in the same run.

    python tools/bench_cider.py [--rounds 5] [--calls 200] [--precisions bf16 fp32] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import recnet_b200  # noqa: E402,F401
from recnet_b200 import train as T  # noqa: E402
from recnet_b200.cider import CiderCorpus  # noqa: E402
from recnet_b200.data import synthetic_batch, synthetic_captions  # noqa: E402
from tests import cider_oracle as CO  # noqa: E402
import bench_sample as BS  # noqa: E402

N_VIDEOS, N_REFS, V, STEPS = 1200, 40, 9000, 31


def candidates(n, seed, vocab=V):
    caps = synthetic_captions(n, 1, vocab, seed=seed)
    rows = np.zeros((STEPS, n), dtype=np.int64)
    for i, (c,) in enumerate(caps):
        rows[: len(c), i] = c
    vids = np.random.default_rng(seed + 1).integers(0, N_VIDEOS, size=n)
    return torch.from_numpy(rows), vids


def time_score(cc, ids, vidx, rounds, calls):
    for _ in range(20):
        cc.score(ids, vidx)
    torch.cuda.synchronize()
    per = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(calls):
            cc.score(ids, vidx)
        e1.record()
        e1.synchronize()
        per.append(e0.elapsed_time(e1) / calls)
    return per


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=200, help="score calls per timed round")
    ap.add_argument("--reps", type=int, default=3, help="SCST steps per arm and round")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--precisions", nargs="+", default=["bf16", "fp32"], choices=["bf16", "fp32"])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_cider.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, limit = BS.gpu_info()
    dev = torch.device("cuda:0")
    refs = synthetic_captions(N_VIDEOS, N_REFS, V, seed=11)
    t0 = time.perf_counter()
    cc = CiderCorpus(refs, dev)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    oracle = CO.Corpus(refs)
    oracle_build_s = time.perf_counter() - t0
    results = []
    for rows in (500, 1024):
        ids, vids = candidates(rows, seed=rows)
        ids_d, vidx = ids.to(dev), torch.from_numpy(vids).to(dev)
        per = time_score(cc, ids_d, vidx, args.rounds, args.calls)
        scores = cc.score(ids_d, vidx).double().cpu()
        t0 = time.perf_counter()
        ref = torch.tensor(oracle.scores(ids.t().tolist(), vids.tolist()), dtype=torch.float64)
        host_ms = (time.perf_counter() - t0) * 1e3
        err = float(((scores - ref).abs() / ref.abs().clamp(min=1.0)).max())
        rec = {"case": "score", "rows": rows, "device_ms": round(statistics.median(per), 4),
               "device_spread_ms": [round(min(per), 4), round(max(per), 4)], "oracle_host_ms": round(host_ms, 1),
               "max_scaled_err_vs_oracle": err, "mean_cider_d": round(float(scores.mean()), 5)}
        print(f"score {rows:5d} rows: device {rec['device_ms']:.4f} ms/call, fp64 oracle {host_ms:.1f} ms, max err {err:.2e}", flush=True)
        results.append(rec)

    s = BS.SHAPE
    scst_refs = synthetic_captions(N_VIDEOS, N_REFS, s["V"], seed=12)
    scst_cc = CiderCorpus(scst_refs, dev)
    f100 = synthetic_batch(100, s["T"], s["E"], s["V"], s["steps"] - 1, seed=3)[0].to(dev)
    cider_reward = scst_cc.reward_fn(scst_cc.index(range(100)))
    synthetic = lambda a, b: (((a >= 3) & (a < 1000)).sum(0).float(), ((b >= 3) & (b < 1000)).sum(0).float())
    for precision in args.precisions:
        dec = BS.build(precision, 100)
        model = dec["model"]

        def scst(reward):
            def run():
                model.train()
                dec["optimizer"].zero_grad(set_to_none=True)
                loss, _, info = T.forward_decoder_self_critical(dec, f100, reward, n_samples=5, max_steps=s["steps"])
                loss.backward()
                dec["optimizer"].step()
                return int(info["ids"].shape[0])
            return run

        per, steps = BS.time_arms({"cider_reward": scst(cider_reward), "synthetic_reward": scst(synthetic)}, args.rounds, args.reps,
                                  args.warmup)
        results.append(BS.record("scst_step", precision, 500, per, steps))
        del dec, model
        torch.cuda.empty_cache()
    out = {"workload": f"CIDEr-D on a seeded MSVD-shaped corpus ({N_VIDEOS} videos x {N_REFS} references, 3-30 words, Zipf ids over "
                       f"V {V}; {int(cc.df_keys.size)} distinct n-grams); candidates: Zipf captions of 3-30 words, {STEPS} steps, "
                       "time-major; scst_step: tools/bench_sample.py's SCST step at 5 x 100 (bf16/fp32, MSVD-shape decoder, V "
                       f"{s['V']}) against a corpus of the same shape over V {s['V']}",
           "rounds": args.rounds, "calls_per_round": args.calls, "corpus_build_host_s": round(build_s, 2),
           "oracle_build_host_s": round(oracle_build_s, 2), "gpu": name, "power_limit": limit, "results": results}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": name, "power_limit": limit, "written": args.out}))


if __name__ == "__main__":
    main()
