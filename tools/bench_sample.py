"""Throughput of the device sampler (Decoder.sample, one C call) and of one self-critical training step, at MSVD shape
(28 frames x 1536, V 4188, H 512, EMB 468, max 31 steps; single-layer LSTM decoder, seeded random weights, <EOS> lifted so that
captions end at different steps):

    sample_vs_greedy : batch 1024, eval and train mode, next to recnet_decoder_greedy on the same inputs
    sample_5x100     : 5 samples of each of 100 videos
    scst_step        : forward_decoder_self_critical at 5 x 100 + backward + ClipAdam step
    per_step_loop    : the reference point -- a Python loop over Decoder.forward with torch.multinomial, 5 x 100, one host read per step

The arms of a case run in ONE process, alternating their order round by round after a warm-up.  Every call ends in a host read or a
device synchronise, so a host clock around it measures the whole call.  Prints one line per arm and writes one JSON record (median ms
over rounds with the per-round spread, captions/s, steps decoded) with the GPU's name and power limit read in the same run.

    python tools/bench_sample.py [--rounds 5] [--reps 3] [--precisions bf16 fp32] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import recnet_b200  # noqa: E402,F401
from recnet_b200 import train as T  # noqa: E402
from recnet_b200.data import synthetic_batch  # noqa: E402

SHAPE = dict(T=28, E=1536, H=512, A=128, EMB=468, V=4188, steps=31)
EOS_BOOST = 4.0


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception:                      # noqa: BLE001 -- name from torch, limit unknown
        return torch.cuda.get_device_name(0), "unknown"


def build(precision, B):
    s, C = SHAPE, T.C
    C.decoder_model, C.decoder_n_layers, C.precision, C.device = "LSTM", 1, precision, "cuda:0"
    C.batch_size, C.caption_max_len, C.encoder_output_len, C.encoder_output_size = B, s["steps"] - 1, s["T"], s["E"]
    C.decoder_hidden_size, C.decoder_attn_size, C.embedding_size = s["H"], s["A"], s["EMB"]
    torch.manual_seed(1)
    dec = T.build_decoder(s["V"])
    with torch.no_grad():
        dec["model"].out.bias[2] += EOS_BOOST
    return dec


def per_step_sample(model, feats, K, steps):
    """Sampling the way a user has to without a device sampler: Decoder.forward step by step, torch.multinomial, host read per step."""
    x = feats.repeat(K, 1, 1).contiguous()
    N = x.shape[0]
    z = torch.zeros(1, N, SHAPE["H"], device=x.device)
    hid, tok = (z, z.clone()), torch.ones(1, N, dtype=torch.long, device=x.device)
    done = torch.zeros(N, dtype=torch.bool, device=x.device)
    ids = []
    with torch.no_grad(), model.cached_uv(x):
        for _ in range(steps):
            logits, hid = model(tok, hid, x)
            v = torch.multinomial(torch.softmax(logits.float(), dim=1), 1).view(-1)
            v = torch.where(done, torch.zeros_like(v), v)
            ids.append(v)
            done = done | (v == 2) | (v == 0)
            tok = v.view(1, -1)
            if bool(done.all()):
                break
    return len(ids)


def time_arms(arms, rounds, reps, warmup):
    steps = {}
    for k, f in arms.items():
        for _ in range(warmup):
            steps[k] = f()
    per = {k: [] for k in arms}
    for r in range(rounds):
        for k in (list(arms) if r % 2 == 0 else list(arms)[::-1]):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                steps[k] = arms[k]()
            torch.cuda.synchronize()
            per[k].append((time.perf_counter() - t0) * 1e3 / reps)
    return per, steps


def record(case, precision, rows, per, steps):
    med = {k: statistics.median(v) for k, v in per.items()}
    rec = {"case": case, "precision": precision, "rows": rows,
           "ms": {k: round(v, 3) for k, v in med.items()},
           "spread_ms": {k: [round(min(v), 3), round(max(v), 3)] for k, v in per.items()},
           "captions_per_s": {k: round(rows / v * 1e3) for k, v in med.items()},
           "steps_decoded": steps}
    for k in med:
        print(f"{case:16s} {precision} {k:14s}: {med[k]:8.2f} ms  ({rec['captions_per_s'][k]} captions/s, {steps[k]} steps)", flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3, help="calls per arm and round")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--precisions", nargs="+", default=["bf16", "fp32"], choices=["bf16", "fp32"])
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "r3_sample.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    s = SHAPE
    name, limit = gpu_info()
    results = []
    f1024, _, _ = synthetic_batch(1024, s["T"], s["E"], s["V"], s["steps"] - 1, seed=3)
    f100 = f1024[:100].cuda()
    f1024 = f1024.cuda()
    for precision in args.precisions:
        dec = build(precision, 1024)
        model = dec["model"]

        def sample(feats, K, train):
            def run():
                model.train(train)
                return int(model.sample(feats, K, max_steps=s["steps"])[3])
            return run

        def greedy():
            model.eval()
            return int(model.greedy(f1024, s["steps"])[1])

        per, steps = time_arms({"greedy": greedy, "sample_eval": sample(f1024, 1, False), "sample_train": sample(f1024, 1, True)},
                               args.rounds, args.reps, args.warmup)
        results.append(record("sample_vs_greedy", precision, 1024, per, steps))
        per, steps = time_arms({"sample_eval": sample(f100, 5, False), "sample_train": sample(f100, 5, True),
                                "per_step_loop": lambda: (model.eval(), per_step_sample(model, f100, 5, s["steps"]))[1]},
                               args.rounds, args.reps, args.warmup)
        results.append(record("sample_5x100", precision, 500, per, steps))
        reward = lambda a, b: (((a >= 3) & (a < 1000)).sum(0).float(), ((b >= 3) & (b < 1000)).sum(0).float())

        def scst():
            model.train()
            dec["optimizer"].zero_grad(set_to_none=True)
            loss, _, info = T.forward_decoder_self_critical(dec, f100, reward, n_samples=5, max_steps=s["steps"])
            loss.backward()
            dec["optimizer"].step()
            return int(info["ids"].shape[0])

        per, steps = time_arms({"scst_step": scst}, args.rounds, args.reps, args.warmup)
        results.append(record("scst_step", precision, 500, per, steps))
        del dec, model
        torch.cuda.empty_cache()
    out = {"workload": "sampling at MSVD shape (28 frames x 1536, V 4188, H 512, EMB 468, max 31 steps), single-layer LSTM decoder, "
                       f"seeded random weights with the <EOS> bias raised by {EOS_BOOST}; temperature 1; dropout p = 0.5 at every site in "
                       "train mode; rows = captions per call",
           "rounds": args.rounds, "reps_per_round": args.reps, "gpu": name, "power_limit": limit, "results": results}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": name, "power_limit": limit, "written": args.out}))


if __name__ == "__main__":
    main()
