"""Decoding throughput of stacked LSTM decoders: the device loops (recnet_decoder_greedy / recnet_decoder_beam, one C call each) against
the per-step loops over Decoder.forward (the step-wise greedy, and eval.beam_search with RECNET_BEAM_DEVICE=0), at n_layers 1, 2 and 4.

    greedy: batch 1024, 28 frames x 1536, max 31 steps (BASELINE config 4 shape)
    beam:   width 5, batch 100, same features and length

Both arms of a case run in ONE process, alternating their order round by round after a warm-up, on the same weights (seeded random init)
and inputs (resident on the device).  Each call ends in a host read, so a host clock around it measures the whole decode.  Prints one line
per case and one JSON record (ms per batch as the median over rounds with the per-round spread, captions/s, the steps each arm decoded,
the share of ids on which the two arms agree) with the GPU's name and power limit read in the same run.

    python tools/bench_stacked_decode.py [--rounds 5] [--reps 3] [--layers 1 2 4] [--precisions bf16 fp32] [--out FILE]
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
from recnet_b200 import eval as E  # noqa: E402
from recnet_b200 import train as T  # noqa: E402
from recnet_b200.data import synthetic_batch  # noqa: E402

SHAPE = dict(T=28, E=1536, H=512, A=128, EMB=468, V=4188, steps=31)
CASES = {"greedy": dict(B=1024), "beam": dict(B=100, width=5)}


class _Vocab:
    def __init__(self, n):
        self.n_vocabs = n
        self.word2idx = {'<PAD>': 0, '<SOS>': 1, '<EOS>': 2}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception:                      # noqa: BLE001 -- name from torch, limit unknown
        return torch.cuda.get_device_name(0), "unknown"


def build_decoder(n_layers, precision, B):
    s, C = SHAPE, T.C
    C.decoder_model, C.decoder_n_layers, C.precision, C.device = "LSTM", n_layers, precision, "cuda:0"
    C.batch_size, C.caption_max_len, C.encoder_output_len, C.encoder_output_size = B, s["steps"] - 1, s["T"], s["E"]
    C.decoder_hidden_size, C.decoder_attn_size, C.embedding_size = s["H"], s["A"], s["EMB"]
    torch.manual_seed(n_layers)
    dec = T.build_decoder(s["V"])["model"].eval()
    assert dec.n_layers == n_layers and dec.uses_fused_sequence
    return dec


def arms(kind, dec, feats):
    """{arm: call returning the decoded ids as a (steps, B) host tensor}; every call ends in a host read."""
    B = feats.shape[0]
    steps = SHAPE["steps"]
    if kind == "greedy":
        def device():
            ids, n = dec.greedy(feats, steps)
            return ids[: int(n)].cpu()

        def per_step():
            ids, n = dec._greedy_stepwise(feats, steps)
            return ids[: int(n)].cpu()
        return {"device": device, "per_step": per_step}
    width, vocab = CASES["beam"]["width"], _Vocab(SHAPE["V"])
    tok = torch.ones(1, B, dtype=torch.long, device=feats.device)
    z = torch.zeros(dec.n_layers, B, SHAPE["H"], device=feats.device)

    def beam(flag):
        def run():
            saved = os.environ.get("RECNET_BEAM_DEVICE")
            os.environ["RECNET_BEAM_DEVICE"] = flag               # read by eval.beam_search on every call
            try:
                seqs = E.beam_search(T.C, width, vocab, dec, tok, (z, z.clone()), feats)
            finally:
                if saved is None:
                    os.environ.pop("RECNET_BEAM_DEVICE")
                else:
                    os.environ["RECNET_BEAM_DEVICE"] = saved
            n = max(len(s) for s in seqs)
            return torch.tensor([s + [-1] * (n - len(s)) for s in seqs]).t()
        return run
    return {"device": beam("1"), "per_step": beam("0")}


def time_call(f, reps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = f()
    return (time.perf_counter() - t0) * 1e3 / reps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3, help="calls per arm and round")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--layers", type=int, nargs="+", default=[1, 2, 4])
    ap.add_argument("--precisions", nargs="+", default=["bf16", "fp32"], choices=["bf16", "fp32"])
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "r3_stacked_decode.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    s = SHAPE
    name, limit = gpu_info()
    results = []
    for kind, case in CASES.items():
        feats, _, _ = synthetic_batch(case["B"], s["T"], s["E"], s["V"], s["steps"] - 1, seed=3)
        feats = feats.cuda()
        for precision in args.precisions:
            for nl in args.layers:
                dec = build_decoder(nl, precision, case["B"])
                fs = arms(kind, dec, feats)
                outs = {}
                for k, f in fs.items():
                    for _ in range(args.warmup):
                        outs[k] = f()
                per = {k: [] for k in fs}
                for r in range(args.rounds):
                    for k in (list(fs) if r % 2 == 0 else list(fs)[::-1]):
                        ms, outs[k] = time_call(fs[k], args.reps)
                        per[k].append(ms)
                med = {k: statistics.median(v) for k, v in per.items()}
                a, b = outs["device"], outs["per_step"]
                n = min(a.shape[0], b.shape[0])
                rec = {"case": kind, "precision": precision, "n_layers": nl, "batch": case["B"], "beam_width": case.get("width"),
                       "ms_per_batch": {k: round(v, 3) for k, v in med.items()},
                       "spread_ms": {k: [round(min(v), 3), round(max(v), 3)] for k, v in per.items()},
                       "captions_per_s": {k: round(case["B"] / v * 1e3) for k, v in med.items()},
                       "speedup": round(med["per_step"] / med["device"], 2),
                       "steps_decoded": {"device": int(a.shape[0]), "per_step": int(b.shape[0])},
                       "id_agreement": round(float((a[:n] == b[:n]).float().mean()), 4) if n else None}
                results.append(rec)
                print(f"{kind:6s} {precision} NL={nl}: device {med['device']:.2f} ms ({rec['captions_per_s']['device']} captions/s), "
                      f"per-step {med['per_step']:.2f} ms ({rec['captions_per_s']['per_step']} captions/s), x{rec['speedup']}, "
                      f"agreement {rec['id_agreement']}", flush=True)
                del dec
                torch.cuda.empty_cache()
    out = {"workload": "decoding, 28 frames x 1536, V 4188, H 512, max 31 steps: greedy batch 1024, beam width 5 batch 100; LSTM decoder, "
                       "seeded random weights, eval mode",
           "rounds": args.rounds, "reps_per_round": args.reps, "gpu": name, "power_limit": limit, "results": results}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": name, "power_limit": limit, "written": args.out}))


if __name__ == "__main__":
    main()
