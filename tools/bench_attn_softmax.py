"""Cost of the opt-in softmax attention on the bench.py train step (MSVD shape, batch 100, 1-layer LSTM decoder + 1-layer LSTM local
reconstructor, train mode, CUDA graph, inputs resident on the device): the step with attn_softmax off (the reference's mean attention,
what bench.py times) and on, captured as two graphs in ONE process and replayed in alternating rounds after a warm-up, so that both arms
see the same clocks and neighbours.  Prints one JSON line: median ms/step per arm, the per-round spread, the relative cost, and the GPU's
name and power limit read in the same run.

    python tools/bench_attn_softmax.py [--rounds 8] [--steps 50] [--warmup 10] [--precision bf16] [--profile DIR]

--profile DIR: additionally one torch.profiler run per arm (separate from the timed rounds), kernel table written to DIR.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import recnet_b200  # noqa: E402,F401
from recnet_b200 import train as T  # noqa: E402
from recnet_b200.data import synthetic_batch  # noqa: E402

SHAPE = dict(B=100, T=28, E=1536, H=512, A=128, EMB=468, V=4188, cap=30, R=1536)     # bench.py's workload


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception:                      # noqa: BLE001 -- name from torch, limit unknown
        return torch.cuda.get_device_name(0), "unknown"


def build_arm(softmax, precision, feats, targets):
    s, C = SHAPE, T.C
    C.decoder_model = C.reconstructor_model = "LSTM"
    C.batch_size, C.caption_max_len, C.encoder_output_len, C.encoder_output_size = s["B"], s["cap"], s["T"], s["E"]
    C.decoder_n_layers, C.decoder_hidden_size, C.decoder_attn_size, C.embedding_size = 1, s["H"], s["A"], s["EMB"]
    C.reconstructor_n_layers, C.reconstructor_hidden_size, C.reconstructor_attn_size = 1, s["R"], s["A"]
    C.use_recon, C.reconstructor_type, C.precision, C.device = True, "local", precision, "cuda:0"
    C.decoder_attn_softmax = C.reconstructor_attn_softmax = softmax
    torch.manual_seed(0)
    dec, rec = T.build_decoder(s["V"]), T.build_reconstructor()
    assert dec["model"].attn_softmax is softmax and rec["model"].attn_softmax is softmax
    loss_d = torch.zeros((), device="cuda:0")

    def step():
        loss, _, _ = T.train_step(dec, rec, feats, targets, n_steps=s["cap"] + 1)
        loss_d.copy_(loss.detach())

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    assert dec["model"].uses_fused_sequence and rec["model"]._fused_ok(torch.empty(31, 1, 1, 1))
    return graph, step, loss_d


def time_replays(graph, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--profile", metavar="DIR")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    s = SHAPE
    feats, targets, _ = synthetic_batch(s["B"], s["T"], s["E"], s["V"], s["cap"], seed=1234)
    feats, targets = feats.cuda(), targets.cuda()
    arms = {"mean": build_arm(False, args.precision, feats, targets), "softmax": build_arm(True, args.precision, feats, targets)}
    for g, _, _ in arms.values():
        for _ in range(args.warmup):
            g.replay()
    torch.cuda.synchronize()
    per = {k: [] for k in arms}
    for r in range(args.rounds):
        order = list(arms) if r % 2 == 0 else list(arms)[::-1]
        for k in order:
            per[k].append(time_replays(arms[k][0], args.steps))
    losses = {k: float(v[2]) for k, v in arms.items()}
    name, limit = gpu_info()
    med = {k: statistics.median(v) for k, v in per.items()}
    out = {"workload": "bench.py train step: MSVD shape, batch 100, LSTM decoder + LSTM local reconstructor, train mode, CUDA graph",
           "precision": args.precision, "rounds": args.rounds, "steps_per_round": args.steps,
           "ms_per_step": {k: round(v, 4) for k, v in med.items()},
           "spread_ms": {k: [round(min(v), 4), round(max(v), 4)] for k, v in per.items()},
           "softmax_cost_pct": round(100.0 * (med["softmax"] / med["mean"] - 1.0), 2),
           "last_loss": losses, "gpu": name, "power_limit": limit}
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(args.profile, exist_ok=True)
        for k, (g, _, _) in arms.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    g.replay()
                torch.cuda.synchronize()
            with open(os.path.join(args.profile, f"attn_softmax_{k}_kernels.txt"), "w") as f:
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=40))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
