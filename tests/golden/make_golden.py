"""Generate golden vectors by running the REAL reference (read-only at /root/reference).

Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

Writes tests/golden/<case>.npz.  Each file holds seeded inputs, the reference's
state_dict tensors, and what the reference's own train.forward_decoder /
forward_{global,local}_reconstructor / eval.greedy_search return on them, run on
CPU in fp64 (truth) -- losses, decoder hiddens, per-step logits, per-parameter
gradients of (decoder_loss + 1.0 * recon_loss) (train.py:260-268) and greedy ids.
Dropout is disabled (module.eval()) because the reference draws masks from
torch's global RNG, which no other implementation can reproduce.

Nothing here is copied into the product; the script only *calls* the reference.
"""
import os
import sys
import types

import numpy as np
import torch

REF = "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))
MAX_BYTES = 1 << 20                                          # largest fixture file kept in the repository
INPUTS = ("feats", "targets", "dec.", "global.", "local.")   # keys every fixture of a case shares (make_inputs + seeded weights)


def round_mantissa(a, bits=36):
    """fp64 rounded to `bits` mantissa bits (relative error <= 2^-(bits+1)); the zeroed low bits compress away."""
    if a.dtype != np.float64:
        return a
    drop = np.uint64(52 - bits)
    u = np.ascontiguousarray(a).view(np.uint64)
    return (((u + (np.uint64(1) << (drop - np.uint64(1)))) >> drop) << drop).view(np.float64).reshape(a.shape)


def save_golden(case, suffix, out):
    """Write <case><suffix>.npz.  A fixture larger than MAX_BYTES keeps its inputs once, exactly, in <case>_inputs.npz (shared by
    the case's eval and train fixtures) and its fp64 results rounded to 36-bit mantissas: a relative error <= 2^-37 = 7.3e-12,
    under 1 % of the tightest tolerance a test applies (1e-9).  tests/golden_util.py merges the two files again."""
    path = os.path.join(OUT, case + suffix + ".npz")
    np.savez_compressed(path, **out)
    if os.path.getsize(path) <= MAX_BYTES:
        return
    inputs = {k: v for k, v in out.items() if k.startswith(INPUTS)}
    np.savez_compressed(os.path.join(OUT, case + "_inputs.npz"), **inputs)
    np.savez_compressed(path, **{k: round_mantissa(v) for k, v in out.items() if k not in inputs})


def import_reference():
    """Stub the reference's off-path imports (SURVEY.md 8c) and import train/eval."""
    sys.path.insert(0, REF)

    def stub(name, **attrs):
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    stub("tensorboardX", SummaryWriter=object)
    stub("h5py")
    stub("coco_caption")
    stub("coco_caption.pycocotools")
    stub("coco_caption.pycocotools.msvd", MSVD=object)
    stub("coco_caption.pycocotools.utils", load_res=lambda *a, **k: None)
    stub("coco_caption.pycocoevalcap")
    stub("coco_caption.pycocoevalcap.eval", COCOEvalCap=object)
    try:
        import torchvision  # noqa: F401  (dataset/MSVD.py:10)
    except Exception:
        tv = stub("torchvision")
        tv.transforms = stub("torchvision.transforms", Compose=lambda x: x)
    import train as ref_train
    import eval as ref_eval
    return ref_train, ref_eval


CASES = {
    # name: dict(B, T, E, H, A, EMB, V, R, dec_layers, rec_layers, cap_len, model)
    "tiny_lstm":        dict(B=4, T=5, E=24, H=16, A=8, EMB=12, V=37, dec_layers=1, rec_layers=1, cap_len=6, dec_model="LSTM", rec_model="LSTM", seed=11),
    "tiny_lstm_ragged": dict(B=5, T=7, E=20, H=12, A=8, EMB=10, V=29, dec_layers=1, rec_layers=1, cap_len=9, dec_model="LSTM", rec_model="LSTM", seed=12, short=True),
    "tiny_lstm_2layer": dict(B=3, T=4, E=16, H=8, A=8, EMB=6, V=23, dec_layers=2, rec_layers=1, cap_len=5, dec_model="LSTM", rec_model="LSTM", seed=13),
    "tiny_gru":         dict(B=4, T=5, E=24, H=16, A=8, EMB=12, V=37, dec_layers=1, rec_layers=1, cap_len=6, dec_model="GRU", rec_model="GRU", seed=14),
    # variants that run through the per-step operator path (no fused sequence driver): stacked GRU decoder, GRU reconstructors over
    # a stacked decoder, multi-layer reconstructors
    "tiny_gru_2layer":  dict(B=3, T=4, E=16, H=8, A=8, EMB=6, V=23, dec_layers=2, rec_layers=1, cap_len=5, dec_model="GRU", rec_model="GRU", seed=16),
    "tiny_lstm_rec2":   dict(B=3, T=4, E=16, H=8, A=8, EMB=6, V=23, dec_layers=1, rec_layers=2, cap_len=5, dec_model="LSTM", rec_model="LSTM", seed=17),
    "tiny_mixed_2x2":   dict(B=3, T=4, E=16, H=8, A=8, EMB=6, V=23, dec_layers=2, rec_layers=2, cap_len=5, dec_model="LSTM", rec_model="GRU", seed=18),
    "small_lstm":       dict(B=8, T=28, E=64, H=32, A=16, EMB=20, V=101, dec_layers=1, rec_layers=1, cap_len=30, dec_model="LSTM", rec_model="LSTM", seed=15),
}


def make_inputs(c):
    g = torch.Generator().manual_seed(c["seed"])
    B, T, E, V, cap = c["B"], c["T"], c["E"], c["V"], c["cap_len"]
    feats = torch.randn(B, T, E, generator=g, dtype=torch.float64)
    lens = torch.randint(min(2, cap), cap + 1, (B,), generator=g)
    if c.get("short"):
        lens = torch.clamp(lens, max=cap - 3)    # forces the early break at train.py:66
    else:
        lens[0] = cap
    targets = torch.zeros(cap + 1, B, dtype=torch.long)
    for b in range(B):
        n = int(lens[b])
        targets[:n, b] = torch.randint(3, V, (n,), generator=g)
        targets[n, b] = 2
    return feats, targets


def run_case(name, c, ref_train, ref_eval):
    C = ref_train.C
    C.device = "cpu"
    ref_eval.C.device = "cpu"
    C.decoder_model, C.reconstructor_model = c["dec_model"], c["rec_model"]
    C.batch_size = c["B"]
    C.caption_max_len = c["cap_len"]
    C.encoder_output_len, C.encoder_output_size = c["T"], c["E"]
    C.decoder_n_layers, C.decoder_hidden_size, C.decoder_attn_size = c["dec_layers"], c["H"], c["A"]
    C.embedding_size = c["EMB"]
    C.reconstructor_n_layers, C.reconstructor_hidden_size, C.reconstructor_attn_size = c["rec_layers"], c["E"], c["A"]
    out = {}
    feats, targets = make_inputs(c)
    masks = targets > 0
    out["feats"], out["targets"] = feats.numpy(), targets.numpy()
    out["meta"] = np.array(repr(c))

    torch.manual_seed(c["seed"])
    dec = ref_train.build_decoder(c["V"])
    dec["model"].double().eval()
    for k, v in dec["model"].state_dict().items():
        out["dec." + k] = v.numpy().copy()

    for kind in ("none", "global", "local"):
        dec["model"].zero_grad()
        dloss, hiddens, _ = ref_train.forward_decoder(dec, feats, targets, masks, 1.0)
        if kind == "none":
            out["dec_loss"] = dloss.detach().numpy()
            out["hiddens"] = hiddens.detach().numpy()
            dloss.backward()
            for k, p in dec["model"].named_parameters():
                out["grad_none.dec." + k] = p.grad.numpy().copy()
            continue
        C.reconstructor_type = kind
        torch.manual_seed(c["seed"] + 100)
        rec = ref_train.build_reconstructor()
        rec["model"].double().eval()
        for k, v in rec["model"].state_dict().items():
            out[f"{kind}." + k] = v.numpy().copy()
        fwd = ref_train.forward_global_reconstructor if kind == "global" else ref_train.forward_local_reconstructor
        rloss = fwd(hiddens, feats, rec)
        out[f"{kind}_loss"] = rloss.detach().numpy()
        (dloss + 1.0 * rloss).backward()                                # train.py:260,268
        for k, p in dec["model"].named_parameters():
            out[f"grad_{kind}.dec." + k] = p.grad.numpy().copy()
        for k, p in rec["model"].named_parameters():
            out[f"grad_{kind}.{kind}." + k] = p.grad.numpy().copy()

    # greedy (eval.py:19-33) and the teacher-forcing-off branch of forward_decoder (train.py:47-51)
    with torch.no_grad():
        B = c["B"]
        tok = torch.full((1, B), 1, dtype=torch.long)
        if c["dec_model"] == "LSTM":
            hid = (torch.zeros(c["dec_layers"], B, c["H"], dtype=torch.float64),
                   torch.zeros(c["dec_layers"], B, c["H"], dtype=torch.float64))
        else:
            hid = torch.zeros(c["dec_layers"], B, c["H"], dtype=torch.float64)
        ids = ref_eval.greedy_search(C, dec["model"], tok, hid, feats)
        out["greedy_ids"] = np.array([[int(x) for x in row] for row in ids], dtype=np.int64)
        # single decoder step logits at t=0 (Decoder.forward, models/decoder.py:45-70)
        logits0, _ = dec["model"](tok, hid, feats)
        out["step0_logits"] = logits0.numpy()
    save_golden(name, "", out)
    print(name, "dec_loss", float(out["dec_loss"]), "global", float(out["global_loss"]), "local", float(out["local_loss"]),
          "L", out["hiddens"].shape[0], "greedy steps", out["greedy_ids"].shape[0])


if __name__ == "__main__":
    if not os.path.isdir(REF):
        sys.exit("reference not mounted; golden files are committed, nothing to do")
    rt, re_ = import_reference()
    # train.forward_* build their zero states with torch.zeros(...) (train.py:28-35): make that fp64 too
    torch.set_default_dtype(torch.float64)
    only = sys.argv[1:]                      # optional: case names to (re)generate; default = all
    for n, c in CASES.items():
        if not only or n in only:
            run_case(n, c, rt, re_)
