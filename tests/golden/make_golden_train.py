"""Golden vectors the eval-mode fixtures of make_golden.py cannot give, again by running the REAL reference
(read-only at /root/reference; build container only):

    python tests/golden/make_golden_train.py

1. ``<case>_train.npz`` -- the reference's train.forward_decoder / forward_{global,local}_reconstructor in TRAIN mode (fp64):
   the reference's three nn.Dropout modules (models/decoder.py:48,69, models/local_reconstructor.py:50,
   models/global_reconstructor.py:38) are swapped for a module that applies caller-supplied inverted-dropout scales, and the
   scales are the ones the CUDA path draws for (seed, offset = 1) -- tests/philox_ref.py, a numpy restatement of the in-kernel
   Philox generator.  So the same masks reach the reference, the oracle and the kernels, and loss + every gradient of
   (decoder_loss + 1.0 * recon_loss) can be compared in the configuration bench.py times (dropout on).
2. ``<case>_beam.npz`` -- the reference's own eval.beam_search (eval.py:36-120) for widths 3 and 5.  Its body builds
   torch.cuda.FloatTensor objects (eval.py:39,57), so it only runs on a GPU as written; here that constructor is aliased to a CPU
   tensor constructor for the duration of the call (nothing else is touched), which pins both our device beam search and the
   oracle's restatement to ids the reference itself produced.

Nothing here is copied into the product; the script only *calls* the reference.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from tests.golden.make_golden import CASES, OUT, REF, import_reference, make_inputs, save_golden      # noqa: E402
from tests.philox_ref import SITE_EMB, SITE_GLOBAL_MP, SITE_LOCAL_X, SITE_LOGITS, dropout_scales      # noqa: E402

SEEDS = {"dec": 0xDEC0, "local": 0x10CA, "global": 0x610B}     # models.py: _init_rng seeds; offset is 1 in the first training forward


class ScaleDropout(torch.nn.Module):
    """Stands in for nn.Dropout: call k multiplies by scales[k] (0 or 1/(1-p)), reshaped to the input."""

    def __init__(self, scales):
        super().__init__()
        self.scales, self.k = scales, 0

    def forward(self, x):
        s = self.scales[self.k].reshape(x.shape)
        self.k += 1
        return x * s


def configure(C, c):
    C.decoder_model, C.reconstructor_model = c["dec_model"], c["rec_model"]
    C.batch_size, C.caption_max_len = c["B"], c["cap_len"]
    C.encoder_output_len, C.encoder_output_size = c["T"], c["E"]
    C.decoder_n_layers, C.decoder_hidden_size, C.decoder_attn_size = c["dec_layers"], c["H"], c["A"]
    C.embedding_size = c["EMB"]
    C.reconstructor_n_layers, C.reconstructor_hidden_size, C.reconstructor_attn_size = c["rec_layers"], c["E"], c["A"]


def train_case(name, c, ref_train):
    C = ref_train.C
    C.device = "cpu"
    configure(C, c)
    B, Tn, H, EMB, V, cap = c["B"], c["T"], c["H"], c["EMB"], c["V"], c["cap_len"]
    feats, targets = make_inputs(c)
    masks = targets > 0
    Lmax = cap + 1
    p_emb, p_out, p_rec = C.embedding_dropout, C.decoder_out_dropout, C.reconstructor_decoder_dropout
    out = {"meta": np.array(repr(c)), "feats": feats.numpy(), "targets": targets.numpy(),
           "p": np.array([p_emb, p_out, p_rec]), "seeds": np.array([SEEDS["dec"], SEEDS["local"], SEEDS["global"]], dtype=np.int64)}
    emb_s = torch.from_numpy(dropout_scales(SEEDS["dec"], 1, SITE_EMB, Lmax * B * EMB, p_emb)).double().view(Lmax, B, EMB)
    log_s = torch.from_numpy(dropout_scales(SEEDS["dec"], 1, SITE_LOGITS, Lmax * B * V, p_out)).double().view(Lmax, B, V)

    torch.manual_seed(c["seed"])
    dec = ref_train.build_decoder(V)
    dec["model"].double().train()
    for k, v in dec["model"].state_dict().items():
        out["dec." + k] = v.numpy().copy()
    for kind in ("none", "global", "local"):
        dec["model"].zero_grad()
        dec["model"].embedding_dropout = ScaleDropout(emb_s)
        dec["model"].out_dropout = ScaleDropout(log_s)
        dloss, hiddens, _ = ref_train.forward_decoder(dec, feats, targets, masks, 1.0)
        L = hiddens.shape[0]
        if kind == "none":
            out["dec_loss"], out["hiddens"] = dloss.detach().numpy(), hiddens.detach().numpy()
            dloss.backward()
            for k, p in dec["model"].named_parameters():
                out["grad_none.dec." + k] = p.grad.numpy().copy()
            continue
        C.reconstructor_type = kind
        torch.manual_seed(c["seed"] + 100)
        rec = ref_train.build_reconstructor()
        rec["model"].double().train()
        for k, v in rec["model"].state_dict().items():
            out[f"{kind}." + k] = v.numpy().copy()
        if kind == "local":
            sc = torch.from_numpy(dropout_scales(SEEDS["local"], 1, SITE_LOCAL_X, Tn * B * H, p_rec)).double().view(Tn, B, H)
        else:
            sc = torch.from_numpy(dropout_scales(SEEDS["global"], 1, SITE_GLOBAL_MP, L * B * H, p_rec)).double().view(L, B, H)
        rec["model"].decoder_dropout = ScaleDropout(sc)
        fwd = ref_train.forward_global_reconstructor if kind == "global" else ref_train.forward_local_reconstructor
        rloss = fwd(hiddens, feats, rec)
        out[f"{kind}_loss"] = rloss.detach().numpy()
        (dloss + 1.0 * rloss).backward()
        for k, p in dec["model"].named_parameters():
            out[f"grad_{kind}.dec." + k] = p.grad.numpy().copy()
        for k, p in rec["model"].named_parameters():
            out[f"grad_{kind}.{kind}." + k] = p.grad.numpy().copy()
    save_golden(name, "_train", out)
    print(name + "_train", "dec_loss", float(out["dec_loss"]), "global", float(out["global_loss"]), "local", float(out["local_loss"]))


class _Vocab:
    def __init__(self, n):
        self.n_vocabs = n
        self.word2idx = {'<PAD>': 0, '<SOS>': 1, '<EOS>': 2}


def beam_case(name, c, ref_train, ref_eval):
    C = ref_train.C
    C.device = "cpu"
    ref_eval.C.device = "cpu"
    configure(C, c)
    feats, _ = make_inputs(c)
    B, H, V = c["B"], c["H"], c["V"]
    saved = torch.cuda.FloatTensor
    torch.cuda.FloatTensor = lambda x: torch.tensor(np.asarray(x), dtype=torch.float64)      # eval.py:39,57 on the CPU
    best = None
    try:
        # default-init logits are almost flat and never emit <EOS>: spread them (out.weight *= scale) and lift <EOS> (bias += boost);
        # of a small fixed grid keep the setting whose captions are the most varied AND contain <EOS> before the last step, so that
        # the beam bookkeeping and the length normalisation of eval.py:51-59 are both exercised
        for scale in (6.0, 12.0, 20.0):
            for boost in (0.5, 1.5, 3.0, 5.0):
                torch.manual_seed(c["seed"])
                dec = ref_train.build_decoder(V)
                dec["model"].double().eval()
                with torch.no_grad():
                    dec["model"].out.weight *= scale
                    dec["model"].out.bias[2] += boost
                res = {}
                for width in (3, 5):
                    tok = torch.full((1, B), 1, dtype=torch.long)
                    z = torch.zeros(1, B, H, dtype=torch.float64)
                    hid = (z, z.clone()) if c["dec_model"] == "LSTM" else z
                    with torch.no_grad():
                        ids = ref_eval.beam_search(C, width, _Vocab(V), dec["model"], tok, hid, feats)
                    n = max(len(r) for r in ids)
                    arr = np.full((B, n), -1, dtype=np.int64)
                    for b, r in enumerate(ids):
                        arr[b, :len(r)] = r
                    res[width] = arr
                a3 = res[3]
                eos_mid = int(((a3[:, :-1] == 2).any(axis=1) & (a3[:, 0] != 2)).sum())
                score = len({tuple(r) for r in a3.tolist()}) + len(np.unique(a3)) + 3 * eos_mid + int((res[3] != res[5][:, :res[3].shape[1]]).any()) * 2 \
                    if res[3].shape == res[5].shape else 0
                if best is None or score > best[0]:
                    best = (score, scale, boost, res, {k: v.numpy().copy() for k, v in dec["model"].state_dict().items()})
    finally:
        torch.cuda.FloatTensor = saved
    score, scale, boost, res, sd = best
    out = {"meta": np.array(repr(c)), "feats": feats.numpy(), "logit_scale": np.array(scale), "eos_boost": np.array(boost)}
    for k, v in sd.items():
        out["dec." + k] = v
    for width, arr in res.items():
        out[f"beam{width}"] = arr
        print(name + "_beam", "scale", scale, "boost", boost, "width", width, "steps", arr.shape[1], arr[:, :10].tolist())
    np.savez_compressed(os.path.join(OUT, name + "_beam.npz"), **out)


if __name__ == "__main__":
    if not os.path.isdir(REF):
        sys.exit("reference not mounted; golden files are committed, nothing to do")
    rt, re_ = import_reference()
    torch.set_default_dtype(torch.float64)
    if "--beam-only" not in sys.argv:
        train_case("small_lstm", CASES["small_lstm"], rt)
        train_case("tiny_lstm_ragged", CASES["tiny_lstm_ragged"], rt)
    for n in ("tiny_lstm", "tiny_gru", "small_lstm"):
        beam_case(n, CASES[n], rt, re_)
