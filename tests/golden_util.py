"""Load the reference-generated golden fixtures (tests/golden/*.npz)."""
import ast
import glob
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_cases():
    """Eval-mode fixtures of make_golden.py (the train-mode / beam fixtures of make_golden_train.py have their own loaders below)."""
    names = sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))
    return [n for n in names if not n.endswith(("_train", "_beam", "_inputs"))]


def _arrays(name, suffix=""):
    """<name><suffix>.npz, plus <name>_inputs.npz where the case keeps its shared inputs apart (make_golden.save_golden)."""
    z = dict(np.load(os.path.join(GOLDEN_DIR, name + suffix + ".npz")))
    shared = os.path.join(GOLDEN_DIR, name + "_inputs.npz")
    if os.path.exists(shared):
        z.update(np.load(shared))
    return z


def load_golden(name, dtype=torch.float64):
    z = _arrays(name)
    meta = ast.literal_eval(str(z["meta"]))

    def group(prefix):
        out = {}
        for k in z:
            if k.startswith(prefix):
                t = torch.from_numpy(z[k])
                out[k[len(prefix):]] = t.to(dtype) if t.is_floating_point() else t
        return out

    g = {
        "meta": meta,
        "feats": torch.from_numpy(z["feats"]).to(dtype),
        "targets": torch.from_numpy(z["targets"]),
        "dec": group("dec."), "global": group("global."), "local": group("local."),
        "dec_loss": float(z["dec_loss"]), "global_loss": float(z["global_loss"]), "local_loss": float(z["local_loss"]),
        "hiddens": torch.from_numpy(z["hiddens"]).to(dtype),
        "greedy_ids": torch.from_numpy(z["greedy_ids"]),
        "step0_logits": torch.from_numpy(z["step0_logits"]).to(dtype),
        "grads": {kind: group(f"grad_{kind}.") for kind in ("none", "global", "local")},
    }
    return g


def load_golden_train(name, dtype=torch.float64):
    """<name>_train.npz: the reference in TRAIN mode with the Philox masks of tests/philox_ref.py injected (make_golden_train.py)."""
    z = _arrays(name, "_train")
    meta = ast.literal_eval(str(z["meta"]))

    def group(prefix):
        out = {}
        for k in z:
            if k.startswith(prefix):
                t = torch.from_numpy(z[k])
                out[k[len(prefix):]] = t.to(dtype) if t.is_floating_point() else t
        return out

    p_emb, p_out, p_rec = (float(x) for x in z["p"])
    seeds = [int(x) for x in z["seeds"]]
    return {"meta": meta, "feats": torch.from_numpy(z["feats"]).to(dtype), "targets": torch.from_numpy(z["targets"]),
            "dec": group("dec."), "global": group("global."), "local": group("local."),
            "dec_loss": float(z["dec_loss"]), "global_loss": float(z["global_loss"]), "local_loss": float(z["local_loss"]),
            "hiddens": torch.from_numpy(z["hiddens"]).to(dtype),
            "grads": {kind: group(f"grad_{kind}.") for kind in ("none", "global", "local")},
            "p_emb": p_emb, "p_out": p_out, "p_rec": p_rec, "seed_dec": seeds[0], "seed_local": seeds[1], "seed_global": seeds[2]}


def load_golden_beam(name, dtype=torch.float64):
    """<name>_beam.npz: ids the reference's own eval.beam_search returned (widths 3 and 5), rows padded with -1."""
    z = np.load(os.path.join(GOLDEN_DIR, name + "_beam.npz"))
    meta = ast.literal_eval(str(z["meta"]))
    dec = {k[4:]: (torch.from_numpy(z[k]).to(dtype) if z[k].dtype.kind == "f" else torch.from_numpy(z[k])) for k in z.files if k.startswith("dec.")}
    beams = {w: [[int(x) for x in row if x >= 0] for row in z[f"beam{w}"]] for w in (3, 5)}
    return {"meta": meta, "feats": torch.from_numpy(z["feats"]).to(dtype), "dec": dec, "beams": beams}


def philox_scales(seed, offset, site, shape, p, dtype=torch.float64):
    from tests.philox_ref import dropout_scales
    n = 1
    for d in shape:
        n *= d
    return torch.from_numpy(dropout_scales(seed, offset, site, n, p)).to(dtype).view(*shape)
