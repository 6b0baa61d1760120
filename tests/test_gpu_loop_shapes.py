"""The weight-resident loop kernels of the bf16 build against the fp64 oracle at the edges of the shapes their planners accept.

  rp::local_fwd_kernel<KS, SM> / rp::local_bwd_kernel<SM>   (csrc/seq_recon_persist.cuh): the local reconstructor's forward loop and BPTT,
                                                               and the global reconstructor's through `global_mode`
  dcl::decoder_fwd_cluster_kernel<NQ, SM>                    (csrc/seq_decoder_cluster.cuh): the decoder's forward loop, pf_bwd_kernel behind it

Every case runs through the public modules and asserts which loop ran, from the launch records of recnet_profile_enable: a KC_LOOP record
(class 9) has K = 0 for the persistent forward (M = steps, N = CTAs), K = 1 for the persistent BPTT, K = 2 for the decoder's cluster loop
(M = steps, N = 16 x clusters).  A shape that silently drops to the kernel-per-phase path fails here.

The reconstructor cases feed random decoder states as a leaf tensor and compare the loss, every parameter gradient and d hiddens, the
gradient that runs back through the loop's attention; lambda_reg = 0, so loss and gradients belong to the loop alone.  The decoder cases
compare the loss, the hiddens and every gradient.  Each tensor must pass the bf16 tolerance relative to its max (2e-2), and each tensor
with a batch axis must pass it for every sample on its own: max|a_b - r_b| / max|r_b|.  One wrong sample out of 128 moves the summed
weight gradients by under 1 %, which the whole-tensor measure alone would let through (tests/test_loop_shapes_host.py shows the margin).

The case tables are imported by tests/test_gemm_planner.py, which pins the planners' decisions for them on the CPU; nothing here touches
a device at import time.
"""
import ctypes as C
import dataclasses
import functools
from typing import Optional, Tuple

import pytest
import torch

import recnet_b200  # noqa: F401
from recnet_b200 import _lib as L
from recnet_b200 import functional as Fn
from recnet_b200 import train as T
from oracle import recnet_oracle as O
from tests import attn_softmax_oracle as S
from tests.golden_util import philox_scales
from tests.philox_ref import SITE_EMB, SITE_GLOBAL_MP, SITE_LOCAL_X, SITE_LOGITS
from tests.test_gpu_attn_softmax import build_sm
from tests.test_gpu_parity import TOL, build, configure, dev

pytestmark = pytest.mark.gpu
BF16_TOL = TOL["bf16"]
KC_LOOP = 9                 # csrc/common.cuh kernel class of the loop kernels' launch records
MAX_RECORDS = 8192
A = 128                     # attention size both loop kernels are written for
CAP = 30                    # caption_max_len (the global reconstructor scales its mean pool by it)
GLOBAL_FRAMES = 28


@dataclasses.dataclass(frozen=True)
class Rec:
    kind: str                               # "local" or "global"
    R: int                                  # reconstructor hidden size = feature size
    H: int                                  # decoder hidden size
    B: int
    S: int                                  # loop steps: frames (local) or decoder steps (global, = L)
    L: int                                  # decoder steps (attention keys of the local reconstructor)
    fwd: Optional[Tuple[int, int]]          # persistent forward: (K-splits, CTAs); None = kernel-per-phase
    bwd: Optional[Tuple[int, int]]          # persistent BPTT: (gate-row splits, CTAs); None = kernel-per-phase


# B200 (148 SMs).  KS / NS / CTAs as recnet_plan_persistent_loops and recnet_plan_global_loops report them (tests/test_gemm_planner.py).
REC_CASES = {
    "R1": Rec("local", 1536, 512, 3, 28, 31, (3, 144), (9, 144)),       # one sample per K-split
    "R2": Rec("local", 1536, 512, 17, 1, 1, (3, 144), (9, 144)),        # one step, one key; NB padding
    "R3": Rec("local", 1536, 512, 113, 28, 31, (3, 144), (9, 144)),     # NB = 128 on a 120-row stage, 2-stage ring
    "R4": Rec("local", 1536, 512, 128, 40, 32, (3, 144), (9, 144)),     # largest batch, all 32 attention lanes
    "R5": Rec("local", 1024, 512, 96, 20, 32, (3, 96), (8, 96)),        # B = UG x KS, NS = 8
    "R6": Rec("local", 768, 256, 48, 28, 17, (2, 48), (12, 96)),        # KS = 2, NS = 12, half the attention columns idle
    "R7": Rec("local", 640, 128, 40, 12, 9, (2, 40), (10, 60)),         # UG = 20, NS = 10
    "R8": Rec("local", 256, 256, 8, 28, 31, (1, 8), (12, 48)),          # KS = 1, 8 CTAs
    "R9": Rec("local", 512, 128, 1, 5, 3, (1, 16), None),               # KS = 1, B = 1; persistent forward feeds kernel-per-phase BPTT
    "R10": Rec("local", 1536, 256, 100, 28, 31, (3, 144), None),        # the same mix at the bench width
    "R11": Rec("local", 512, 512, 64, 28, 31, None, (12, 96)),          # kernel-per-phase forward feeds persistent BPTT
    "G1": Rec("global", 1536, 512, 128, 31, 31, (3, 144), (12, 144)),   # global mode, largest batch
    "G2": Rec("global", 1024, 256, 96, 9, 9, (2, 64), (12, 96)),        # B > UG x KS (global mode only)
    "G3": Rec("global", 512, 128, 48, 1, 1, (1, 16), (12, 48)),         # KS = 1, one step
}


@dataclasses.dataclass(frozen=True)
class Dec:
    B: int
    Tn: int
    clusters: Optional[int]                 # 16-CTA clusters of the cluster loop; None = kernel-per-phase loop


# The cluster kernel's shape: H = 512, A = 128; small E, EMB and V keep the oracle cheap.  Samples per cluster MS = ceil(B / 7): 7 clusters
# are co-resident on a B200 (cudaOccupancyMaxActiveClusters), so B > 112 drops to the per-step loop.
DEC_E, DEC_H, DEC_EMB, DEC_V, DEC_CAP = 256, 512, 72, 301, 15
DEC_CASES = {
    "D1": Dec(1, 28, 1),          # MS = 1, one cluster
    "D2": Dec(8, 16, 4),          # MS = 2; no CTA has a second frame
    "D3": Dec(15, 17, 5),         # MS = 3; one CTA with two frames
    "D4": Dec(97, 28, 7),         # MS = 14, last cluster 13
    "D5": Dec(106, 29, 7),        # MS = 16, last cluster 10, NQ = 32
    "D6": Dec(112, 32, 7),        # MS = 16 everywhere, two frames in every CTA
    "D7": Dec(113, 28, None),     # more than 7 x 16 samples
    "D8": Dec(20, 33, None),      # Tn > 32
}

SOFTMAX_CASES = [("R2", {}), ("R4", {}), ("R6", {}), ("D1", {"Tn": 1}), ("D5", {}), ("D6", {})]
TRAIN_CASES = ["R3", "R6", "R9", "G2", "D2", "D5"]


def case(cid, **overrides):
    c = REC_CASES.get(cid) or DEC_CASES[cid]
    return dataclasses.replace(c, **overrides)


def seed_of(cid):
    return sum(ord(ch) * 31 ** i for i, ch in enumerate(cid)) % 10007


# ---- inputs and fp64 oracle (shared with tests/test_loop_shapes_host.py) ------------------------------------------------------------
def rec_inputs(c, seed):
    """Decoder states (L, 1, B, H) in (-1, 1) as an LSTM leaves them, features, reconstructor parameters (fp32)."""
    g = torch.Generator().manual_seed(seed)
    hid = torch.rand(c.L, 1, c.B, c.H, generator=g) * 2 - 1
    if c.kind == "global" and c.L < CAP:
        # the global reconstructor scales its mean pool by caption_max_len / L (global_reconstructor.py:37): 30x at L = 1.  Unit-scale
        # states would then put its gate pre-activations at ~5 rms, where the gate derivatives are as exact as the pre-activation's
        # bf16 operand rounding, ~2 % (rounding only the operands of the fp64 oracle already moves d W_ih by 2.2e-2).  Scaled by
        # L / caption_max_len the pooled input keeps unit scale and the check measures the loops, not the saturated cells.
        hid = hid * (c.L / CAP)
    feats = torch.randn(c.B, c.S if c.kind == "local" else GLOBAL_FRAMES, c.R, generator=g)
    Q = O.init_reconstructor_params(c.kind, c.H, c.R, A, seed=seed + 1)
    return hid, feats, Q


def rec_drop(c, seed):
    """Philox scales of the reconstructor's dropout site, as the module draws them on its first training forward after seed_dropout(seed)."""
    p = T.C.reconstructor_decoder_dropout
    if c.kind == "local":
        return philox_scales(seed, 1, SITE_LOCAL_X, (c.S, c.B, c.H), p)
    return philox_scales(seed, 1, SITE_GLOBAL_MP, (c.L, c.B, c.H), p)


def rec_oracle(c, hid, feats, Q, softmax=False, drop=None):
    """fp64: loss, every parameter gradient and d hiddens (L, 1, B, H); lambda_reg = 0."""
    Qr = {k: v.to(torch.float64, copy=True).requires_grad_(True) for k, v in Q.items()}
    h = hid.to(torch.float64, copy=True).requires_grad_(True)
    if c.kind == "local":
        loss, _ = S.forward_local_reconstructor(Qr, h, feats.double(), lambda_reg=0.0, drop_x=drop, attn_softmax=softmax)
    else:
        loss, _ = O.forward_global_reconstructor(Qr, h, feats.double(), caption_max_len=CAP, lambda_reg=0.0, drop_mp=drop)
    loss.backward()
    return dict(loss=loss.detach(), d_hiddens=h.grad, **{k: v.grad for k, v in Qr.items()})


def dec_inputs(c, seed):
    feats, targets, masks = O.synthetic_batch(c.B, c.Tn, DEC_E, DEC_V, DEC_CAP, seed=seed)
    P = O.init_decoder_params(DEC_V, DEC_EMB, DEC_E, DEC_H, A, seed=seed + 1)
    # A unit-scale embedding drowns the attention context, the part the loop kernels compute, in the gate input: losing one frame of 29
    # then moves the hiddens by ~2 %, inside the bf16 tolerance.  At a tenth of it the context carries the gates and the same fault moves
    # them by > 10 % (tests/test_loop_shapes_host.py).
    P["embedding.weight"] = P["embedding.weight"] * 0.1
    return feats, targets, masks, P


def dec_drops(masks, seed):
    Lsteps, B = T._num_steps(masks, DEC_CAP), masks.shape[1]
    return dict(emb=philox_scales(seed, 1, SITE_EMB, (Lsteps, B, DEC_EMB), T.C.embedding_dropout),
                logits=philox_scales(seed, 1, SITE_LOGITS, (Lsteps, B, DEC_V), T.C.decoder_out_dropout))


def dec_oracle(feats, targets, masks, P, softmax=False, drops=None):
    """fp64: loss, hiddens (L, 1, B, H) and every parameter gradient; lambda_reg = 0."""
    Pr = {k: v.to(torch.float64, copy=True).requires_grad_(True) for k, v in P.items()}
    d = drops or {}
    loss, hid, _, _ = S.forward_decoder(Pr, feats.double(), targets, masks, caption_max_len=DEC_CAP, lambda_reg=0.0,
                                        drop_emb=d.get("emb"), drop_logits=d.get("logits"), attn_softmax=softmax)
    loss.backward()
    return dict(loss=loss.detach(), hiddens=hid.detach(), **{k: v.grad for k, v in Pr.items()})


# ---- the checks -------------------------------------------------------------------------------------------------------------------------
BATCH_AXIS = {"hiddens": 2, "d_hiddens": 2}        # (L, 1, B, H)


def rel(a, r):
    a, r = a.detach().double().cpu(), r.detach().double().cpu()
    assert a.shape == r.shape, (a.shape, r.shape)
    return float((a - r).abs().max() / (r.abs().max() + 1e-30))


def rel_per_sample(a, r, axis):
    """max over samples b of max|a_b - r_b| / max|r_b|."""
    a, r = a.detach().double().cpu(), r.detach().double().cpu()
    assert a.shape == r.shape, (a.shape, r.shape)
    a, r = a.movedim(axis, 0).reshape(a.shape[axis], -1), r.movedim(axis, 0).reshape(r.shape[axis], -1)
    return float(((a - r).abs().amax(1) / (r.abs().amax(1) + 1e-30)).max())


def errors(got, ref):
    """name -> error under every metric that applies to it: the whole-tensor one, and per sample where the tensor has a batch axis."""
    out = {}
    for k, r in ref.items():
        out[k] = rel(got[k], r)
        if k in BATCH_AXIS:
            out[k + "/sample"] = rel_per_sample(got[k], r, BATCH_AXIS[k])
    return out


# ---- device side ------------------------------------------------------------------------------------------------------------------------
def _profile_start():
    L.check(L.lib().recnet_profile_enable(1, MAX_RECORDS), "recnet_profile_enable")


def _loop_records():
    """(M, N, K) of every KC_LOOP launch since _profile_start(), sorted."""
    buf = (C.c_float * (5 * MAX_RECORDS))()
    n = L.lib().recnet_profile_collect(C.cast(buf, C.c_void_p), MAX_RECORDS)
    L.lib().recnet_profile_enable(0, 0)
    assert 0 <= n < MAX_RECORDS, n             # every launch was recorded
    return sorted((int(buf[5 * i + 1]), int(buf[5 * i + 2]), int(buf[5 * i + 3])) for i in range(n) if int(buf[5 * i]) == KC_LOOP)


def expected_records(c, steps=None):
    if isinstance(c, Dec):
        return [] if c.clusters is None else [(steps, 16 * c.clusters, 2)]
    out = []
    if c.fwd:
        out.append((c.S, c.fwd[1], 0))
    if c.bwd:
        out.append((c.S, c.bwd[1], 1))
    return sorted(out)


def _run_rec(c, hid, feats, Q, softmax, train, seed):
    m = dict(B=c.B, T=feats.shape[1], E=c.R, H=c.H, A=A, EMB=64, cap_len=CAP, dec_layers=1, rec_layers=1, dec_model="LSTM",
             rec_model="LSTM")
    configure(m, "bf16", c.kind)
    T.C.reconstructor_attn_softmax = softmax
    try:
        rec = T.build_reconstructor()
    finally:
        T.C.reconstructor_attn_softmax = False
    model = rec["model"]
    model.load_state_dict({k: v.float() for k, v in Q.items()})
    rec["lambda_reg"] = torch.zeros((), device=dev())
    model.train(train)
    if train:
        model.seed_dropout(seed)
    h = hid.to(dev()).requires_grad_(True)
    _profile_start()
    loss = T.forward_reconstructor_for(c.kind)(h, feats.to(dev()), rec)
    loss.backward()
    Fn.check_loop_status()
    records = _loop_records()
    return dict(loss=loss.detach(), d_hiddens=h.grad, **{k: p.grad for k, p in model.named_parameters()}), records


def _run_dec(c, feats, targets, masks, P, softmax, train, seed):
    m = dict(B=c.B, T=c.Tn, E=DEC_E, H=DEC_H, A=A, EMB=DEC_EMB, V=DEC_V, cap_len=DEC_CAP, dec_layers=1, rec_layers=1, dec_model="LSTM",
             rec_model="LSTM")
    dec, _ = build_sm(m, "bf16", P, None) if softmax else build(m, "bf16", "none", P, {})
    dec["lambda_reg"] = torch.zeros((), device=dev())
    model = dec["model"]
    model.train(train)
    if train:
        model.seed_dropout(seed)
    _profile_start()
    dloss, hiddens, _ = T.forward_decoder(dec, feats.to(dev()), targets.to(dev()), masks.to(dev()), 1.0)
    dloss.backward()
    Fn.check_loop_status()
    records = _loop_records()
    return dict(loss=dloss.detach(), hiddens=hiddens.detach(), **{k: p.grad for k, p in model.named_parameters()}), records


@functools.lru_cache(maxsize=None)
def _reference(cid, softmax, train, overrides=()):
    """Inputs and fp64 oracle results of one case, computed once per module."""
    c, seed = case(cid, **dict(overrides)), seed_of(cid)
    if isinstance(c, Rec):
        hid, feats, Q = rec_inputs(c, seed)
        return c, seed, (hid, feats, Q), rec_oracle(c, hid, feats, Q, softmax, rec_drop(c, seed) if train else None)
    feats, targets, masks, P = dec_inputs(c, seed)
    return c, seed, (feats, targets, masks, P), dec_oracle(feats, targets, masks, P, softmax, dec_drops(masks, seed) if train else None)


def check_case(cid, softmax=False, train=False, **overrides):
    c, seed, inputs, ref = _reference(cid, softmax, train, tuple(sorted(overrides.items())))
    if isinstance(c, Rec):
        got, records = _run_rec(c, *inputs, softmax, train, seed)
        want = expected_records(c)
    else:
        got, records = _run_dec(c, *inputs, softmax, train, seed)
        want = expected_records(c, ref["hiddens"].shape[0])
    err = errors(got, ref)
    name, worst = max(err.items(), key=lambda kv: kv[1])
    mode = ("softmax " if softmax else "") + ("train" if train else "eval")
    print(f"{cid} {mode}: worst error {worst:.2e} ({name}); loop records {records}")
    assert records == want, (cid, records, want)
    bad = {k: v for k, v in err.items() if not v < BF16_TOL}
    assert not bad, (cid, bad)


# ---- tests ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cid", sorted(REC_CASES))
def test_reconstructor_loops_match_the_oracle(cid):
    check_case(cid)


@pytest.mark.parametrize("cid", sorted(DEC_CASES))
def test_decoder_loop_matches_the_oracle(cid):
    check_case(cid)


@pytest.mark.parametrize("cid,overrides", SOFTMAX_CASES, ids=[c + "".join(f"-{k}{v}" for k, v in o.items()) for c, o in SOFTMAX_CASES])
def test_softmax_attention_loops_match_the_oracle(cid, overrides):
    check_case(cid, softmax=True, **overrides)


@pytest.mark.parametrize("cid", TRAIN_CASES)
def test_train_mode_loops_match_the_oracle_with_the_same_masks(cid):
    check_case(cid, train=True)
