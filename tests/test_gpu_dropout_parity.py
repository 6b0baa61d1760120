"""Parity of what bench.py actually times: TRAIN mode, dropout on at all three sites (embedding, logits-before-CE, reconstructor
input), plus the reference-pinned beam search and two regressions from the round-1 review.

The kernels draw their masks from an in-kernel Philox generator keyed by the module's (seed, offset).  tests/philox_ref.py restates
that generator in numpy; `recnet_debug_dropout_mask` exports what the device function returns, so the restatement is checked
bit for bit, and the SAME masks are then given to (a) the real reference -- fixtures of tests/golden/make_golden_train.py, where they
replace the reference's nn.Dropout modules -- and (b) the CPU oracle at the full MSVD size.  A forward/backward mask mismatch in any
kernel (a `drop_base` off by one between a forward and its backward, say) shows up as a gradient error here.
"""
import copy

import numpy as np
import pytest
import torch

import recnet_b200
from recnet_b200 import _lib as L
from recnet_b200 import eval as E
from recnet_b200 import functional as Fn
from recnet_b200 import train as T
from recnet_b200.optim import ClipAdam
from oracle import recnet_oracle as O
from tests.golden_util import load_golden, load_golden_beam, load_golden_train, philox_scales
from tests.philox_ref import SITE_EMB, SITE_GLOBAL_MP, SITE_LAYER0, SITE_LOCAL_X, SITE_LOGITS, dropout_scales
from tests.test_gpu_parity import FULL, TOL, _Vocab, _full_inputs, build, dev, rel

pytestmark = pytest.mark.gpu


# inter-layer dropout of a stacked decoder (sites 17..19): the (L, B, H) of the benchmarked 2-layer step and of the 3- and 4-layer
# cases of test_gpu_stacked.py
@pytest.mark.parametrize("site,n,p", [(SITE_EMB, 31 * 100 * 468, 0.5), (SITE_LOGITS, 7 * 4188 + 3, 0.5), (SITE_LOCAL_X, 28 * 100 * 512, 0.5),
                                      (SITE_GLOBAL_MP, 12345, 0.3), (SITE_LAYER0 + 1, 31 * 100 * 512, 0.5),
                                      (SITE_LAYER0 + 2, 13 * 13 * 256 + 1, 0.5), (SITE_LAYER0 + 3, 13 * 13 * 256, 0.3)])
def test_device_dropout_masks_equal_the_numpy_philox_restatement(site, n, p):
    seed, offset = 0xDEC0 + site, 3
    rng = torch.tensor([seed, offset], dtype=torch.int64, device=dev())
    out = torch.empty(n, dtype=torch.float32, device=dev())
    L.check(L.lib().recnet_debug_dropout_mask(rng.data_ptr(), site, n, p, out.data_ptr(), Fn._stream()), "recnet_debug_dropout_mask")
    ref = dropout_scales(seed, offset, site, n, p)
    assert np.array_equal(out.cpu().numpy(), ref)
    assert 0.4 < float((out == 0).float().mean()) / p < 1.6


def _train_step_grads(dec, rec, kind, feats, targets, seeds):
    dec["model"].train(); dec["model"].seed_dropout(seeds["dec"])
    if rec is not None:
        rec["model"].train(); rec["model"].seed_dropout(seeds[kind])
    dloss, hiddens, _ = T.forward_decoder(dec, feats, targets, targets > 0, 1.0)
    rloss = T.forward_reconstructor_for(kind)(hiddens, feats, rec) if rec is not None else None
    (dloss if rloss is None else dloss + rloss).backward()
    Fn.check_loop_status()
    return dloss, rloss, hiddens


# tiny_lstm_ragged (H = 12, E = 20) is fp32 only: the bf16 build needs 16-byte operand rows for TMA (H, E multiples of 8) and says so
# with RECNET_ERR_ALIGNMENT -- same split as GOLDEN in test_gpu_parity.py
@pytest.mark.parametrize("kind", ["none", "global", "local"])
@pytest.mark.parametrize("name,precision", [("small_lstm", "fp32"), ("small_lstm", "bf16"), ("tiny_lstm_ragged", "fp32")])
def test_train_mode_losses_and_grads_match_the_reference_with_the_same_masks(name, precision, kind):
    """Reference-generated fixture: train.forward_* of the real reference in train mode with these Philox masks injected."""
    g = load_golden_train(name)
    # bf16 on contractions of K <= 64 does not average its operand rounding out: same documented allowance as the other tiny fixtures
    tol = TOL[precision] if precision == "fp32" else 4e-2
    dec, rec = build(g["meta"], precision, kind, g["dec"], g[kind] if kind != "none" else {})
    feats, targets = g["feats"].float().to(dev()), g["targets"].to(dev())
    seeds = {"dec": g["seed_dec"], "local": g["seed_local"], "global": g["seed_global"]}
    dloss, rloss, hiddens = _train_step_grads(dec, rec, kind, feats, targets, seeds)
    assert abs(float(dloss) - g["dec_loss"]) / abs(g["dec_loss"]) < tol
    assert rel(hiddens, g["hiddens"]) < tol
    if kind != "none":
        assert abs(float(rloss) - g[f"{kind}_loss"]) / abs(g[f"{kind}_loss"]) < tol
    named = {"dec." + k: p for k, p in dec["model"].named_parameters()}
    if rec is not None:
        named.update({f"{kind}." + k: p for k, p in rec["model"].named_parameters()})
    for k, ref in g["grads"][kind].items():
        assert rel(named[k].grad, ref) < tol, k


@pytest.mark.parametrize("kind", ["local", "global"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_full_size_train_mode_parity_against_oracle_with_the_same_masks(precision, kind):
    """The benchmarked configuration (MSVD shape, batch 100, L = 31, dropout 0.5 at three sites): loss + every gradient, fp32 1e-3 / bf16 2e-2.
    With kind = local and bf16 this runs the weight-resident persistent loops (csrc/seq_recon_persist.cuh), forward and BPTT."""
    feats, targets, masks = _full_inputs()
    P = O.init_decoder_params(FULL["V"], FULL["EMB"], FULL["E"], FULL["H"], FULL["A"], seed=0)
    Q = O.init_reconstructor_params(kind, FULL["H"], FULL["E"], FULL["A"], seed=1)
    seeds = {"dec": 0xDEC0, "local": 0x10CA, "global": 0x610B}
    C = T.C
    B, Lmax, Tn, H = 100, 31, FULL["T"], FULL["H"]
    Pr = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    Qr = {k: v.clone().requires_grad_(True) for k, v in Q.items()}
    de = philox_scales(seeds["dec"], 1, SITE_EMB, (Lmax, B, FULL["EMB"]), C.embedding_dropout, torch.float32)
    dl_ = philox_scales(seeds["dec"], 1, SITE_LOGITS, (Lmax, B, FULL["V"]), C.decoder_out_dropout, torch.float32)
    dl, hid, _, _ = O.forward_decoder(Pr, feats, targets, masks, drop_emb=de, drop_logits=dl_)
    assert hid.shape[0] == Lmax
    if kind == "local":
        rl, _ = O.forward_local_reconstructor(Qr, hid, feats, drop_x=philox_scales(seeds["local"], 1, SITE_LOCAL_X, (Tn, B, H),
                                                                                 C.reconstructor_decoder_dropout, torch.float32))
    else:
        rl, _ = O.forward_global_reconstructor(Qr, hid, feats, drop_mp=philox_scales(seeds["global"], 1, SITE_GLOBAL_MP, (Lmax, B, H),
                                                                                   C.reconstructor_decoder_dropout, torch.float32))
    (dl + rl).backward()
    dec, rec = build(FULL, precision, kind, P, Q)
    assert dec["model"].embedding_dropout_p == C.embedding_dropout and dec["model"].out_dropout_p == C.decoder_out_dropout
    tol = TOL[precision]
    dloss, rloss, hiddens = _train_step_grads(dec, rec, kind, feats.to(dev()), targets.to(dev()), seeds)
    assert rel(dloss, dl.detach()) < tol and rel(rloss, rl.detach()) < tol and rel(hiddens, hid.detach()) < tol
    for k, p in dec["model"].named_parameters():
        assert rel(p.grad, Pr[k].grad) < tol, k
    for k, p in rec["model"].named_parameters():
        assert rel(p.grad, Qr[k].grad) < tol, k


@pytest.mark.parametrize("loop", ["device", "host"])
@pytest.mark.parametrize("name", ["tiny_lstm", "tiny_gru", "small_lstm"])
def test_beam_search_matches_the_references_own_beam_search(name, loop, monkeypatch):
    """Fixtures hold what the reference's eval.beam_search itself returned (make_golden_train.py); fp32 build, widths 3 and 5.
    loop=device: recnet_decoder_beam (the whole loop in one C call); loop=host: the per-step path used for stacked decoders."""
    monkeypatch.setenv("RECNET_BEAM_DEVICE", "1" if loop == "device" else "0")
    g = load_golden_beam(name)
    m = dict(g["meta"], rec_model="LSTM")
    P = {k: v.float() for k, v in g["dec"].items()}
    dec, _ = build(m, "fp32", "none", P, {})
    feats = g["feats"].float().to(dev())
    B, H = feats.shape[0], m["H"]
    T.C.batch_size = B
    for width in (3, 5):
        tok = torch.full((1, B), 1, dtype=torch.long, device=dev())
        z = torch.zeros(1, B, H, device=dev())
        hid = (z, z.clone()) if m["dec_model"] == "LSTM" else z
        got = E.beam_search(T.C, width, _Vocab(m["V"]), dec["model"], tok, hid, feats)
        assert got == g["beams"][width], (width, got, g["beams"][width])


@pytest.mark.parametrize("width", [1, 4, 8])
def test_device_beam_loop_agrees_with_the_per_step_loop_on_a_larger_batch(width, monkeypatch):
    """The fixture's weights (well-separated scores) on 48 perturbed copies of its features: the one-call device loop and the per-step
    loop must return the same sequences; width 1 must also equal greedy decoding up to the first <EOS>-free prefix."""
    g = load_golden_beam("small_lstm")
    m = dict(g["meta"], rec_model="LSTM")
    P = {k: v.float() for k, v in g["dec"].items()}
    dec, _ = build(m, "fp32", "none", P, {})
    f0 = g["feats"].float()
    gen = torch.Generator().manual_seed(11)
    reps = (48 + f0.shape[0] - 1) // f0.shape[0]
    feats = (f0.repeat(reps, 1, 1)[:48] * (1.0 + 0.2 * torch.randn(48, 1, 1, generator=gen))).to(dev())
    B, H = 48, m["H"]
    T.C.batch_size = B

    def decode():
        tok = torch.full((1, B), 1, dtype=torch.long, device=dev())
        z = torch.zeros(1, B, H, device=dev())
        return E.beam_search(T.C, width, _Vocab(m["V"]), dec["model"], tok, (z, z.clone()), feats)

    monkeypatch.setenv("RECNET_BEAM_DEVICE", "1")
    a = decode()
    monkeypatch.setenv("RECNET_BEAM_DEVICE", "0")
    b = decode()
    assert a == b
    assert len({tuple(x) for x in a}) > 1          # not degenerate


def test_beam_search_recomputes_the_feature_projection_for_every_batch():
    """Round-1 review: an implicit U.v cache keyed by (data_ptr, _version) survived across batches when the allocator reused the
    address.  Two batches decoded back to back through the same tensor address must each match a fresh decode."""
    g = load_golden_beam("small_lstm")
    m = dict(g["meta"], rec_model="LSTM")
    P = {k: v.float() for k, v in g["dec"].items()}
    dec, _ = build(m, "fp32", "none", P, {})
    B, H = g["feats"].shape[0], m["H"]
    T.C.batch_size = B
    f1 = g["feats"].float()
    f2 = torch.roll(f1, 1, dims=0) * 0.5 + 0.1

    def decode(feats_dev):
        tok = torch.full((1, B), 1, dtype=torch.long, device=dev())
        z = torch.zeros(1, B, H, device=dev())
        return E.beam_search(T.C, 3, _Vocab(m["V"]), dec["model"], tok, (z, z.clone()), feats_dev)

    buf = f1.to(dev())
    a1 = decode(buf)
    buf.copy_(f2)                              # same tensor object, same address, same _version semantics as a reused allocation
    a2 = decode(buf)
    fresh = decode(f2.to(dev()).clone())
    assert a1 == g["beams"][3]
    assert a2 == fresh
    assert dec["model"]._uv_scope is None      # nothing is remembered after the call


def test_clip_adam_state_loaded_into_torch_adam_advances_one_step_per_iteration():
    """Round-1 review: the per-parameter `step` entries aliased one device scalar; loaded into torch.optim.Adam they were advanced
    n_params times per iteration."""
    torch.manual_seed(3)
    ours = [torch.nn.Parameter(torch.randn(s, device=dev())) for s in ((5, 7), (11,), (3, 4))]
    opt = ClipAdam(ours, lr=1e-3, weight_decay=1e-5, amsgrad=True)
    for it in range(2):
        for p in ours:
            p.grad = torch.randn_like(p)
        opt.step()
    sd = copy.deepcopy(opt.state_dict())
    steps = [st["step"] for st in sd["state"].values()]
    assert len({s.data_ptr() for s in steps}) == len(steps)                 # independent storage
    fresh = [torch.nn.Parameter(p.detach().clone()) for p in ours]
    ref = torch.optim.Adam(fresh, lr=1e-3, weight_decay=1e-5, amsgrad=True)
    ref.load_state_dict(sd)
    for q in fresh:
        q.grad = torch.randn_like(q)
    ref.step()
    assert [float(st["step"]) for st in ref.state_dict()["state"].values()] == [3.0, 3.0, 3.0]


def test_checkpoint_restores_optimizer_state(tmp_path):
    g = load_golden("tiny_lstm")
    dec, rec = build(g["meta"], "fp32", "local", g["dec"], g["local"])
    feats, targets = g["feats"].float().to(dev()), g["targets"].to(dev())
    for _ in range(2):
        T.train_step(dec, rec, feats, targets, n_steps=g["hiddens"].shape[0])
    path = str(tmp_path / "2_checkpoint.tar")
    E.save_checkpoint(path, 2, dec, rec, loss=torch.tensor(0.0), config=None)
    dec2, rec2 = build(g["meta"], "fp32", "local", g["dec"], g["local"])
    assert E.load_checkpoint(path, dec2, rec2) == 2
    for a, b in ((dec, dec2), (rec, rec2)):
        sa, sb = a["optimizer"].state_dict()["state"], b["optimizer"].state_dict()["state"]
        assert sa.keys() == sb.keys() and len(sa) > 0
        for k in sa:
            assert float(sb[k]["step"]) == 2.0
            assert torch.equal(sa[k]["exp_avg"], sb[k]["exp_avg"]) and torch.equal(sa[k]["exp_avg_sq"], sb[k]["exp_avg_sq"])


def test_bf16_greedy_on_projected_feature_kernels_agrees_with_the_per_step_api():
    """recnet_decoder_greedy in the bf16 build runs on the projected-feature kernels (EW gather + VW, 4 launches per step).  Its ids are
    compared with an argmax-feedback loop over the per-step Decoder.forward API (operator kernels, the reference's own formulation) on
    weights with well-separated logits (the beam fixture): the two bf16 paths round differently, so a small disagreement is allowed; the
    fp32 build keeps the bit-exact general path (test_full_size_greedy_bit_exact_fp32_batch1024_shape)."""
    g = load_golden_beam("small_lstm")
    m = dict(g["meta"], rec_model="LSTM")
    P = {k: v.float() for k, v in g["dec"].items()}
    dec, _ = build(m, "bf16", "none", P, {})
    model = dec["model"]
    feats = g["feats"].float().to(dev())
    B, H, steps = feats.shape[0], m["H"], m["cap_len"] + 1
    ids, n = model.greedy(feats, steps)
    tok = torch.ones(1, B, dtype=torch.long, device=dev())
    hid = (torch.zeros(1, B, H, device=dev()), torch.zeros(1, B, H, device=dev()))
    ref = []
    with torch.no_grad(), model.cached_uv(feats):
        for _ in range(int(n)):
            logits, hid = model(tok, hid, feats)
            tok = logits.argmax(dim=1).view(1, -1)
            ref.append(tok[0].clone())
    ref = torch.stack(ref)
    agree = float((ids[: int(n)] == ref).float().mean())
    assert torch.equal(ids[0], ref[0]), (ids[0], ref[0])          # first step: same state, same token
    assert agree >= 0.9, agree
    # and against the fp64 oracle on the same weights
    oracle = O.greedy_search({k: v.double() for k, v in g["dec"].items()}, g["feats"], caption_max_len=m["cap_len"])
    k = min(int(n), oracle.shape[0])
    assert float((ids[:k].cpu() == oracle[:k]).float().mean()) >= 0.85
