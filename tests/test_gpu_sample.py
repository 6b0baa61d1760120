"""GPU checks of the device sampler (Decoder.sample / recnet_decoder_sample) and of self-critical training
(train.forward_decoder_self_critical) against the fp64 sampling oracle of tests/sample_oracle.py:
  * fp32 ids, lengths and n bit-exact, logp within 1e-4, eval and train mode (dropout p = 0.5 at every site), LSTM with 1, 2 and 4
    layers, single-layer GRU, the paper's softmax attention, 1 and 5 samples per video;
  * the teacher-forced replay's log-likelihood of every sampled token equals the sampler's logp (fp32, train mode, tau = 1);
  * the step-0 token counts of 4096 identical rows against softmax(z / tau) (chi-square), both precisions;
  * the noise is a function of (seed, offset) only, and torch's generator supplies it when no seed is given;
  * the self-critical loss and every decoder gradient against the oracle (fp32 1e-3, bf16 2e-2), and at zero advantage;
  * Decoder.sample never steps through Decoder.forward; batch 1024 at MSVD shape.
A mismatching id prints the oracle's smallest top-2 gap of the noisy values, so that a near tie can be told apart from a bug."""
import pytest
import torch
from scipy import stats

from recnet_b200 import functional as Fn
from recnet_b200 import models as M
from recnet_b200 import train as T
from oracle import recnet_oracle as O
from tests import sample_oracle as SM
from tests.golden_util import philox_scales
from tests.philox_ref import SITE_LOGITS
from tests.test_gpu_attn_softmax import build_sm
from tests.test_gpu_parity import FULL, TOL, _full_inputs, dev, rel
from tests.test_gpu_stacked import MID

pytestmark = pytest.mark.gpu

D = torch.float64
STEPS = MID["cap_len"] + 1
P_DROP = 0.5
DSEED, NSEED = 0xD00D, 0x5A3D1E
CASES = [("LSTM", 1, False), ("LSTM", 2, False), ("LSTM", 4, False), ("GRU", 1, False), ("LSTM", 1, True)]


def _params(model_name, NL, eos_boost=5.0):
    """fp32-representable fp64 weights; logits spread (x 4) and <EOS> lifted (+5) so that rows finish at different steps."""
    P = O.init_decoder_params(MID["V"], MID["EMB"], MID["E"], MID["H"], MID["A"], n_layers=NL, model_name=model_name, seed=4, dtype=D)
    P["out.weight"] = P["out.weight"] * 4
    P["out.bias"] = P["out.bias"].clone()
    P["out.bias"][2] += eos_boost
    return {k: v.float().double() for k, v in P.items()}


def _model(model_name, NL, softmax, prec, train, P):
    dec, _ = build_sm(dict(MID, dec_layers=NL, dec_model=model_name), prec, P, None, softmax=softmax)
    model = dec["model"]
    model.embedding_dropout_p = model.out_dropout_p = model.dropout_p = P_DROP
    if train:
        model.train()
        model.seed_dropout(DSEED)          # the sampler's _next_rng() makes it (DSEED, 1)
    return dec, model


def _feats(seed=7):
    feats, _, _ = O.synthetic_batch(MID["B"], MID["T"], MID["E"], MID["V"], MID["cap_len"], seed=seed, dtype=D)
    return feats


def _drops(train, N, NL, L=STEPS):
    if not train:
        return None
    return SM.Drops(DSEED, 1, L=L, B=N, EMB=MID["EMB"], V=MID["V"], H=MID["H"], n_layers=NL, p_emb=P_DROP, p_out=P_DROP, p_layer=P_DROP)


# ---- 1. fp32 against the oracle -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 5])
@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("model_name,NL,softmax", CASES)
def test_fp32_sample_matches_the_fp64_oracle(model_name, NL, softmax, train, K):
    P = _params(model_name, NL)
    _, model = _model(model_name, NL, softmax, "fp32", train, P)
    feats = _feats()
    ids, logp, lengths, n = model.sample(feats.float().to(dev()), K, max_steps=STEPS, seed=NSEED)
    tiled = feats.repeat(K, 1, 1)
    ref = SM.sample(P, tiled, max_steps=STEPS, noise=(NSEED, 0), model_name=model_name, n_layers=NL,
                    drops=_drops(train, tiled.shape[0], NL), attn_softmax=softmax)
    ids, logp, lengths = ids.cpu(), logp.cpu(), lengths.cpu()
    bad = (ids != ref["ids"]).nonzero()
    first = None if bad.numel() == 0 else tuple(int(x) for x in bad[0])
    err = float((logp.double() - ref["logp"]).abs().max())
    print(f"[sample] {model_name} NL={NL} softmax={softmax} train={train} K={K}: n {int(n)} / oracle {ref['n']}, rows finished "
          f"{int((ref['lengths'] < STEPS).sum())} / {tiled.shape[0]}, first id mismatch {first}, smallest oracle top-2 noisy gap "
          f"{float(ref['gap'].min()):.3e}, max logp err {err:.2e}")
    assert int((ref["lengths"] < STEPS).sum()) > 0
    assert torch.equal(ids, ref["ids"])
    assert torch.equal(lengths, ref["lengths"]) and int(n) == ref["n"]
    assert err < 1e-4


# ---- 2. the replay differentiates the sampler's logits --------------------------------------------------------------------------
@pytest.mark.parametrize("model_name,NL", [("LSTM", 1), ("LSTM", 2), ("GRU", 1)])
def test_fp32_replay_log_likelihood_equals_the_sampler_logp(model_name, NL):
    P = _params(model_name, NL)
    _, model = _model(model_name, NL, False, "fp32", True, P)
    K = 5
    f = _feats().float().to(dev()).repeat(K, 1, 1).contiguous()
    ids, logp, lengths, n = model._sample(f, STEPS, 1.0, 2, torch.tensor([NSEED, 3], device=dev()))
    rng = model._rng.clone()
    n = int(n)
    N = f.shape[0]
    tokens_in = torch.cat((torch.ones(1, N, dtype=torch.long, device=dev()), ids[: n - 1]))
    z, _ = Fn.decoder_teacher_forced_logits(model._meta(), f, tokens_in, rng, model._params())
    mask = philox_scales(DSEED, 1, SITE_LOGITS, (n, N, MID["V"]), P_DROP).to(dev())
    lp = torch.log_softmax(z.double() * mask, dim=-1).gather(2, ids[:n].unsqueeze(2)).squeeze(2)
    valid = torch.arange(n, device=dev()).unsqueeze(1) < lengths.long().unsqueeze(0)
    err = float(((lp - logp[:n].double()) * valid).abs().max())
    print(f"[sample] replay {model_name} NL={NL}: {n} steps, {int(valid.sum())} sampled tokens, max |replay logp - sampler logp| {err:.2e}")
    assert err < 1e-5


# ---- 3. distribution ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("tau", [0.5, 1.0, 2.0])
def test_step0_counts_follow_the_tempered_softmax(prec, tau):
    P = _params("LSTM", 1, eos_boost=0.0)                    # no dominant token: the counts spread over many bins at every tau
    _, model = _model("LSTM", 1, False, prec, False, P)
    feats = _feats()[:1]
    R = 4096
    ids, _, _, _ = model.sample(feats.float().to(dev()), R, max_steps=1, temperature=tau, seed=2024)
    z, _ = O.decoder_step(P, torch.ones(1, 1, dtype=torch.long), O.zero_hidden("LSTM", 1, 1, MID["H"], feats), feats)
    p = torch.softmax(z[0] / tau, dim=0)
    obs = torch.bincount(ids[0].cpu(), minlength=MID["V"]).double()
    exp = p * R
    big = exp >= 5                                            # bins with an expected count below 5 are pooled into one
    o = torch.cat((obs[big], obs[~big].sum().view(1)))
    e = torch.cat((exp[big], exp[~big].sum().view(1)))
    chi2, pval = stats.chisquare(o.numpy(), e.numpy())
    print(f"[sample] {prec} tau={tau}: step-0 chi-square {chi2:.1f} over {o.numel()} bins, p-value {pval:.3f}")
    assert pval > 1e-3


# ---- 4. determinism ------------------------------------------------------------------------------------------------------------
def test_noise_depends_on_seed_and_offset_only():
    P = _params("LSTM", 2)
    _, model = _model("LSTM", 2, False, "fp32", False, P)
    f = _feats().float().to(dev()).repeat(5, 1, 1).contiguous()
    run = lambda s, o: model._sample(f, STEPS, 1.0, 2, torch.tensor([s, o], device=dev()))[0]
    a = run(NSEED, 0)
    assert torch.equal(a, run(NSEED, 0))
    assert not torch.equal(a, run(NSEED + 1, 0)) and not torch.equal(a, run(NSEED, 1))
    g = f[: MID["B"]]
    torch.manual_seed(0)
    x1, x2 = model.sample(g, 5, max_steps=STEPS)[0], model.sample(g, 5, max_steps=STEPS)[0]
    torch.manual_seed(0)
    y1, y2 = model.sample(g, 5, max_steps=STEPS)[0], model.sample(g, 5, max_steps=STEPS)[0]
    assert torch.equal(x1, y1) and torch.equal(x2, y2) and not torch.equal(x1, x2)
    assert torch.equal(model.sample(g, 5, max_steps=STEPS, seed=NSEED)[0], a)


# ---- 5. self-critical training -------------------------------------------------------------------------------------------------
def _reward(sample_ids, greedy_ids):
    """Synthetic reward: how many ids of a caption fall into [3, 300); the baseline gets one extra, so that advantages take both signs."""
    r = lambda ids: ((ids >= 3) & (ids < 300)).sum(dim=0).float()
    return r(sample_ids), r(greedy_ids) + 1.0


def _oracle_scst(P, feats, info, K, NL, lam, zero=False):
    ids = info["ids"].cpu()
    n, N = ids.shape
    tokens_in = torch.cat((torch.ones(1, N, dtype=torch.long), ids[:-1]))
    mask = (torch.arange(n).unsqueeze(1) < info["lengths"].cpu().long().unsqueeze(0)).double()
    w = mask * info["advantage"].cpu().double() / N
    assert zero == bool((w == 0).all())
    Pr = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    loss = SM.replay_loss(Pr, feats.repeat(K, 1, 1), tokens_in, ids, w, n_layers=NL, drops=_drops(True, N, NL, n), lambda_reg=lam)
    loss.backward()
    return loss, {k: v.grad for k, v in Pr.items()}


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("NL", [1, 2])
def test_self_critical_loss_and_gradients_against_the_oracle(prec, NL):
    P = _params("LSTM", NL)
    dec, model = _model("LSTM", NL, False, prec, True, P)
    feats = _feats()
    K = 5
    torch.manual_seed(11)
    loss, hiddens, info = T.forward_decoder_self_critical(dec, feats.float().to(dev()), _reward, n_samples=K, max_steps=STEPS)
    loss.backward()
    lam = float(dec["lambda_reg"])
    ref_loss, ref_grads = _oracle_scst(P, feats, info, K, NL, lam)
    errs = {"loss": rel(loss, ref_loss)}
    for k, p in model.named_parameters():
        errs[k] = rel(p.grad, ref_grads[k])
    worst = max(errs, key=errs.get)
    adv = info["advantage"]
    print(f"[sample] SCST {prec} NL={NL}: {info['ids'].shape[0]} steps, advantage in [{float(adv.min()):.1f}, {float(adv.max()):.1f}], "
          f"worst rel err {errs[worst]:.3e} ({worst})")
    assert float(adv.min()) < 0 < float(adv.max()) and hiddens.shape[2] == K * MID["B"]
    assert errs[worst] < TOL[prec], (worst, errs[worst])


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_self_critical_with_zero_advantage_leaves_only_the_regulariser(prec):
    P = _params("LSTM", 1)
    dec, model = _model("LSTM", 1, False, prec, True, P)
    feats = _feats()
    zero = lambda s, g: (torch.zeros(s.shape[1], device=s.device), torch.zeros(g.shape[1], device=g.device))
    loss, _, info = T.forward_decoder_self_critical(dec, feats.float().to(dev()), zero, n_samples=3, max_steps=STEPS)
    loss.backward()
    lam = float(dec["lambda_reg"])
    ref_loss, ref_grads = _oracle_scst(P, feats, info, 3, 1, lam, zero=True)
    worst = max([rel(loss, ref_loss)] + [rel(p.grad, ref_grads[k]) for k, p in model.named_parameters()])
    print(f"[sample] SCST zero advantage {prec}: worst rel err {worst:.3e}")
    assert worst < TOL[prec]


# ---- 6. no step-wise fallback; full size ----------------------------------------------------------------------------------------
def test_sample_never_calls_decoder_forward(monkeypatch):
    P = _params("LSTM", 2)
    _, model = _model("LSTM", 2, False, "bf16", False, P)

    def no_forward(*a, **kw):
        raise AssertionError("Decoder.forward called")

    monkeypatch.setattr(M.Decoder, "forward", no_forward)
    f = _feats().float().to(dev())
    for train in (False, True):
        model.train(train)
        ids, _, _, n = model.sample(f, 2, max_steps=STEPS, seed=1)
        assert ids.shape == (STEPS, 2 * MID["B"]) and 1 <= int(n) <= STEPS


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_full_size_batch1024(prec):
    B = 1024
    feats, _, _ = _full_inputs(B, seed=77)
    P = O.init_decoder_params(FULL["V"], FULL["EMB"], FULL["E"], FULL["H"], FULL["A"], seed=0)
    dec, _ = build_sm(dict(FULL, B=B), prec, P, None, softmax=False)
    model = dec["model"]
    model.train()
    ids, logp, lengths, n = model.sample(feats.to(dev()), 1, max_steps=31, seed=3)
    n = int(n)
    steps = torch.arange(31, device=dev()).unsqueeze(1)
    after = steps >= lengths.long().unsqueeze(0)
    print(f"[sample] B=1024 {prec}: n {n}, lengths {int(lengths.min())}..{int(lengths.max())}")
    assert ((ids >= 0) & (ids < FULL["V"])).all()
    assert (lengths >= 1).all() and (lengths <= n).all()
    assert (ids[after] == 0).all() and (logp[after] == 0).all() and (logp <= 0).all()
