"""GPU parity of the opt-in softmax attention (``attn_softmax=True``, the RecNet paper's attention) against the fp64 CPU oracle
(tests/attn_softmax_oracle.py): per-step kernel, fused sequence paths in eval and train mode (same Philox masks), the other cell /
depth variants, greedy and beam search, the CUDA-graph train step, and the opt-in kernel paths.  Tolerances as everywhere:
fp32 1e-3, bf16 2e-2 (relative to the tensor's max)."""
import os
import subprocess
import sys

import pytest
import torch

import recnet_b200
from recnet_b200 import _lib as L
from recnet_b200 import eval as E
from recnet_b200 import functional as Fn
from recnet_b200 import ops
from recnet_b200 import train as T
from oracle import recnet_oracle as O
from tests import attn_softmax_oracle as S
from tests.golden_util import load_golden, load_golden_beam, philox_scales
from tests.philox_ref import SITE_EMB, SITE_LOCAL_X, SITE_LOGITS
from tests.test_gpu_parity import FULL, TOL, _Vocab, _full_inputs, configure, dev, rel

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build_sm(m, precision, P, Q, softmax=True):
    """train.build_* with both attention switches set (kind = local or none)."""
    configure(m, precision, "local")
    T.C.decoder_attn_softmax = T.C.reconstructor_attn_softmax = softmax
    try:
        dec = T.build_decoder(m["V"])
        rec = T.build_reconstructor() if Q is not None else None
    finally:
        T.C.decoder_attn_softmax = T.C.reconstructor_attn_softmax = False
    assert dec["model"].attn_softmax is softmax
    dec["model"].load_state_dict({k: v.float() for k, v in P.items()})
    dec["model"].eval()
    if rec is not None:
        rec["model"].load_state_dict({k: v.float() for k, v in Q.items()})
        rec["model"].eval()
    return dec, rec


def oracle_grads(m, P, Q, feats, targets, masks, drops=None):
    Pr = {k: v.double().clone().requires_grad_(True) for k, v in P.items()}
    Qr = {k: v.double().clone().requires_grad_(True) for k, v in Q.items()}
    d = drops or {}
    dl, hid, _, aux = S.forward_decoder(Pr, feats.double(), targets, masks, model_name=m["dec_model"], n_layers=m["dec_layers"],
                                        caption_max_len=m["cap_len"], drop_emb=d.get("emb"), drop_logits=d.get("logits"), attn_softmax=True)
    rl, _ = S.forward_local_reconstructor(Qr, hid, feats.double(), model_name=m["rec_model"], drop_x=d.get("x"), attn_softmax=True)
    (dl + rl).backward()
    return dict(dl=dl.detach(), rl=rl.detach(), hid=hid.detach(), logits=aux["logits"].detach(),
                gP={k: v.grad for k, v in Pr.items()}, gQ={k: v.grad for k, v in Qr.items()})


def check_step(dec, rec, o, feats, targets, masks, tol):
    dloss, hiddens, _ = T.forward_decoder(dec, feats, targets, masks, 1.0)
    rloss = T.forward_local_reconstructor(hiddens, feats, rec)
    (dloss + rloss).backward()
    Fn.check_loop_status()
    assert rel(dloss, o["dl"]) < tol and rel(rloss, o["rl"]) < tol and rel(hiddens, o["hid"]) < tol
    for k, p in dec["model"].named_parameters():
        assert rel(p.grad, o["gP"][k]) < tol, k
    for k, p in rec["model"].named_parameters():
        assert rel(p.grad, o["gQ"][k]) < tol, k
    return float(dloss.detach()), float(rloss.detach())


# ---- per-step kernel ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec,tol", [(L.PREC_FP32, 1e-5), (L.PREC_BF16, 2e-2)])
@pytest.mark.parametrize("B,Tn,A,D", [(100, 28, 128, 1536), (100, 31, 128, 512), (7, 40, 16, 64), (3, 1, 8, 8)])
def test_softmax_attention_kernel_fwd_bwd(prec, tol, B, Tn, A, D):
    g = torch.Generator().manual_seed(B * Tn + 1)
    mk = lambda *s: torch.randn(*s, generator=g).to(dev())
    Wh, Uv, b, w, V = mk(B, A), mk(B, Tn, A), mk(A), mk(1, A) * 0.3, mk(B, Tn, D)
    ins = [t.clone().requires_grad_(True) for t in (Wh, Uv, b, w, V)]
    out = ops.additive_attention(*ins, prec, softmax=True)
    gout = mk(B, D)
    out.backward(gout)
    refs = [t.clone().double().requires_grad_(True) for t in (Wh, Uv, b, w, V)]
    rWh, rUv, rb, rw, rV = refs
    e = torch.tanh(rWh.unsqueeze(1) + rUv + rb) @ rw.t()
    ref = (torch.softmax(e, dim=1) * rV).sum(1)
    ref.backward(gout.double())
    assert rel(out, ref) < tol
    for a, r, name in zip(ins, refs, ("Wh", "Uv", "b", "w", "V")):
        assert rel(a.grad, r.grad) < tol, name


def test_softmax_weights_written_by_the_kernel_sum_to_one():
    B, Tn, A, D = 100, 28, 128, 1536
    g = torch.Generator().manual_seed(9)
    mk = lambda *s: torch.randn(*s, generator=g).to(dev())
    Wh, Uv, b, w, V = mk(B, A), mk(B, Tn, A), mk(A), mk(A) * 0.3, mk(B, Tn, D)
    for prec, dt in ((L.PREC_FP32, torch.float32), (L.PREC_BF16, torch.bfloat16)):
        alpha = torch.empty(B, Tn, device=dev())
        out = torch.empty(B, D, dtype=dt, device=dev())
        Vo = V.to(dt)
        L.check(L.lib().recnet_attn_fwd(prec, Wh.data_ptr(), 1, 0, Uv.data_ptr(), Tn * A, A, b.data_ptr(), w.data_ptr(), Vo.data_ptr(),
                                        Tn * D, D, B, Tn, A, D, 1, None, alpha.data_ptr(), out.data_ptr(), D, 0.0, None, 0, 0,
                                        Fn._stream()), "recnet_attn_fwd")
        torch.cuda.synchronize()
        assert float((alpha.double().sum(1) - 1).abs().max()) < 1e-6 and float(alpha.min()) >= 0


# ---- fused sequence paths, eval mode ---------------------------------------------------------------------------------
@pytest.mark.parametrize("size", ["small", "full"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_eval_mode_losses_hiddens_grads_match_oracle(size, precision):
    if size == "full":
        m = FULL
        feats, targets, masks = _full_inputs()
        P = O.init_decoder_params(m["V"], m["EMB"], m["E"], m["H"], m["A"], seed=0)
        Q = O.init_reconstructor_params("local", m["H"], m["E"], m["A"], seed=1)
    else:
        gl = load_golden("small_lstm")
        m = dict(gl["meta"], rec_model="LSTM")
        feats, targets = gl["feats"].float(), gl["targets"]
        masks = targets > 0
        P, Q = gl["dec"], gl["local"]
    o = oracle_grads(m, P, Q, feats, targets, masks)
    dec, rec = build_sm(m, precision, P, Q)
    assert dec["model"].uses_fused_sequence and rec["model"]._fused_ok(o["hid"])
    f, t, k = feats.to(dev()), targets.to(dev()), masks.to(dev())
    check_step(dec, rec, o, f, t, k, TOL[precision])
    Lsteps = o["hid"].shape[0]
    tokens_in = torch.cat((torch.ones(1, f.shape[0], dtype=torch.long, device=dev()), t[: Lsteps - 1]), 0)
    logits, _ = dec["model"].teacher_forced_logits(tokens_in, f)
    assert rel(logits, o["logits"]) < TOL[precision]


def test_softmax_and_mean_attention_give_different_losses():
    gl = load_golden("small_lstm")
    m = dict(gl["meta"], rec_model="LSTM")
    f, t = gl["feats"].float().to(dev()), gl["targets"].to(dev())
    out = []
    for flag in (False, True):
        dec, rec = build_sm(m, "bf16", gl["dec"], gl["local"], softmax=flag)
        with torch.no_grad():
            dl, hid, _ = T.forward_decoder(dec, f, t, t > 0, 1.0)
            rl = T.forward_local_reconstructor(hid, f, rec)
        out.append((float(dl), float(rl)))
    assert abs(out[0][0] - gl["dec_loss"]) / abs(gl["dec_loss"]) < 2e-2       # flag off: the reference's numbers
    assert abs(out[0][0] - out[1][0]) > 1e-4 * abs(out[0][0]) and abs(out[0][1] - out[1][1]) > 1e-4 * abs(out[0][1])


# ---- train mode, same Philox masks as the oracle ------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_full_size_train_mode_parity_with_the_same_masks(precision):
    m = FULL
    feats, targets, masks = _full_inputs()
    P = O.init_decoder_params(m["V"], m["EMB"], m["E"], m["H"], m["A"], seed=0)
    Q = O.init_reconstructor_params("local", m["H"], m["E"], m["A"], seed=1)
    C = T.C
    B, Lmax, Tn, H = 100, 31, m["T"], m["H"]
    drops = dict(emb=philox_scales(0xDEC0, 1, SITE_EMB, (Lmax, B, m["EMB"]), C.embedding_dropout),
                 logits=philox_scales(0xDEC0, 1, SITE_LOGITS, (Lmax, B, m["V"]), C.decoder_out_dropout),
                 x=philox_scales(0x10CA, 1, SITE_LOCAL_X, (Tn, B, H), C.reconstructor_decoder_dropout))
    o = oracle_grads(m, P, Q, feats, targets, masks, drops)
    dec, rec = build_sm(m, precision, P, Q)
    dec["model"].train(); rec["model"].train()
    dec["model"].seed_dropout(0xDEC0); rec["model"].seed_dropout(0x10CA)
    check_step(dec, rec, o, feats.to(dev()), targets.to(dev()), masks.to(dev()), TOL[precision])


# ---- other cells / depths ----------------------------------------------------------------------------------------------------
SMALL = dict(B=6, T=7, E=64, H=32, A=16, EMB=24, V=101, cap_len=6, rec_layers=1, rec_model="LSTM")
VARIANTS = {
    "gru_decoder": dict(SMALL, dec_model="GRU", dec_layers=1, fused=(True, True)),
    "lstm_decoder_2_layers": dict(SMALL, dec_model="LSTM", dec_layers=2, fused=(True, True)),
    "gru_2_layers_gru_rec": dict(SMALL, dec_model="GRU", dec_layers=2, rec_model="GRU", fused=(False, False)),   # both step-wise
}


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_variants_match_oracle(variant, precision):
    m = VARIANTS[variant]
    feats, targets, masks = O.synthetic_batch(m["B"], m["T"], m["E"], m["V"], m["cap_len"], seed=5)
    P = O.init_decoder_params(m["V"], m["EMB"], m["E"], m["H"], m["A"], n_layers=m["dec_layers"], model_name=m["dec_model"], seed=2)
    Q = O.init_reconstructor_params("local", m["H"], m["E"], m["A"], model_name=m["rec_model"], seed=3)
    o = oracle_grads(m, P, Q, feats, targets, masks)
    dec, rec = build_sm(m, precision, P, Q)
    assert (dec["model"].uses_fused_sequence, rec["model"]._fused_ok(o["hid"])) == m["fused"]
    check_step(dec, rec, o, feats.to(dev()), targets.to(dev()), masks.to(dev()), TOL[precision])


# ---- search ------------------------------------------------------------------------------------------------------------------
def test_fp32_greedy_ids_equal_the_oracle():
    feats, _, _ = _full_inputs(100, seed=77)
    P = O.init_decoder_params(FULL["V"], FULL["EMB"], FULL["E"], FULL["H"], FULL["A"], seed=0)
    P["out.bias"][0] += 3.0                     # lets the <PAD>-stop rule fire
    ref = S.greedy_search(P, feats, attn_softmax=True)
    dec, _ = build_sm(FULL, "fp32", P, None)
    ids, n = dec["model"].greedy(feats.to(dev()), 31)
    assert int(n) == ref.shape[0]
    assert torch.equal(ids[: int(n)].cpu(), ref)


def _per_step_greedy(model, feats, steps):
    B = feats.shape[0]
    z = torch.zeros(model.n_layers, B, model.hidden_size, device=dev())
    hid = (z, z.clone()) if model.model_name == "LSTM" else z
    tok = torch.ones(1, B, dtype=torch.long, device=dev())
    out = []
    with torch.no_grad(), model.cached_uv(feats):
        for _ in range(steps):
            logits, hid = model.forward(tok, hid, feats)
            tok = logits.argmax(dim=1).view(1, -1)
            out.append(tok[0])
    return torch.stack(out)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_device_greedy_equals_the_per_step_api_loop(precision):
    g = load_golden_beam("small_lstm")
    m = dict(g["meta"], rec_model="LSTM")
    dec, _ = build_sm(m, precision, g["dec"], None)
    feats = g["feats"].float().to(dev())
    ids, n = dec["model"].greedy(feats, m["cap_len"] + 1)
    ref = _per_step_greedy(dec["model"], feats, int(n))
    assert torch.equal(ids[: int(n)], ref)


@pytest.mark.parametrize("width", [3, 5])
def test_beam_device_loop_equals_per_step_loop_and_oracle(width, monkeypatch):
    g = load_golden("tiny_lstm")
    m = dict(g["meta"], rec_model="LSTM")
    P = {k: v.float() for k, v in g["dec"].items()}
    P["out.bias"] = P["out.bias"].clone()
    P["out.bias"][2] += 1.5                      # <EOS> likely enough that the length normalisation is exercised
    dec, _ = build_sm(m, "fp32", P, None)
    feats = g["feats"].float().to(dev())
    B, H = feats.shape[0], m["H"]
    T.C.batch_size = B
    got = {}
    for loop in ("1", "0"):                      # RECNET_BEAM_DEVICE: 1 = recnet_decoder_beam, 0 = loop over Decoder.forward
        monkeypatch.setenv("RECNET_BEAM_DEVICE", loop)
        tok = torch.ones(1, B, dtype=torch.long, device=dev())
        z = torch.zeros(1, B, H, device=dev())
        got[loop] = E.beam_search(T.C, width, _Vocab(m["V"]), dec["model"], tok, (z, z.clone()), feats)
    ref = S.beam_search(P, g["feats"].float(), width, caption_max_len=m["cap_len"], attn_softmax=True)
    assert got["1"] == got["0"] == ref, (got, ref)


# ---- CUDA graph ----------------------------------------------------------------------------------------------------------------
def test_train_step_cuda_graph_replay_equals_eager():
    gl = load_golden("small_lstm")
    m = dict(gl["meta"], rec_model="LSTM")
    feats, targets = gl["feats"].float().to(dev()), gl["targets"].to(dev())
    Lsteps = gl["hiddens"].shape[0]
    arms = [build_sm(m, "bf16", gl["dec"], gl["local"]) for _ in range(2)]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for dec, rec in arms:
            for _ in range(3):
                T.train_step(dec, rec, feats, targets, n_steps=Lsteps)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    out = torch.zeros((), device=dev())
    with torch.cuda.graph(graph):
        loss, _, _ = T.train_step(*arms[1], feats, targets, n_steps=Lsteps)
        out.copy_(loss.detach())
    for _ in range(2):
        eager, _, _ = T.train_step(*arms[0], feats, targets, n_steps=Lsteps)
        graph.replay()
        torch.cuda.synchronize()
        assert rel(out, eager.detach()) < 1e-5
    for (k, a), b in zip(arms[0][0]["model"].named_parameters(), arms[1][0]["model"].parameters()):
        assert rel(b, a) < 1e-5, k
    for (k, a), b in zip(arms[0][1]["model"].named_parameters(), arms[1][1]["model"].parameters()):
        assert rel(b, a) < 1e-5, k


# ---- opt-in kernel paths (switches are read once per process: child processes) --------------------------------------------------------
SELECT = "eval_mode or train_mode or variants or greedy or cuda_graph"


@pytest.mark.parametrize("switches", [
    {"RECNET_DEC_CLUSTER": "0", "RECNET_GREEDY_PF": "0"},      # decoder forward loop / greedy on the per-step projected-feature kernels
    {"RECNET_PERSIST": "0", "RECNET_PERSIST_BWD": "0"},        # kernel-per-phase reconstructor loops
    {"RECNET_BG_WGRAD": "0"},                                  # no background lane
], ids=["no_cluster", "kernel_per_phase", "no_background_lane"])
def test_opt_in_paths_stay_parity_green_with_softmax(switches):
    if os.environ.get("RECNET_ATTN_SOFTMAX_CHILD"):
        pytest.skip("already in a child process")
    env = dict(os.environ, RECNET_ATTN_SOFTMAX_CHILD="1", **switches)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider",
                        "-k", SELECT], capture_output=True, text=True, timeout=1200, cwd=ROOT, env=env)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and " failed" not in r.stdout, tail
