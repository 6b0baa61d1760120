"""CPU tests of the host-side mirror: module surface (ctor kwargs, state_dict keys/shapes/order, initialiser
parity with the reference's seeds), config names, loop-length logic, sharding, and the 2-rank gloo path of the
gradient all-reducer."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import recnet_b200
from recnet_b200 import train as T
from recnet_b200.data import shard_range, synthetic_batch
from recnet_b200.parallel import GradAllReducer
from oracle import recnet_oracle as O
from tests.golden_util import golden_cases, load_golden


def test_state_dict_matches_reference_fixture_keys_and_shapes():
    g = load_golden("tiny_lstm")
    m = g["meta"]
    dec = recnet_b200.Decoder("LSTM", 1, m["E"], m["EMB"], 1, m["H"], m["A"], m["V"], 0.5, 0.5, 0.5)
    assert list(dec.state_dict().keys()) == list(g["dec"].keys())          # same keys in the same order
    dec.load_state_dict({k: v.float() for k, v in g["dec"].items()})
    loc = recnet_b200.LocalReconstructor("LSTM", 1, m["H"], m["E"], 0.5, 0.5, m["A"])
    assert list(loc.state_dict().keys()) == list(g["local"].keys())
    loc.load_state_dict({k: v.float() for k, v in g["local"].items()})
    glo = recnet_b200.GlobalReconstructor("LSTM", 1, m["H"], m["E"], 0.5, 0.5, m["cap_len"])
    assert list(glo.state_dict().keys()) == list(g["global"].keys())
    glo.load_state_dict({k: v.float() for k, v in g["global"].items()})


def test_default_shapes_are_the_msvd_ones():
    dec = recnet_b200.Decoder("LSTM", 1, 1536, 468, 1, 512, 128, 4188, 0.5, 0.5, 0.5)
    sd = dec.state_dict()
    assert tuple(sd["rnn.weight_ih_l0"].shape) == (2048, 2004) and tuple(sd["out.weight"].shape) == (4188, 512)
    assert bool((sd["attn_b"] == 1).all())                                  # decoder.py:27 initialises the bias to ones
    assert sum(p.numel() for p in dec.parameters()) == 9527692              # SURVEY 8a A0


def test_same_seed_same_initial_weights_as_reference():
    """Every fixture's decoder weights are what the reference's own constructor drew after torch.manual_seed(seed), with fp64 as
    the default dtype (tests/golden/make_golden.py): the same seed draws the same weights here, bit for bit."""
    for name in golden_cases():
        g = load_golden(name)
        m = g["meta"]
        saved = torch.get_default_dtype()
        torch.set_default_dtype(torch.float64)
        try:
            torch.manual_seed(m["seed"])
            b = recnet_b200.Decoder(m["dec_model"], m["dec_layers"], m["E"], m["EMB"], 1, m["H"], m["A"], m["V"], 0.5, 0.5, 0.5).state_dict()
        finally:
            torch.set_default_dtype(saved)
        assert list(b) == list(g["dec"]), name
        for k, a in g["dec"].items():
            assert torch.equal(a, b[k]), (name, k)


def test_config_keeps_reference_attribute_names():
    # the defaults as config.py declares them: other tests reconfigure the shared TrainConfig in place
    import importlib.util
    from recnet_b200 import config
    spec = importlib.util.spec_from_file_location("recnet_config_defaults", config.__file__)
    fresh = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fresh)
    C = fresh.TrainConfig
    for name, val in dict(decoder_model="GRU", reconstructor_model="LSTM", caption_max_len=30, batch_size=100, embedding_size=468,
                          encoder_output_size=1536, encoder_output_len=28, decoder_hidden_size=512, decoder_attn_size=128,
                          reconstructor_hidden_size=1536, reconstructor_attn_size=128, decoder_teacher_forcing_ratio=1.0,
                          gradient_clip=50.0, decoder_learning_rate=1e-5, reconstructor_learning_rate=1e-6).items():
        assert hasattr(recnet_b200.TrainConfig, name) and getattr(C, name) == val, name
    assert C.init_word2idx == {'<PAD>': 0, '<SOS>': 1, '<EOS>': 2}


def test_every_reference_variant_is_accepted_and_unknown_names_raise():
    gru = recnet_b200.Decoder("GRU", 1, 16, 8, 1, 8, 8, 11, 0.5, 0.5, 0.5)
    assert tuple(gru.state_dict()["rnn.weight_ih_l0"].shape) == (24, 24)    # 3 gates: checkpoint-compatible holder
    # variants without a fused sequence driver run as a loop over the per-step kernels -- visible, never silent
    assert not recnet_b200.Decoder("GRU", 2, 16, 8, 1, 8, 8, 11, 0.5, 0.5, 0.5).uses_fused_sequence
    rec = recnet_b200.LocalReconstructor("LSTM", 2, 8, 16, 0.5, 0.5, 8)
    assert not rec._fused_ok(torch.zeros(3, 2, 8))
    assert tuple(rec.state_dict()["rnn.weight_ih_l1"].shape) == (64, 16)
    with pytest.raises(RuntimeError):           # ... and the per-step kernels have no CPU path either
        rec.forward_sequence(torch.zeros(3, 2, 8), torch.zeros(2, 4, 16))
    with pytest.raises(NotImplementedError):
        T.forward_reconstructor_for("bogus")


def test_num_steps_follows_reference_break_rule():
    feats, targets, masks = synthetic_batch(6, 4, 8, 20, caption_max_len=9, seed=3, full_length_first=False)
    lens = masks.sum(0)
    assert T._num_steps(masks, 9) == int(lens.max())                        # loop stops after the last non-empty row
    feats, targets, masks = synthetic_batch(6, 4, 8, 20, caption_max_len=9, seed=3)
    assert T._num_steps(masks, 9) == 10


def test_synthetic_batch_equals_oracle_generator():
    a = synthetic_batch(5, 7, 8, 30, 12, seed=99)
    b = O.synthetic_batch(5, 7, 8, 30, 12, seed=99)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_shard_range_partitions():
    for n, w in ((800, 8), (100, 3), (7, 8)):
        got = [shard_range(n, r, w) for r in range(w)]
        assert got[0][0] == 0 and got[-1][1] == n and all(got[i][1] == got[i + 1][0] for i in range(w - 1))


def _gloo_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.manual_seed(0)
    m = torch.nn.Linear(4, 3)
    red = GradAllReducer([m])
    red.start_iteration()
    # emulate what the sequence Functions do: all gradients of the module are views of ONE flat buffer that is created INSIDE
    # backward and referenced by nothing but its views afterwards (every later `.grad._base` is then a fresh Python wrapper)

    class Fn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, w, b):
            return (w.sum() + b.sum()) * 0

        @staticmethod
        def backward(ctx, g):
            flat = torch.arange(15, dtype=torch.float32) * (rank + 1)
            return flat[:12].view(3, 4), flat[12:15]

    Fn.apply(m.weight, m.bias).backward()
    red.wait()
    expect = torch.arange(15, dtype=torch.float32) * (sum(range(1, world + 1)) / world)
    ok = torch.allclose(m.weight.grad.flatten(), expect[:12]) and torch.allclose(m.bias.grad, expect[12:])
    ok = ok and red.bytes_last == 15 * 4
    # gradients written into ONE flat buffer by a sequence Function (functional._flat_grads): autograd stores the views detached,
    # RECNET_DP_FLAT=1 finds the buffer again and sends ONE all-reduce for the module (padding included), default = one per tensor
    from recnet_b200 import functional as RF
    for flat_on in (True, False):
        m3 = torch.nn.Linear(4, 3)
        red3 = GradAllReducer([m3]); red3.flat_lookup = flat_on; red3.start_iteration()

        class SeqFn(torch.autograd.Function):
            @staticmethod
            def forward(ctx, w, b):
                ctx.save_for_backward(w, b)
                return (w.sum() + b.sum()) * 0

            @staticmethod
            def backward(ctx, g):
                flat, views, _ = RF._flat_grads(ctx.saved_tensors)
                flat.fill_(float("nan"))                                     # padding between the views: must not matter
                views[0].copy_(torch.arange(12, dtype=torch.float32).view(3, 4) * (rank + 1))
                views[1].copy_(torch.arange(3, dtype=torch.float32) * (rank + 1))
                return tuple(views)

        SeqFn.apply(m3.weight, m3.bias).backward()
        assert m3.weight.grad._base is None                                  # what autograd does to the views it is handed
        red3.wait()
        scale = sum(range(1, world + 1)) / world
        ok = ok and torch.allclose(m3.weight.grad, torch.arange(12, dtype=torch.float32).view(3, 4) * scale)
        ok = ok and torch.allclose(m3.bias.grad, torch.arange(3, dtype=torch.float32) * scale)
        ok = ok and red3.bytes_last == ((64 + 64) * 4 if flat_on else 15 * 4)
    # per-tensor fallback when grads are not flat views
    m2 = torch.nn.Linear(2, 2)
    red2 = GradAllReducer([m2]); red2.start_iteration()
    m2(torch.ones(1, 2) * (rank + 1)).sum().backward()
    red2.wait()
    ok = ok and torch.allclose(m2.bias.grad, torch.ones(2)) and torch.allclose(m2.weight.grad, torch.full((2, 2), (1 + world) / 2))
    out[rank] = bool(ok)
    dist.destroy_process_group()


def test_grad_allreducer_two_ranks_gloo():
    world = 2
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_gloo_worker, args=(world, 29533, out), nprocs=world, join=True)
        assert all(out[r] for r in range(world)), dict(out)


def test_beam_search_bookkeeping_matches_oracle_on_cpu():
    """recnet_b200.eval.beam_search's batched bookkeeping (top-k, state gather, <EOS>-length tracking) against the
    oracle's loop restatement of eval.py:36-120, using the oracle's decoder step as the decoder callable (CPU)."""
    from recnet_b200 import eval as E

    for name in ("tiny_lstm", "tiny_gru"):
        g = load_golden(name, dtype=torch.float32)
        m = g["meta"]
        P = dict(g["dec"])
        P["out.bias"] = P["out.bias"].clone()
        P["out.bias"][2] += 1.5

        class Cfg:
            caption_max_len, decoder_model = m["cap_len"], m["dec_model"]

        class Vocab:
            n_vocabs, word2idx = m["V"], {'<PAD>': 0, '<SOS>': 1, '<EOS>': 2}

        def decoder(tok, hid, feats):
            return O.decoder_step(P, tok, hid, feats, model_name=m["dec_model"], n_layers=1)

        B = g["feats"].shape[0]
        tok = torch.full((1, B), 1, dtype=torch.long)
        hid = O.zero_hidden(m["dec_model"], 1, B, m["H"], g["feats"])
        for width in (2, 5):
            ref = O.beam_search(P, g["feats"], width, model_name=m["dec_model"], n_layers=1, caption_max_len=m["cap_len"])
            got = E.beam_search(Cfg, width, Vocab, decoder, tok, hid, g["feats"])
            assert got == ref, (name, width)


def test_clip_adam_host_side_validation_and_optimizer_selection(monkeypatch):
    """optim.ClipAdam (the fused clip + Adam of train.py:269-273): argument checks run on the host; there is no CPU compute path."""
    import torch
    from recnet_b200.optim import ClipAdam
    from recnet_b200 import train as T
    p = [torch.zeros(4, requires_grad=True)]
    with pytest.raises(ValueError):
        ClipAdam(p, lr=-1.0)
    with pytest.raises(ValueError):
        ClipAdam(p, lr=1e-3, betas=(1.0, 0.999))
    with pytest.raises(NotImplementedError):
        ClipAdam([{"params": p}, {"params": [torch.zeros(2, requires_grad=True)]}], lr=1e-3)
    o = ClipAdam(p, lr=1e-3, weight_decay=1e-5, amsgrad=True, max_grad_norm=50.0)
    g = o.param_groups[0]
    assert (g["lr"], g["betas"], g["eps"], g["weight_decay"], g["amsgrad"], g["max_grad_norm"]) == (1e-3, (0.9, 0.999), 1e-8, 1e-5, True, 50.0)
    p[0].grad = torch.zeros(4)
    with pytest.raises(RuntimeError, match="no CPU path"):
        o.step()
    monkeypatch.setenv("RECNET_OPTIMIZER", "recnet")
    assert T._optimizer_impl() == "recnet"
    monkeypatch.setenv("RECNET_OPTIMIZER", "sgd")
    with pytest.raises(ValueError):
        T._optimizer_impl()
    monkeypatch.delenv("RECNET_OPTIMIZER")
    assert T._optimizer_impl() == T.C.optimizer_impl


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): exactly one JSON line with the contract keys."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "decoder + local reconstructor" in d["config"]["workload"]


def test_bench_roofline_work_formulas():
    """bench.py's algorithmic-work helpers (DESIGN.md section 5): GEMM flops count useful rows only, GEMM bytes are operands once +
    result once, and a skinny per-step GEMM sits below the machine balance (so its binding roofline is bytes, not the tensor pipe)."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    bound, flops = bench.algorithmic_work(1, 100, 6144, 2048, 2)
    assert bound == "tensor" and flops == 2.0 * 100 * 6144 * 2048
    nbytes = bench.gemm_bytes(100, 6144, 2048, 2)
    assert nbytes == (100 * 2048 + 6144 * 2048) * 2 + 100 * 6144 * 4
    pk = bench.peaks()
    balance = pk["tf_sust"] * 1e12 / (pk["hbm"] * 1e9)
    assert flops / nbytes < balance                                   # per-step gate GEMM: memory-bound
    big = bench.algorithmic_work(1, 6144, 1536, 2800, 2)[1] / bench.gemm_bytes(6144, 1536, 2800, 2)
    assert big > balance                                              # batched weight-gradient GEMM: tensor-bound
    for cls in (3, 4, 5, 6, 7, 8, 10, 11):
        b, work = bench.algorithmic_work(cls, 100, 28, 512, 2)
        assert b == "hbm" and work > 0
    assert set(bench.KCLASS) >= {1, 3, 4, 5, 6, 10, 11}
