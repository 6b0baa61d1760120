"""The checks of tests/test_gpu_loop_shapes.py are sharp enough to see a loop kernel that is subtly wrong: each fault below, applied to the
fp64 oracle's inputs the way a kernel bug would corrupt them, moves some checked quantity (loss, a gradient, hiddens or d hiddens, per
sample where there is a batch axis) by more than 5x the bf16 tolerance.  Oracle only, no GPU."""
import contextlib
import functools

import pytest
import torch

from oracle import recnet_oracle as O
from tests.test_gpu_loop_shapes import (BF16_TOL, case, dec_drops, dec_inputs, dec_oracle, errors, rec_drop, rec_inputs, rec_oracle,
                                        seed_of)

MARGIN = 5


def _other_sample(x, axis):
    """The last sample takes the second-to-last one's data (a kernel that indexes samples one off)."""
    x = x.clone()
    x.select(axis, -1).copy_(x.select(axis, -2))
    return x


def _zero(x, index):
    x = x.clone()
    x[index] = 0
    return x


REC_FAULTS = {
    "last sample reads the previous sample's decoder states": lambda hid, drop: (_other_sample(hid, 2), drop),
    "last key of one sample zeroed": lambda hid, drop: (_zero(hid, (-1, slice(None), -1)), drop),
    "unit H-1 of the decoder states zeroed": lambda hid, drop: (_zero(hid, (Ellipsis, -1)), drop),
}
REC_TRAIN_FAULTS = dict(REC_FAULTS, **{
    "site-3 dropout mask shifted by one element": lambda hid, drop: (hid, drop.flatten().roll(1).view_as(drop)),
})


@contextlib.contextmanager
def _lstm_drops_last_unit():
    """The decoder's cell writes h[:, H-1] = 0 at every step (a kernel that drops the last unit of its tile)."""
    cell = O.lstm_cell

    def faulty(*args):
        h, c = cell(*args)
        return _zero(h, (slice(None), -1)), c

    O.lstm_cell = faulty
    try:
        yield
    finally:
        O.lstm_cell = cell


DEC_FAULTS = {
    "last sample reads the previous sample's features": lambda feats: (_other_sample(feats, 0), contextlib.nullcontext()),
    "last frame of one sample zeroed": lambda feats: (_zero(feats, (-1, -1)), contextlib.nullcontext()),
    "unit H-1 of the decoder states zeroed": lambda feats: (feats, _lstm_drops_last_unit()),
}

CASES = ([("R3", False, f) for f in REC_FAULTS] + [("R6", False, f) for f in REC_FAULTS] + [("D5", False, f) for f in DEC_FAULTS] +
         [("R6", True, f) for f in REC_TRAIN_FAULTS])


@functools.lru_cache(maxsize=None)
def _clean(cid, train):
    c, seed = case(cid), seed_of(cid)
    if cid.startswith("D"):
        feats, targets, masks, P = dec_inputs(c, seed)
        drops = dec_drops(masks, seed) if train else None
        return c, (feats, targets, masks, P, drops), dec_oracle(feats, targets, masks, P, drops=drops)
    hid, feats, Q = rec_inputs(c, seed)
    drop = rec_drop(c, seed) if train else None
    return c, (hid, feats, Q, drop), rec_oracle(c, hid, feats, Q, drop=drop)


@pytest.mark.parametrize("cid,train,fault", CASES, ids=[f"{c}-{'train' if t else 'eval'}-{f}" for c, t, f in CASES])
def test_each_fault_moves_a_checked_quantity_beyond_five_times_the_tolerance(cid, train, fault):
    c, inputs, ref = _clean(cid, train)
    if cid.startswith("D"):
        feats, targets, masks, P, drops = inputs
        feats, ctx = DEC_FAULTS[fault](feats)
        with ctx:
            got = dec_oracle(feats, targets, masks, P, drops=drops)
    else:
        hid, feats, Q, drop = inputs
        hid, drop = (REC_TRAIN_FAULTS if train else REC_FAULTS)[fault](hid, drop)
        got = rec_oracle(c, hid, feats, Q, drop=drop)
    err = errors(got, ref)
    name, worst = max(err.items(), key=lambda kv: kv[1])
    print(f"{cid} {fault}: {name} moves by {worst:.3g} = {worst / BF16_TOL:.1f}x the tolerance")
    assert worst > MARGIN * BF16_TOL, (cid, fault, sorted(err.items(), key=lambda kv: -kv[1])[:4])
