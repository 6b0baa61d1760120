"""CPU checks of the decode entry points' coverage: recnet_decoder_greedy / recnet_decoder_beam take LSTM decoders with 1-4 layers and
single-layer GRU; a stacked GRU and more than RECNET_MAX_LAYERS layers are refused with RECNET_ERR_UNSUPPORTED before anything is
launched (null buffers, no GPU needed)."""
import ctypes as C

import pytest

from recnet_b200 import _lib as L

UNSUPPORTED = -4
SHAPE = dict(B=6, T=5, E=16, H=8, A=8, EMB=8, V=11, L=1)


def _desc(cell, n_layers, precision):
    return L.decoder_desc(precision=precision, train=0, embedding_scale=1.0, p_emb_drop=0.0, p_out_drop=0.0, cell=cell, n_layers=n_layers,
                          **SHAPE)


@pytest.mark.parametrize("precision", [L.PREC_FP32, L.PREC_BF16])
@pytest.mark.parametrize("cell,n_layers", [(L.CELL_GRU, 2), (L.CELL_LSTM, L.MAX_LAYERS + 1)])
def test_decode_entry_points_refuse_what_they_do_not_cover(cell, n_layers, precision):
    lib = L.lib()
    w = L.decoder_tensors()
    for sm in (0, L.ATTN_SOFTMAX):
        d = C.byref(_desc(cell | sm, n_layers, precision))
        assert lib.recnet_decoder_greedy(d, C.byref(w), None, 31, None, 0, None, None, None) == UNSUPPORTED
        assert lib.recnet_decoder_beam(d, C.byref(w), None, 3, 31, 2, None, 0, None, None, None) == UNSUPPORTED
