"""numpy restatement of the in-kernel Philox4x32-10 dropout masks (csrc/common.cuh:Philox / dropout_scale) -- TEST INFRASTRUCTURE.

A dropout site draws, for element ``idx`` of that site's tensor, word ``idx & 3`` of Philox(counter = idx >> 2,
stream = (offset << 8) | site, key = seed); the element is kept when (word >> 8) / 2**24 >= p and scaled by 1 / (1 - p)
(inverted dropout, what nn.Dropout does: models/decoder.py:48,69, models/local_reconstructor.py:50,
models/global_reconstructor.py:38).  (seed, offset) is the module's ``_rng`` buffer; the offset is bumped once per training forward.

Sites and element order (must match the kernels):
  1 SITE_EMB      : [L, B, EMB]   embedding * scale, then dropout            (misc.cuh:embed_gather_kernel)
  2 SITE_LOGITS   : [L, B, V]     logits dropped BEFORE the cross entropy    (losses.cuh:ce_fwd_kernel)
  3 SITE_LOCAL_X  : [S, B, H]     attended decoder state of the local reconstructor (attention_lean.cuh / seq_recon_persist.cuh);
                    over a stacked decoder [S, NLd, B, H]: outer step t, decoder layer l is pseudo-step q = t*NLd + l
                    (seq_recon.cuh:local_forward, drop_base = q*B*H)
  4 SITE_GLOBAL_MP: [L, B, H]     mean-pooled decoder state of the global reconstructor, a fresh mask every step (misc.cuh:global_x_kernel)
 17..19           : [L, B, H]     inter-layer dropout of a stacked LSTM decoder (nn.LSTM(dropout=p)): the input of layer l
                    (1 <= l <= NL-1) uses site SITE_LAYER0 + l; it multiplies only the copy of h^{l-1}_t fed to layer l
                    (seq_decoder.cuh: lstm_cell.cuh h_op2 in the forward, q_drop in the backward)
"""
import numpy as np

SITE_EMB, SITE_LOGITS, SITE_LOCAL_X, SITE_GLOBAL_MP = 1, 2, 3, 4
SITE_LAYER0 = 16                     # + l: input of decoder layer l >= 1
M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, stream, seed):
    """ctr: uint64 array; stream, seed: python ints.  Returns four uint32 arrays (as uint64 holding 32-bit values)."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    c0, c1 = ctr & M32, ctr >> np.uint64(32)
    c2 = np.full_like(c0, np.uint64(stream & 0xFFFFFFFF))
    c3 = np.full_like(c0, np.uint64((stream >> 32) & 0xFFFFFFFF))
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    A, Bc = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    for _ in range(10):
        p0, p1 = A * c0, Bc * c2                       # 32 x 32 -> 64 bit products fit uint64
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & M32, p1 >> np.uint64(32), p1 & M32
        c0, c1, c2, c3 = hi1 ^ c1 ^ np.uint64(k0), lo1, hi0 ^ c3 ^ np.uint64(k1), lo0
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return c0, c1, c2, c3


def dropout_scales(seed, offset, site, n, p):
    """float32 array [n]: 0 or 1/(1-p) for elements 0..n-1 of the site (1 everywhere when p <= 0)."""
    if p <= 0.0:
        return np.ones(n, dtype=np.float32)
    idx = np.arange(n, dtype=np.uint64)
    words = philox4x32_10(idx >> np.uint64(2), (int(offset) << 8) | int(site), int(seed))
    sel = (idx & np.uint64(3)).astype(np.int64)
    w = np.choose(sel, words)
    u = (w >> np.uint64(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    return np.where(u >= np.float32(p), np.float32(1.0 / (1.0 - p)), np.float32(0.0)).astype(np.float32)
