"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the act kernel's dropout masks
(jsrl_corl_b200/csrc/common.cuh::philox_act_dropout_quad), built on oracle/philox.py's Philox4x32-10."""
import numpy as np

from oracle.philox import dropout_threshold, philox4x32_10

STREAM_ACT_DROPOUT_BASE = 0x80000000


def philox_act_dropout_mask(seed: int, step: int, layer: int, n: int, p: float) -> np.ndarray:
    """Keep-mask (uint8) of the n units of hidden layer ``layer`` in the training-mode act at act counter ``step``:
    unit j is kept iff word j & 3 of Philox4x32-10(counter = (j >> 2, step lo, step hi, 0x80000000 + layer),
    key = (seed lo, seed hi)) is >= floor(p * 2^32)."""
    quads = np.arange((n + 3) // 4, dtype=np.uint64)
    x, y, z, w = philox4x32_10(quads, step & 0xFFFFFFFF, (step >> 32) & 0xFFFFFFFF, STREAM_ACT_DROPOUT_BASE + layer,
                               seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    words = np.stack([x, y, z, w], axis=1).reshape(-1)[:n]
    return (words >= np.uint32(dropout_threshold(p))).astype(np.uint8)
