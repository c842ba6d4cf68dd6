"""Dropout masks of a shard of a larger batch (checker side): the mask rule of ``oracle/train_ref.py`` with the global
sequence index ``2 * (first + b) + part`` of ``aft_forward_train_offset``."""
from typing import List

import numpy as np
import torch

from oracle import train_ref as T


def masks_for(seed: int, samples: int, part: int, layers: int, p: float, first: int = 0) -> List[List[torch.Tensor]]:
    """masks[layer][site]: float64 [samples, *SITE_SHAPES[site]] of one pass (part 0 = real, 1 = imaginary) for the
    global samples ``first .. first + samples - 1``.  With ``first = 0`` this is ``oracle.train_ref.masks_for``."""
    return [[torch.from_numpy(np.stack([T.keep_mask(seed, 2 * (first + b) + part, l, s, T.SITE_SHAPES[s], p)
                                        for b in range(samples)]).astype(np.float64))
             for s in range(4)] for l in range(layers)]
