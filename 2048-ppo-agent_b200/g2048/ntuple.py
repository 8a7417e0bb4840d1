"""N-tuple networks: the value function of the strong learned 2048 players (Szubert & Jaśkowski 2014; Yeh et al. 2016).

    net = g2048.NTupleNetwork.four_six()                     # 4 six-cell tuples x 8 symmetries, 2^26 weights
    learner = g2048.NTupleTDLearner(0, batch_size=1 << 16, network=net)
    learner.train(4000)
    player = g2048.ExpectimaxPolicy(depth=1, network=net, reward_weight=1.0)

A network is an ordered list of placements over one flat float32 weight array ``W``.  Placement p reads k cells of the
board and indexes its table with their exponents (nibble j = the exponent in cells[j]):
``V(b) = W[off_0 + idx_0(b)] + ... + W[off_{P-1} + idx_{P-1}(b)]`` in float32, left to right (include/g2048.h).
Placements with the same offset share a table: the 8 symmetric images of a tuple learn one set of weights.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native as N

# G2048TuplePlacement (include/g2048.h), 12 bytes
PLACEMENT_DTYPE = np.dtype([("offset", "<u4"), ("n_cells", "u1"), ("cells", "u1", (6,)), ("reserved", "u1")])
MAX_PLACEMENTS = 64
MAX_WEIGHTS = 1 << 28

# the 8 symmetries of the square, as maps of (row, col), in the order of NTupleNetwork.from_tuples
SYMMETRIES = (
    lambda r, c: (r, c), lambda r, c: (r, 3 - c), lambda r, c: (3 - r, c), lambda r, c: (3 - r, 3 - c),
    lambda r, c: (c, r), lambda r, c: (c, 3 - r), lambda r, c: (3 - c, r), lambda r, c: (3 - c, 3 - r),
)
FOUR_SIX_TUPLES = ((0, 1, 2, 3, 4, 5), (4, 5, 6, 7, 8, 9), (0, 1, 2, 4, 5, 6), (4, 5, 6, 8, 9, 10))


def symmetric_images(cells) -> list[tuple[int, ...]]:
    """The 8 images of a tuple of cells (cell = 4 * row + col) under SYMMETRIES, in that order."""
    out = []
    for f in SYMMETRIES:
        out.append(tuple(4 * r + c for r, c in (f(x >> 2, x & 3) for x in cells)))
    return out


def make_placements(rows) -> np.ndarray:
    """A placement array from (offset, cells) pairs."""
    pl = np.zeros(len(rows), PLACEMENT_DTYPE)
    for i, (offset, cells) in enumerate(rows):
        cells = [int(c) for c in cells]
        if not 1 <= len(cells) <= 6 or any(not 0 <= c < 16 for c in cells):
            raise ValueError(f"a placement has 1..6 cells in 0..15, got {cells}")
        pl[i]["offset"] = int(offset)
        pl[i]["n_cells"] = len(cells)
        pl[i]["cells"][: len(cells)] = cells
    return pl


def check_placements(placements, n_weights: int) -> np.ndarray:
    """The checks of the C entry points (include/g2048.h): a C-contiguous PLACEMENT_DTYPE copy, or ValueError."""
    n_weights = int(n_weights)
    if not 1 <= n_weights <= MAX_WEIGHTS:
        raise ValueError(f"n_weights must be in [1, 2^28], got {n_weights}")
    pl = np.ascontiguousarray(np.asarray(placements))
    if pl.dtype != PLACEMENT_DTYPE or pl.ndim != 1:
        raise ValueError("placements must be a 1-d array of PLACEMENT_DTYPE")
    if not 1 <= pl.shape[0] <= MAX_PLACEMENTS:
        raise ValueError(f"a network has 1..64 placements, got {pl.shape[0]}")
    for i, p in enumerate(pl):
        k = int(p["n_cells"])
        if not 1 <= k <= 6:
            raise ValueError(f"placement {i}: n_cells must be in 1..6 and every cell < 16")
        cells = [int(c) for c in p["cells"][:k]]
        if any(c >= 16 for c in cells) or len(set(cells)) != k:
            raise ValueError(f"placement {i}: cells must be < 16 and distinct, got {cells}")
        if int(p["reserved"]) != 0:
            raise ValueError(f"placement {i}: reserved must be 0")
        if int(p["offset"]) + 16 ** k > n_weights:
            raise ValueError(f"placement {i}: offset + 16^{k} exceeds n_weights = {n_weights}")
    return pl.copy()


def _check_weights(weights, n_weights: int) -> torch.Tensor:
    w = weights.detach() if isinstance(weights, torch.Tensor) else torch.from_numpy(np.asarray(weights, np.float32))
    if w.numel() != n_weights:
        raise ValueError(f"weights must hold n_weights = {n_weights} values, got {w.numel()}")
    w = w.reshape(n_weights).to(torch.float32)
    if not bool(torch.isfinite(w).all()):
        raise ValueError("weights must be finite")
    return w


class NTupleNetwork:
    """``placements`` (PLACEMENT_DTYPE host array, 1..64 entries), ``n_weights`` (1 .. 2^28) and ``weights``, the
    float32 (n_weights,) device tensor: zeros, or a copy of the given finite values.  The placements are checked as
    the C entry points check them, before anything touches a device."""

    def __init__(self, placements, n_weights: int, weights=None, device=None):
        self.placements = check_placements(placements, n_weights)
        self.n_weights = int(n_weights)
        if weights is not None:
            weights = _check_weights(weights, self.n_weights)
        device = N.require_cuda() if device is None else torch.device(device)
        if weights is None:
            self.weights = torch.zeros(self.n_weights, dtype=torch.float32, device=device)
        else:
            self.weights = weights.to(device).clone()

    @property
    def n_placements(self) -> int:
        return int(self.placements.shape[0])

    @classmethod
    def from_tuples(cls, tuples, symmetric: bool = True, weights=None, device=None) -> "NTupleNetwork":
        """One table per tuple, packed in order (offset of table j = sum of 16^k over the tuples before it); with
        ``symmetric`` each tuple is placed 8 times, once per symmetry (tuple-major), all sharing its table."""
        rows, offset = [], 0
        for cells in tuples:
            cells = tuple(int(c) for c in cells)
            if not 1 <= len(cells) <= 6 or any(not 0 <= c < 16 for c in cells):
                raise ValueError(f"a tuple has 1..6 cells in 0..15, got {cells}")
            images = symmetric_images(cells) if symmetric else [cells]
            rows += [(offset, im) for im in images]
            offset += 16 ** len(cells)
        if not 1 <= len(rows) <= MAX_PLACEMENTS:
            raise ValueError(f"a network has 1..64 placements, got {len(rows)}")
        return cls(make_placements(rows), offset, weights, device)

    @classmethod
    def four_six(cls, weights=None, device=None) -> "NTupleNetwork":
        """The 4x6 network: the 6-cell shapes of FOUR_SIX_TUPLES under the 8 symmetries, table j at j * 2^24."""
        return cls.from_tuples(FOUR_SIX_TUPLES, True, weights, device)

    @classmethod
    def lines(cls, weights=None, device=None) -> "NTupleNetwork":
        """One 65 536-entry table over the 4 rows, then the 4 columns: V is the row heuristic H of the same table."""
        rows = [(0, (4 * r, 4 * r + 1, 4 * r + 2, 4 * r + 3)) for r in range(4)]
        rows += [(0, (c, c + 4, c + 8, c + 12)) for c in range(4)]
        return cls(make_placements(rows), 65536, weights, device)

    def weights_on(self, device) -> torch.Tensor:
        return self.weights.to(device=device, dtype=torch.float32).contiguous()
