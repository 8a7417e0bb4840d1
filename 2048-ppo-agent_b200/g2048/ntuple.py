"""N-tuple networks: the value function of the strong learned 2048 players (Szubert & Jaśkowski 2014; Yeh et al. 2016).

    net = g2048.NTupleNetwork.four_six()                     # 4 six-cell tuples x 8 symmetries, 2^26 weights
    learner = g2048.NTupleTDLearner(0, batch_size=1 << 16, network=net)
    learner.train(4000)
    player = g2048.ExpectimaxPolicy(depth=1, network=net, reward_weight=1.0)

A network is an ordered list of placements over one flat float32 weight array ``W``.  Placement p reads k cells of the
board and indexes its table with their exponents (nibble j = the exponent in cells[j]):
``V(b) = W[off_0 + idx_0(b)] + ... + W[off_{P-1} + idx_{P-1}(b)]`` in float32, left to right (include/g2048.h).
Placements with the same offset share a table: the 8 symmetric images of a tuple learn one set of weights.

A multi-stage network (Yeh et al. 2016; Jaśkowski 2018) splits the game into S stages by the largest tile on the board,
and gives each stage its own copy of every table, ``stage_stride`` entries after the previous stage's:
``stage(b)`` is the number of ``stage_thresholds`` (tile exponents) that the board's largest exponent reaches, and
``V_S(b) = W[stage(b) * stride + off_0 + idx_0(b)] + ...``.  ``NTupleNetwork.staged(net, (13,))`` splits a trained
single-stage network into stages that start as copies of it.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native as N

# G2048TuplePlacement (include/g2048.h), 12 bytes
PLACEMENT_DTYPE = np.dtype([("offset", "<u4"), ("n_cells", "u1"), ("cells", "u1", (6,)), ("reserved", "u1")])
MAX_PLACEMENTS = 64
MAX_WEIGHTS = 1 << 28
# G2048TupleStages (include/g2048.h), 20 bytes
STAGES_DTYPE = np.dtype([("stride", "<u4"), ("n_thresholds", "u1"), ("thresholds", "u1", (15,))])
MAX_STAGES = 16
# G2048_NTUPLE_MAX_HORIZON (include/g2048.h): the longest window of the TD(lambda) / TC(lambda) learners
MAX_HORIZON = 8

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


def make_stages(thresholds, stride: int) -> np.ndarray:
    """A (1,) STAGES_DTYPE array (a G2048TupleStages) from tile exponents and a stride, unchecked."""
    thresholds = [int(t) for t in thresholds]
    if len(thresholds) > MAX_STAGES - 1 or any(not 0 <= t < 256 for t in thresholds) or not 0 <= int(stride) < 1 << 32:
        raise ValueError(f"stages have at most 15 thresholds in 1..15 and a uint32 stride, got {thresholds}, {stride}")
    st = np.zeros(1, STAGES_DTYPE)
    st[0]["stride"] = int(stride)
    st[0]["n_thresholds"] = len(thresholds)
    st[0]["thresholds"][: len(thresholds)] = thresholds
    return st


def check_stages(stages, placements, n_weights: int) -> np.ndarray:
    """The stage checks of the staged C entry points (include/g2048.h), for a network that check_placements accepts: a
    C-contiguous (1,) STAGES_DTYPE copy, or ValueError."""
    st = np.ascontiguousarray(np.asarray(stages)).reshape(-1)
    if st.dtype != STAGES_DTYPE or st.shape[0] != 1:
        raise ValueError("stages must be one STAGES_DTYPE record")
    k, stride = int(st[0]["n_thresholds"]), int(st[0]["stride"])
    thresholds = [int(t) for t in st[0]["thresholds"]]
    if k > MAX_STAGES - 1:
        raise ValueError(f"a network has at most 15 stage thresholds, got {k}")
    if any(not 1 <= t <= 15 for t in thresholds[:k]) or any(a >= b for a, b in zip(thresholds[:k], thresholds[1:k])):
        raise ValueError(f"stage thresholds must be strictly increasing tile exponents in 1..15, got {thresholds[:k]}")
    if any(thresholds[k:]):
        raise ValueError("unused stage threshold bytes must be 0")
    if (k == 0) != (stride == 0):
        raise ValueError(f"the stage stride must be 0 exactly for a single-stage network, got {stride} with {k + 1} stages")
    pl = np.asarray(placements)
    for i, p in enumerate(pl):
        if k * stride + int(p["offset"]) + 16 ** int(p["n_cells"]) > int(n_weights):
            raise ValueError(f"placement {i}: its table in the last stage exceeds n_weights = {n_weights}")
    return st.copy()


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
    float32 (n_weights,) device tensor: zeros, or a copy of the given finite values.  ``stage_thresholds`` (strictly
    increasing tile exponents in 1..15, at most 15) and ``stage_stride`` (0 exactly when there are none) make it a
    network of ``n_stages = len(stage_thresholds) + 1`` stages.  The placements and stages are checked as the C entry
    points check them, before anything touches a device."""

    def __init__(self, placements, n_weights: int, weights=None, device=None, stage_thresholds=(), stage_stride: int = 0):
        self.placements = check_placements(placements, n_weights)
        self.n_weights = int(n_weights)
        self._stages = check_stages(make_stages(stage_thresholds, stage_stride), self.placements, self.n_weights)
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

    @property
    def stage_thresholds(self) -> tuple[int, ...]:
        return tuple(int(t) for t in self._stages[0]["thresholds"][: self._stages[0]["n_thresholds"]])

    @property
    def stage_stride(self) -> int:
        return int(self._stages[0]["stride"])

    @property
    def n_stages(self) -> int:
        return len(self.stage_thresholds) + 1

    @property
    def stages(self) -> np.ndarray | None:
        """The G2048TupleStages record of the staged entry points, or None for a single-stage network, which takes the
        unstaged ones."""
        return self._stages if self.n_stages > 1 else None

    @classmethod
    def staged(cls, base: "NTupleNetwork", thresholds) -> "NTupleNetwork":
        """``base`` split into ``len(thresholds) + 1`` stages at these tile exponents: its placements, stride =
        ``base.n_weights``, and every stage starting as a copy of ``base.weights`` (whole-stage promotion), so that the
        new network has exactly ``base``'s values until it learns.  ``base`` must have one stage."""
        if not isinstance(base, NTupleNetwork) or base.n_stages != 1:
            raise ValueError("staged() splits a single-stage NTupleNetwork")
        thresholds = tuple(int(t) for t in thresholds)
        n_stages = len(thresholds) + 1
        n_weights = n_stages * base.n_weights
        stride = base.n_weights if n_stages > 1 else 0
        if n_weights > MAX_WEIGHTS:
            raise ValueError(f"{n_stages} stages of {base.n_weights} weights exceed 2^28 weights")
        check_stages(make_stages(thresholds, stride), base.placements, n_weights)  # before the copy touches a device
        return cls(base.placements, n_weights, base.weights.repeat(n_stages), base.weights.device, thresholds, stride)

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
