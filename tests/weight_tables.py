"""Edge-weight tables other than the reference's beta = 0.4, and level inputs that reach every part of them (no GPU needed).

rtdd_load_weights(ctx, beta) fills w[i] = expf(-beta * i), i = 0..255, and w[256] = 0.  Every solve reads its weights, and
the sweeps' exact division depends on the range of a free pixel's weight sum ((w_l + w_r) + w_u) + w_d:
- div_fast needs sums in [2^-100, 8]; sums below 2^-100 go through the per-pixel fallbacks (div_rare, badDen);
- the resident kernel rescales sums below 2^-21 by a power of two (pow2_scale);
- a sum of exactly +0 (all four links at zero weights) makes the oracle's result 0 (`count == 0`), and the kernels' 0 / 0.
Which of these occur depends on beta: the grid below names one regime per value and claims the index ranges of its
normal, denormal and zero entries; tests/test_weight_tables_cpu.py checks each claim against oracle.binding.load_weights."""
import numpy as np

from oracle import binding as ob
from tests.test_gpu_parity import enclosed_zero_level, random_level

# (beta, regime, claimed index ranges [lo, hi) of the normal, denormal and zero entries among w[0..255]; None = no such entry).
# Every table has w[0] = 1; beta = 0 and -0.0 give all ones.  (A list: as dict keys 0.0 and -0.0 would be one entry.)
GRID = [
    (0.0, "all ones", (0, 256), None, None),
    (0.05, "all normal", (0, 256), None, None),
    (0.35, "denormal tail, no zeros", (0, 250), (250, 256), None),
    (0.4, "the reference's table", (0, 219), (219, 256), None),
    (0.45, "denormals and zeros", (0, 195), (195, 232), (232, 256)),
    (1.0, "zeros from 104", (0, 88), (88, 104), (104, 256)),
    (8.0, "mostly zero", (0, 11), (11, 13), (13, 256)),
    (1e4, "only w[0]", (0, 1), None, (1, 256)),
    (-0.0, "all ones, negative zero", (0, 256), None, None),
]
BETAS = [g[0] for g in GRID]

TWO_M100 = np.float32(2.0 ** -100)     # lower end of div_fast's proven denominator range
TWO_M21 = np.float32(2.0 ** -21)       # pow2_scale rescales sums below this
FLT_MIN = np.float32(2.0 ** -126)      # smallest normal float


def beta_id(beta):
    return "beta=%r" % beta


def table(beta):
    """The oracle's 257-entry table (host expf in fp32, like rtdd_load_weights)."""
    return ob.load_weights(beta)


def entry_classes(lut):
    """Index sets of w[0..255]: (normal, denormal, zero)."""
    w = lut[:256]
    zero = np.flatnonzero(w == 0)
    den = np.flatnonzero((w > 0) & (w < FLT_MIN))
    normal = np.flatnonzero(w >= FLT_MIN)
    return normal, den, zero


def salt_and_pepper_level(rows, cols, seed):
    """The input of test_salt_and_pepper_image_tiny_weight_sums (tests/test_gpu_parity.py), same generator calls: a grey plane
    with 3 % salt (255), 3 % pepper (0) and a 4x4 checkerboard at (10, 10), so isolated pixels sit across 127+ grey-level edges."""
    rng = np.random.default_rng(seed)
    gray = np.full((rows, cols), 128, np.uint8)
    gray[rng.random((rows, cols)) < 0.03] = 255
    gray[rng.random((rows, cols)) < 0.03] = 0
    board = np.array([[0, 255, 0, 255], [255, 0, 255, 0], [0, 255, 0, 255], [255, 0, 255, 0]], np.uint8)
    gray[10:14, 10:14] = board[:max(rows - 10, 0), :max(cols - 10, 0)]
    depth = rng.uniform(0, 255, (rows, cols)).astype(np.float32)
    depth[20:30, 20:60] = 0.0
    scribble = np.where(rng.random((rows, cols)) < 0.05, 255, 0).astype(np.uint8)
    return gray, depth, scribble


def gray_steps_level(rows, cols, seed):
    """Gray plane whose link indices cover the table's tail.  Left half: a checkerboard of 0 and v = (x + 3y) mod 256, so every
    pixel at v sees index v on all four links (weight sum 4 w[v], rounded) and every v in 0..255 occurs once cols + 3 rows >= 256.
    Right half: 0/255 blocks 3 wide and 5 high, so links carry index 0 inside a block and 255 across its edges.  Depths are
    uniform in [0, 255) so that the depth-gated levels keep most gray indices; 5 % of the pixels are scribbles."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:rows, 0:cols]
    gray = np.where((x + y) % 2 == 1, (x + 3 * y) % 256, 0)
    half = cols // 2
    gray[:, half:] = np.where(((x[:, half:] // 3) + (y[:, half:] // 5)) % 2 == 0, 0, 255)
    depth = rng.uniform(0, 255, (rows, cols)).astype(np.float32)
    scribble = np.where(rng.random((rows, cols)) < 0.05, 255, 0).astype(np.uint8)
    return gray.astype(np.uint8), depth, scribble


INPUTS = {
    "random": lambda rows, cols, seed: random_level(rows, cols, seed),
    "salt-and-pepper": salt_and_pepper_level,
    "enclosed-zero": enclosed_zero_level,
    "gray-steps": gray_steps_level,
}


# The level solves of tests/test_gpu_weight_tables.py: (level shape, level, levels).  Level 0 of 2 is depth-gated with threshold
# 0, level 1 of 3 with threshold 4, level 1 of 2 is the ungated coarsest level.
LEVEL_CASES = [((135, 241), 0, 2), ((67, 121), 1, 3), ((33, 61), 1, 2)]


def level_input(kind, rows, cols, level):
    return INPUTS[kind](rows, cols, 1000 + rows + cols + level)


def weight_sums(gray, depth, scribble, level, max_level, lut):
    """Each free pixel's weight sum in the oracle's order ((w_l + w_r) + w_u) + w_d in fp32 (a missing neighbour adds w[256] = 0,
    which changes no sum); -> (sums [rows, cols] float32, free mask)."""
    idx = ob.index_to_weight(gray, depth, level, max_level)
    w = lut[idx]                                   # [rows, cols, 4] float32
    s = (w[..., 0] + w[..., 1]) + w[..., 2]
    s = s + w[..., 3]
    assert s.dtype == np.float32
    return s, scribble != 255


def table_allows(lut, bound):
    """Whether four copies of the smallest non-zero weight sum to below `bound`: a sum in (0, bound) is possible."""
    w = lut[:256]
    nz = w[w > 0]
    return bool(len(nz)) and float(4 * np.float64(nz.min())) < float(bound)
