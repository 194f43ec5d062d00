"""Integer-coded probes of the Stage-1 score path and their exact references (shared by tests/test_gpu_score_probes.py
and the CPU sensitivity test in tests/test_host_logic.py; numpy only, no GPU).

The score path has three indexing decisions that tolerances cannot see: the fc1 epilogue splits each warp's 32 rows at
the image boundary (gemm_tcgen05.cuh: `seg_split`) into two partial rows per 32-row sub-tile, the finisher
(kernels.cuh: score_norms_all_kernel) picks one of the two for every sub-tile of an image, and score_accumulate_kernel
adds the per-image norms in image order. A row counted in the neighbouring image moves that image's norm by about
1/(2T): 2.5e-3 at T = 197, 4.9e-4 at T = 1025.

Integer operands make every intermediate exact. Row r and column c get integer codes f(r), g(c), h(c):
a[r, 0] = f(r), a[r, 1] = 1, w[c, 0] = 1, w[c, 1] = g(c), bias[c] = h(c), every other K entry 0, so
z[r, c] = f(r) + g(c) + h(c) exactly (the MMA adds two integer products). Then
  * "pre" codes (scores taken before the activation): |z| <= 60, so bf16(z) = z and one image's sum of squares is at
    most 1025 * 3600 < 2^24: the squares, the partial sums in any order and the finisher's sums are exact in fp32;
  * "post" codes (scores of the stored erf-GELU activations): f, g, h in {0} U [6, 20], so z is in {0} U [6, 60], where
    gelu(z) = z - z q(z) with z q(z) < 1e-8, far below half an fp32 ulp of z: the stored activation is z itself.
The expected norm of (image, neuron) is float32(sqrt(exact int64 sum of z^2)): CUDA's sqrtf is correctly rounded (the
library is built without --use_fast_math), and rounding the double square root of an integer below 2^24 to fp32 gives
the same value (double rounding is innocuous for sqrt from 53 to 24 bits).

The codes are discriminating: f is nonzero on every row and differs between the rows on either side of every image
boundary and every 32/128/256-row edge, and g + h differs between the two columns of every lane pair. Moving, dropping
or double-counting one row, or swapping a lane's two columns, changes an integer sum; `emulate` reproduces the kernels'
indexing with switches for such faults, and the sensitivity test pins that each fault breaks bit equality.
"""
from __future__ import annotations

import numpy as np

# (T, images, N): every T where the boundary sits at a different place in the 32-row sub-tiles (multiples of 32, one
# past and one before them, the ViT / DeiT / CLIP / DINOv2 sequence lengths, two query tiles, 1025 = the longest),
# with image counts that leave M off the 32/128/256-row grids where T allows it, and widths of full and pruned fc1 layers
# (2040, 1000, 264 and 136 end in a partial 64-column chunk; 136 and 264 also in a partial 256-column tile).
PROBE_SHAPES = [
    (32, 5, 264), (33, 7, 136), (37, 9, 2040), (50, 5, 1000), (63, 3, 768), (64, 5, 264), (65, 3, 136),
    (127, 3, 1000), (128, 3, 136), (129, 3, 2040), (197, 3, 3072), (198, 3, 768), (201, 5, 264), (257, 3, 1000),
    (261, 3, 136), (577, 3, 2040), (1025, 3, 264),
]
# widths of the tile-count cases: one 256-column tile, so that the single-CTA tile count is ceil(M / 128)
SM_CASE_N = 136
SM_CASE_T = {"sms+1": 37, "2sms-1": 50, "2sms+1": 65}


def sm_case_images(tiles: int, T: int) -> int:
    """The image count whose M = n T needs exactly `tiles` 128-row tiles (T < 128 always has one)."""
    n = (128 * (tiles - 1)) // T + 1
    assert -(-n * T // 128) == tiles, (tiles, T)
    return n


def sm_cases(sms: int):
    """(name, T, images, N) of the three tile-count cases around the SM count."""
    tiles = {"sms+1": sms + 1, "2sms-1": 2 * sms - 1, "2sms+1": 2 * sms + 1}
    return [(k, SM_CASE_T[k], sm_case_images(tiles[k], SM_CASE_T[k]), SM_CASE_N) for k in tiles]


def _edges(M: int, T: int) -> np.ndarray:
    """Rows next to an image boundary or a 32/128/256-row edge: the last row before it and the first after it."""
    cuts = set(range(T, M, T)) | set(range(32, M, 32)) | {M}
    rows = set()
    for c in cuts:
        rows.update((c - 2, c - 1, c, c + 1))
    return np.array(sorted(r for r in rows if 0 <= r < M), dtype=np.int64)


def row_codes(M: int, T: int, kind: str, seed: int = 0) -> np.ndarray:
    """f(r), int64 [M]: pre codes in [-20, -1] U [1, 20], post codes in [6, 20]; pseudo-random, nonzero everywhere,
    and consecutive rows around every boundary and edge distinct."""
    rng = np.random.default_rng(seed * 7919 + M + 31 * T)
    vals = np.concatenate([np.arange(-20, 0), np.arange(1, 21)]) if kind == "pre" else np.arange(6, 21)
    f = rng.choice(vals, size=M)
    for r in _edges(M, T):
        if r > 0:
            while f[r] == f[r - 1] or (r >= 2 and f[r] == f[r - 2]):
                f[r] = rng.choice(vals)
    return f.astype(np.int64)


def col_codes(N: int, kind: str, seed: int = 0):
    """(g, h), int64 [N] each: pre codes in [-20, 20], post codes with g in {0} U [6, 20] and h in [6, 20] (so z >= 6
    everywhere); g + h differs between columns 2l and 2l + 1."""
    rng = np.random.default_rng(seed * 104729 + N)
    if kind == "pre":
        g, h = rng.integers(-20, 21, N), rng.integers(-20, 21, N)
        gv = np.arange(-20, 21)
    else:
        gv = np.concatenate([[0], np.arange(6, 21)])
        g, h = rng.choice(gv, N), rng.integers(6, 21, N)
    for c in range(1, N, 2):
        while g[c] + h[c] == g[c - 1] + h[c - 1]:
            g[c] = rng.choice(gv)
    return g.astype(np.int64), h.astype(np.int64)


def operands(f: np.ndarray, g: np.ndarray, h: np.ndarray, K: int):
    """(a [M, K], w [N, K], bias [N]) as float32 arrays with z = a @ w.T + bias = f[:, None] + g + h."""
    M, N = f.size, g.size
    a = np.zeros((M, K), np.float32)
    a[:, 0], a[:, 1] = f, 1
    w = np.zeros((N, K), np.float32)
    w[:, 0], w[:, 1] = 1, g
    return a, w, h.astype(np.float32)


def z_of(f, g, h) -> np.ndarray:
    return f[:, None] + (g + h)[None, :]


def image_sums(z: np.ndarray, T: int) -> np.ndarray:
    """Exact per-(image, neuron) sums of squares, int64 [n_img, N] (M = n_img T)."""
    n = z.shape[0] // T
    return (z.astype(np.int64) ** 2).reshape(n, T, -1).sum(1)


def norms_of(sums: np.ndarray) -> np.ndarray:
    assert int(sums.max(initial=0)) < 2 ** 24
    return np.sqrt(sums.astype(np.float32))


def accumulate(norms: np.ndarray, base: np.ndarray | None = None) -> np.ndarray:
    """scores += norms[0] + norms[1] + ... in fp32, one add at a time in image order (score_accumulate_kernel)."""
    acc = np.zeros(norms.shape[1], np.float32) if base is None else base.astype(np.float32).copy()
    for row in norms.astype(np.float32):
        acc = acc + row
    return acc


FAULTS = ("split+1", "split-1", "seg_from_last_row", "drop_last_tail_row", "swap_lane_pair", "slot1_inside_image")


def emulate(z: np.ndarray, T: int, M: int | None = None, fault: str | None = None):
    """The epilogue's partials [ceil(M/32)][2][N] and the finisher's norms [M / T][N], index for index as the kernels
    compute them (fp32 throughout; exact for the integer codes). `fault`, one of FAULTS:
      split+1 / split-1       seg_split = min(valid, (img0 + 1) T - row0 +- 1);
      seg_from_last_row       the finisher picks the slot from the sub-tile's last row, ((s << 5) + 31) / T;
      drop_last_tail_row      the last valid row of the M tail's partial sub-tile is not counted;
      swap_lane_pair          each lane writes its two columns (2l, 2l + 1) to each other's place;
      slot1_inside_image      the finisher reads slot 1 of a sub-tile that lies inside one image (where the epilogue
                              wrote 0)."""
    assert fault is None or fault in FAULTS, fault
    M = z.shape[0] if M is None else M
    N = z.shape[1]
    sq = z.astype(np.float32) ** 2
    subs = (M + 31) // 32
    partials = np.zeros((subs, 2, N), np.float32)
    for s in range(subs):
        row0 = 32 * s
        valid = min(32, max(0, M - row0))
        if fault == "drop_last_tail_row" and valid < 32:
            valid -= 1
        img0 = row0 // T
        d = {"split+1": 1, "split-1": -1}.get(fault, 0)
        seg_split = min(valid, (img0 + 1) * T - row0 + d)
        seg_end = valid
        partials[s, 0] = sq[row0:row0 + seg_split].sum(0)
        partials[s, 1] = sq[row0 + seg_split:row0 + seg_end].sum(0)
    if fault == "swap_lane_pair":
        partials = partials.reshape(subs, 2, N // 2, 2)[..., ::-1].reshape(subs, 2, N)
    n_img = M // T
    norms = np.zeros((n_img, N), np.float32)
    for img in range(n_img):
        r_begin, r_end = img * T, img * T + T
        acc = np.zeros(N, np.float32)
        for s in range(r_begin >> 5, ((r_end - 1) >> 5) + 1):
            first = ((s << 5) + 31) if fault == "seg_from_last_row" else (s << 5)
            seg = 0 if first // T == img else 1
            if fault == "slot1_inside_image" and (s << 5) // T == img and min((s << 5) + 31, M - 1) // T == img:
                seg = 1
            acc = acc + partials[s, seg]
        norms[img] = np.sqrt(acc)
    return partials, norms


def finisher_slots(n_img: int, T: int):
    """(sub-tile, slot) pairs the finisher reads for each image, in its order: [(img, s, seg), ...]."""
    out = []
    for img in range(n_img):
        for s in range((img * T) >> 5, ((img * T + T - 1) >> 5) + 1):
            out.append((img, s, 0 if (s << 5) // T == img else 1))
    return out


# ------------------------------------------------------------------------------------------------ bf16 rounding
def bf16_rne(x: np.ndarray) -> np.ndarray:
    """Round float64 values to the nearest bf16 (ties to even) in ONE rounding, returned as float64 (normal range)."""
    x = np.asarray(x, np.float64)
    m, e = np.frexp(x)
    scale = np.ldexp(1.0, 8 - e)
    return np.where(x == 0, 0.0, np.rint(x * scale) / scale)


def bf16_ulp(x: np.ndarray) -> np.ndarray:
    """The bf16 ulp at float64 values x (of the binade of |x|)."""
    _, e = np.frexp(np.asarray(x, np.float64))
    return np.ldexp(1.0, e - 8)


def gelu_erf64(x: np.ndarray) -> np.ndarray:
    from scipy.special import erf
    x = np.asarray(x, np.float64)
    return 0.5 * x * (1.0 + erf(x / np.sqrt(2.0)))


def quick_gelu64(x: np.ndarray) -> np.ndarray:
    from scipy.special import expit
    x = np.asarray(x, np.float64)
    return x * expit(1.702 * x)
