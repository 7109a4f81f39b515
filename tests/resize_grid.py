"""A designed grid of cv2.resize geometries and source data, shared by the CPU test of the resize restatement
(tests/test_resize_cv2.py) and the device test of the resize kernels (tests/test_resize_gpu.py).

Each geometry class is a list of (sw, sh, dw, dh); each data kind makes a float32 (sh, sw) source from a seed."""
import numpy as np

from oracle import preprocess_oracle as po

FRAME_SIZES = (8, 24, 32, 48, 64)


def _pairs(seed, n, lo, hi):
    rng = np.random.default_rng(seed)
    return [(int(a), int(b)) for a, b in rng.integers(lo, hi, size=(n, 2))]


def _aspect():
    # aspect-preserving targets as resize_and_pad computes them, from sources of 1..100 on each side
    srcs = [(1, 1), (1, 100), (100, 1), (2, 3), (41, 1), (100, 100), (99, 37)] + _pairs(11, 24, 1, 101)
    return [(sw, sh) + po.resized_size(sw, sh, (s, s)) for s in FRAME_SIZES for sw, sh in srcs]


def _thin():
    out = [(1, 1, 64, 64), (1, 1, 1, 7), (1, 1, 9, 1), (1, 1, 3, 2)]
    for k in (2, 3, 5, 17, 41, 64, 100):
        for d in (1, 2, k // 2 + 1, k + 1, 3 * k, 64):
            out += [(k, 1, d, 1), (1, k, 1, d), (k, 1, d, 5), (1, k, 5, d), (k, 1, 2, d), (1, k, d, 2)]
    return sorted(set(out))


def _integer_scales():
    out = []
    for k in (2, 3, 4):  # downscales by k on both sides, on one side, and mixed
        for dw, dh in [(1, 1), (3, 5), (16, 16), (31, 7)]:
            out += [(dw * k, dh * k, dw, dh), (dw * k, dh, dw, dh), (dw * k, dh * 2, dw, dh)]
    for k in (2, 3, 4, 5, 8):  # upscales
        for sw, sh in [(2, 2), (3, 7), (16, 9), (2, 11)]:
            out += [(sw, sh, sw * k, sh * k), (sw, sh, sw * k, sh)]
    return out


def _integer_landing():
    # (d + 0.5) * sn / dn - 0.5 is an integer k when sn / dn = (2k + 1) / (2d + 1): sn = (2k + 1) m, dn = (2d + 1) m.
    # In double, 1 / (dn / sn) misses such a coordinate by an ULP on either side; cv2 (IPP) lands on it.
    out = []
    for k, d, m in [(1, 8, 2), (31, 47, 1), (13, 7, 3), (6, 2, 3), (10, 12, 2), (2, 9, 5), (0, 3, 4), (25, 12, 1), (4, 4, 3)]:
        sn, dn = (2 * k + 1) * m, (2 * d + 1) * m
        if sn == dn:
            continue
        out += [(sn, 7, dn, 11), (7, sn, 11, dn), (sn, sn + 1, dn, dn), (sn, 1, dn, 3), (1, sn, 3, dn)]
    return out


GEOMETRIES = {
    "identity": [(1, 1, 1, 1), (1, 9, 1, 9), (9, 1, 9, 1), (7, 5, 7, 5), (64, 64, 64, 64), (100, 3, 100, 3)],
    "one_side_unchanged": [(sw, sh, sw, dh) for sw, sh, dh in [(7, 5, 9), (33, 64, 32), (2, 40, 41), (64, 3, 1)]]
    + [(sw, sh, dw, sh) for sw, sh, dw in [(7, 5, 9), (64, 33, 32), (40, 2, 41), (3, 64, 1)]],
    "aspect_preserving": _aspect(),
    "thin": _thin(),
    "free": [(sw, sh, dw, dh) for (sw, sh), (dw, dh) in zip(_pairs(12, 60, 1, 100), _pairs(13, 60, 1, 100))],
    "integer_scale": _integer_scales(),
    "integer_landing": _integer_landing(),
}


def make_source(kind, sh, sw, seed):
    rng = np.random.default_rng(seed)
    if kind == "u16":
        return rng.integers(0, 65536, size=(sh, sw)).astype(np.float32)
    if kind == "negative":
        return rng.integers(-300, 301, size=(sh, sw)).astype(np.float32)
    if kind == "half":
        return (rng.integers(-4000, 4001, size=(sh, sw)) * 0.5).astype(np.float32)
    if kind == "real":
        return (rng.standard_normal((sh, sw)) * rng.choice([1.0, 37.0, 3000.0])).astype(np.float32)
    if kind == "constant":
        return np.full((sh, sw), np.float32(rng.standard_normal() * 100.0), np.float32)
    if kind == "signed_zero":
        return rng.choice(np.float32([0.0, -0.0]), size=(sh, sw))
    raise ValueError(kind)


DATA = ("u16", "negative", "half", "real", "constant", "signed_zero")


def cases(geometry, kind):
    """(sw, sh, dw, dh, src) for every geometry of a class, each with its own seeded source."""
    for i, (sw, sh, dw, dh) in enumerate(GEOMETRIES[geometry]):
        yield sw, sh, dw, dh, make_source(kind, sh, sw, seed=(list(GEOMETRIES).index(geometry), DATA.index(kind), i))


def same_bits(a, b):
    """Bitwise equality of two float32 arrays: -0.0 and 0.0 differ."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype == np.float32 and np.array_equal(a.view(np.uint32), b.view(np.uint32))
