"""Adversarial 256-bin histograms for the Otsu threshold (oracle/restate.py: otsu_from_hists, otsu_kernel_model;
tests/test_gpu_otsu.py).  Every generator takes a numpy Generator, a count k and optionally a pixel count n, and
returns k histograms as an int64 array [k, 256] whose row sums lie in 1..2^24 (a unit's pixel count), all equal to n
when it is given (n >= 16).

The pixel counts are drawn log-uniformly over 1..2^24, densely around 2^23 (FLT_EPSILON = 2^-23: above it a class of
one pixel is below FLT_EPSILON of the unit, and OpenCV's scan skips that split) and at 2^24."""
import numpy as np

NMAX = 1 << 24


def pixel_counts(rng, k, lo=1, n=None):
    if n is not None:
        return np.full(k, n, np.int64)
    u = rng.random(k)
    n = np.exp(rng.uniform(np.log(lo), np.log(NMAX), k)).astype(np.int64)
    near = (1 << 23) + rng.integers(-2048, 2049, k)
    wide = (1 << 23) + rng.integers(-(1 << 21), (1 << 21) + 1, k)
    top = NMAX - rng.integers(0, 64, k)
    n = np.where(u < 0.4, n, np.where(u < 0.65, near, np.where(u < 0.8, wide, np.where(u < 0.9, top, NMAX))))
    return np.clip(n, lo, NMAX)


def log_split(rng, n):
    """m in 1..n-1, log-uniform, and mirrored half the time (n >= 2)."""
    m = np.exp(rng.uniform(0, np.log(np.maximum(n - 1, 1)))).astype(np.int64)
    m = np.clip(m, 1, n - 1)
    return np.where(rng.random(len(n)) < 0.5, m, n - m)


def two_spikes(rng, k, n=None):
    """m pixels at a, n - m at b > a: every split between a and b has the same variance (an exact tie)."""
    n = pixel_counts(rng, k, 2, n)
    a = rng.integers(0, 255, k)
    b = a + 1 + (rng.integers(0, 256, k) % (255 - a))
    m = log_split(rng, n)
    H = np.zeros((k, 256), np.int64)
    r = np.arange(k)
    H[r, a] += m
    H[r, b] += n - m
    return H


def spikes(rng, k, n=None):
    """3 to 5 spikes at random bins, random weights (a spike may come out empty)."""
    n = pixel_counts(rng, k, 1, n)
    H = np.zeros((k, 256), np.int64)
    for j in range(k):
        s = rng.integers(3, 6)
        bins = rng.choice(256, s, replace=False)
        H[j, bins] = rng.multinomial(n[j], rng.dirichlet(np.full(s, 0.7)))
    return H


def bimodal(rng, k, n=None):
    """Two Gaussian modes; a third of them mirror-symmetric about 127.5 (then their split at 127 ties its mirror)."""
    n = pixel_counts(rng, k, 1, n)
    x = np.arange(256)
    H = np.zeros((k, 256), np.int64)
    for j in range(k):
        m1, m2 = np.sort(rng.uniform(0, 255, 2))
        s1, s2 = rng.uniform(0.3, 40, 2)
        if j % 3 == 0:
            m2, s2 = 255 - m1, s1
            p = np.exp(-0.5 * ((x - m1) / s1) ** 2) + np.exp(-0.5 * ((x - m2) / s2) ** 2)
            half = np.floor(p / p.sum() * (n[j] // 2)).astype(np.int64)
            h = half + half[::-1]
            r, b = n[j] - h.sum(), int(m1)                     # the rest at the mode and its mirror (one apart if odd)
            h[b] += r // 2
            h[255 - b] += r - r // 2
            H[j] = h
        else:
            w = rng.uniform(0.02, 0.98)
            p = w * np.exp(-0.5 * ((x - m1) / s1) ** 2) / s1 + (1 - w) * np.exp(-0.5 * ((x - m2) / s2) ** 2) / s2
            H[j] = rng.multinomial(n[j], p / p.sum())
    return H


def sparse(rng, k, n=None):
    """2 to 12 occupied bins anywhere, some with a single pixel."""
    n = pixel_counts(rng, k, 1, n)
    H = np.zeros((k, 256), np.int64)
    for j in range(k):
        s = rng.integers(2, 13)
        bins = rng.choice(256, s, replace=False)
        c = rng.multinomial(n[j], rng.dirichlet(np.full(s, 0.3)))
        one = (rng.random(s) < 0.3) & (c > 1)
        top = np.argmax(c)
        one[top] = False
        c[top] += (c[one] - 1).sum()
        c[one] = 1
        H[j, bins] = c
    return H


def edge_mass(rng, k, n=None):
    """All pixels in bin 0 or 255, or all but a few of them there and the rest anywhere."""
    n = pixel_counts(rng, k, 1, n)
    H = np.zeros((k, 256), np.int64)
    edge = np.where(rng.random(k) < 0.5, 0, 255)
    r = np.where(rng.random(k) < 0.5, 0, rng.integers(1, 4, k))
    r = np.minimum(r, n - 1)
    H[np.arange(k), edge] = n - r
    for j in np.nonzero(r)[0]:
        H[j, rng.integers(0, 256, r[j])] += 1
    return H


def single_bin(rng, k, n=None):
    n = pixel_counts(rng, k, 1, n)
    H = np.zeros((k, 256), np.int64)
    H[np.arange(k), rng.integers(0, 256, k)] = n
    return H


def moment_bound(rng, k, n=NMAX):
    """Nearly all at 255, N = 2^24 unless given: the 32-bit moment sum i * h_i is close to 2^32."""
    H = np.zeros((k, 256), np.int64)
    for j in range(k):
        r = min(int(np.exp(rng.uniform(0, np.log(1 << 20)))), n // 2)
        s = rng.integers(1, 6)
        bins = rng.choice(255, s, replace=False)
        H[j, bins] = rng.multinomial(r, np.full(s, 1.0 / s))
        H[j, 255] = n - r
    return H


def trigger(rng, k, n=None):
    """1 pixel at x0, m at a > x0, the rest at a + gap (gap 1..5, m log-uniform): above 2^23 pixels the lone dark
    pixel's split is one the reference skips, and its float32 variance is the largest."""
    n = pixel_counts(rng, k, 8, n)
    gap = rng.integers(1, 6, k)
    a = rng.integers(1, 256 - gap, k)
    x0 = (rng.integers(0, 256, k) % a)
    m = np.clip(np.exp(rng.uniform(0, np.log(n - 2))).astype(np.int64), 1, n - 2)
    H = np.zeros((k, 256), np.int64)
    r = np.arange(k)
    H[r, x0] += 1
    H[r, a] += m
    H[r, a + gap] += n - 1 - m
    return H


def trigger_mirror(rng, k, n=None):
    """The trigger family reflected: the lone pixel at the bright end."""
    return trigger(rng, k, n)[:, ::-1].copy()


def lone_pixels(rng, k, n=None):
    """One mode with 1 to 4 lone pixels either side: the best splits cut off a tiny class at either end, and above
    2^23 pixels the darkest lone pixel is one the reference skips (and leaves out of its lower-class mean)."""
    n = pixel_counts(rng, k, 16, n)
    H = np.zeros((k, 256), np.int64)
    for j in range(k):
        a = rng.integers(2, 254)
        lo = rng.choice(a, min(rng.integers(1, 5), a), replace=False)
        hi = a + 1 + rng.choice(255 - a, min(rng.integers(1, 5), 255 - a), replace=False)
        H[j, lo] = 1
        H[j, hi] = 1
        H[j, a] = n[j] - len(lo) - len(hi)
    return H


FAMILIES = {f.__name__: f for f in (two_spikes, spikes, bimodal, sparse, edge_mass, single_bin, moment_bound,
                                    trigger, trigger_mirror, lone_pixels)}


def mixed(rng, k_per_family):
    """k_per_family histograms of every family, concatenated, and the family name of each row."""
    hs, names = [], []
    for name, f in FAMILIES.items():
        hs.append(f(rng, k_per_family))
        names += [name] * k_per_family
    return np.concatenate(hs), np.array(names)


def image_of(hist, rng, shape=None):
    """A uint8 image whose pixel multiset is the histogram, in random order."""
    px = np.repeat(np.arange(256, dtype=np.uint8), hist)
    rng.shuffle(px)
    return px.reshape(shape if shape is not None else (1, -1))
