"""The numpy twin of the median residual stage (oracle/restate.py: residual_mask_lattice) on the adversarial inputs of
tests/rank_families.py: its mask equals cv2's absdiff(g, medianBlur(g, 21)) > thr, the list entries it predicts equal
a pixel-by-pixel reading of the kernel's thresholds (vi_rank.cuh: rank_code_thresholds, rank_dirty_cell), and the
families reach the counts where a bracket or an exact count flips.  The model of the kernel's level choice
(select_levels) equals a direct reading of its rule.  CPU only."""
import numpy as np
import pytest

from oracle import restate as S
import rank_families as F

SHAPES = [(1, 1), (2, 5), (4, 22), (23, 33), (25, 31), (47, 35), (22, 77)]


def brute_entries(gray, thr, levels, roi):
    """Per ROI pixel: its cell's bracket from the exact window counts at the cell centre, the four byte thresholds
    as the kernel clamps them, one entry per open test of a pixel that is neither defect nor clean for sure."""
    h, w = gray.shape
    p = np.pad(gray, 13, mode='edge').astype(np.int32)
    n = 0
    for y, x in zip(*np.nonzero(roi)):
        cy, cx = 3 * (y // 3) + 1, 3 * (x // 3) + 1
        win = p[cy + 3:cy + 24, cx + 3:cx + 24]
        cnt = [int((win <= v).sum()) for v in levels]
        n179, n263 = sum(c >= 179 for c in cnt), sum(c >= 263 for c in cnt)
        LO = levels[3 - n179 - 1] if n179 < 3 else -1
        HI = levels[3 - n263] if n263 > 0 else 255
        u1, u4 = min(max(LO - thr + 1, 0), 255), min(HI + thr, 255)
        u2, u3 = max(HI - thr, 0), min(LO + thr + 1, 255)
        g = int(gray[y, x])
        if u1 <= g <= u4:
            n += (g < u2) + (g > u3)
    return n


def cases(seed, shapes=SHAPES, thrs=F.THRS):
    rng = np.random.default_rng(seed)
    for (h, w) in shapes:
        for name, img in F.IMAGES.items():
            thr = int(rng.choice(thrs))
            g = img(rng, h, w, thr)
            for lname, lv in F.level_sets(rng, g, thr).items():
                rname = list(F.ROIS)[int(rng.integers(0, len(F.ROIS)))]
                yield (h, w, name, thr, lname, rname), g, thr, sorted(lv), F.ROIS[rname](rng, h, w)


def test_twin_equals_cv2_and_entries_equal_a_brute_count():
    for key, g, thr, lv, roi in cases(1):
        st = {}
        got = S.residual_mask_lattice(g, thr, lv, roi=roi, stats=st) & roi
        assert np.array_equal(got, F.reference(g, thr, roi)), key
        assert st['entries'] == brute_entries(g, thr, lv, roi), key
        assert st['entries'] == len(st['pivot_counts']), key


def test_families_reach_the_boundaries():
    """Some cell centres count exactly 178 / 179 / 262 / 263 at a level, some exact counts land on 220 / 221 at a pivot,
    and every bracket code with n263 <= n179 occurs on a dirty ROI cell."""
    centre, pivot = set(), set()
    codes = np.zeros(16, np.int64)
    blocks_on_end = 0
    for key, g, thr, lv, roi in cases(2, shapes=[(23, 33), (47, 35), (31, 64)], thrs=(0, 1, 2, 7, 24, 60)):
        st = {}
        S.residual_mask_lattice(g, thr, lv, roi=roi, stats=st)
        centre |= set(np.unique(st['centre_counts']).tolist())
        pivot |= set(st['pivot_counts'].tolist())
        codes += st['codes']
    for key, g, thr, lv, roi in cases(3, shapes=[(33, 45)], thrs=(2, 7, 24)):
        if key[2] != 'blocks3' or key[4] != 'select':
            continue
        st = {}
        S.residual_mask_lattice(g, thr, lv, stats=st)
        C = st['centre_counts']
        LO = np.array([-1] + lv)[3 - (C >= 179).sum(0)]
        HI = np.array(lv + [255])[3 - (C >= 263).sum(0)]
        cg = g[:33, :45].astype(np.int32).reshape(11, 3, 15, 3)
        blocks_on_end += int(((cg.min(axis=(1, 3)) == HI - thr) | (cg.max(axis=(1, 3)) == LO + thr + 1)).sum())
    assert {178, 179, 262, 263} <= centre, sorted(centre & set(range(170, 270)))
    assert {220, 221} <= pivot
    reachable = [n179 * 4 + n263 for n179 in range(4) for n263 in range(n179 + 1)]
    assert all(codes[c] > 0 for c in reachable), codes
    assert all(codes[c] == 0 for c in range(16) if c not in reachable), codes
    assert blocks_on_end > 0


@pytest.mark.parametrize("bright", [False, True])
def test_select_levels_model_reads_the_kernel_rule(bright):
    """The lower median of the class (the ceil(n / 2)-th smallest pixel of it), then [m - s, m, m + s] with s the
    largest power of two <= thr / 3 (at least 1, at most 16), clamped to 0..254; an empty class centres on t."""
    rng = np.random.default_rng(5 + bright)
    for _ in range(400):
        n = int(rng.integers(1, 3000))
        pix = np.clip(rng.normal(rng.uniform(0, 255), rng.uniform(1, 80), n), 0, 255).astype(np.int64)
        if rng.random() < 0.2:
            pix[:] = int(rng.integers(0, 256))
        t, thr = int(rng.integers(0, 256)), int(rng.integers(0, 256))
        cls = np.sort(pix[pix > t] if bright else pix[pix <= t])
        m = int(cls[(len(cls) + 1) // 2 - 1]) if len(cls) else t
        s = min(16, 1 << (max(thr // 3, 1).bit_length() - 1))
        want = [min(254, max(0, m + d)) for d in (-s, 0, s)]
        assert S.select_levels(np.bincount(pix, minlength=256), t, thr, bright) == want, (n, t, thr)
