"""The vectorised Otsu scan (oracle/restate.py: otsu_from_hists) against the scalar one, and the CPU model of the
device's two-step Otsu (otsu_kernel_model) against both, on the adversarial histogram families of
tests/otsu_families.py.  The device stops the exact scan at the bound `last` of a float32 estimate
(vi_pipeline.cuh: otsu_approx_warp); these tests hold that bound to the reference's arg max.  CPU only."""
import numpy as np
import pytest

from oracle import restate as S
import otsu_families as F

# unit sizes of the arena kernel around and above 2^23 pixels, and controls at and below it
UNITS = [(4096, 2049), (4096, 3000), (4096, 4096), (2048, 8192), (4096, 2048), (2048, 2048)]


def test_vectorised_scan_equals_the_scalar_scan():
    rng = np.random.default_rng(11)
    H, _ = F.mixed(rng, 400)
    small = rng.multinomial(rng.integers(1, 5000), rng.dirichlet(np.full(256, 0.05)), size=400)
    H = np.concatenate([H, small])
    want = np.array([S.otsu_from_hist(h) for h in H])
    assert np.array_equal(S.otsu_from_hists(H), want)


@pytest.mark.parametrize("family", sorted(F.FAMILIES))
def test_scan_bound_holds_with_division_slack(family):
    """The reference's arg max lies at or before `last` even when every float32 variance is 1e-6 (relative) low and
    the maximum 1e-6 high (__fdividef and the float32 rounding of the kernel), and the scan stopped there gives the
    reference's threshold."""
    rng = np.random.default_rng(sorted(F.FAMILIES).index(family) + 20)
    H = F.FAMILIES[family](rng, 4000)
    ref = S.otsu_from_hists(H)
    t, last = S.otsu_kernel_model(H)
    _, last_slack = S.otsu_kernel_model(H, slack=1e-6)
    assert (last_slack <= last).all()
    bad = np.nonzero(last_slack < ref)[0]
    assert bad.size == 0, (family, H[bad[0]].sum(), np.nonzero(H[bad[0]])[0], ref[bad[0]], last_slack[bad[0]])
    assert np.array_equal(t, ref)


@pytest.mark.parametrize("wh", UNITS)
def test_lone_dark_pixel_at_unit_sizes(wh):
    """1 pixel at x0, m at a > x0 and the rest at a + gap (and the mirror) at the pixel counts of large units: above
    2^23 pixels the lone pixel's split is below FLT_EPSILON of the unit and the reference skips it."""
    n = wh[0] * wh[1]
    rng = np.random.default_rng(n % 1000)
    for H in (F.trigger(rng, 400, n), F.trigger_mirror(rng, 400, n)):
        ref = S.otsu_from_hists(H)
        t, last = S.otsu_kernel_model(H)
        assert (last >= ref).all() and np.array_equal(t, ref), wh


def test_skipped_lone_pixel_drops_its_moment_from_later_variances():
    """A lone darkest pixel at 15 that the reference skips (N > 2^23) is left out of its mu1 from then on: with a
    second and third lone pixel at 20 and 31, the exact variances peak at 31 but the reference's at 88."""
    h = np.zeros(256, np.int64)
    h[[15, 20, 31, 146, 189]] = 1
    h[88] = (1 << 23) + 100 - 5
    assert S.otsu_from_hist(h) == 88
    t, last = S.otsu_kernel_model(h[None])
    assert t[0] == 88 and last[0] >= 88


def test_issue_example_against_opencv():
    """N = 2^24: 1 pixel at 0, 30,000 at 200, the rest at 201.  OpenCV's C++ scan (IPP off) gives 200."""
    cv2 = pytest.importorskip("cv2")
    h = np.zeros(256, np.int64)
    h[0], h[200] = 1, 30000
    h[201] = (1 << 24) - 30001
    assert S.otsu_from_hist(h) == 200
    t, last = S.otsu_kernel_model(h[None])
    assert t[0] == 200 and last[0] >= 200
    im = F.image_of(h, np.random.default_rng(0), (4096, 4096))
    ipp = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    try:
        assert int(cv2.threshold(im, 0, 255, cv2.THRESH_BINARY_INV + cv2.THRESH_OTSU)[0]) == 200
    finally:
        cv2.ipp.setUseIPP(ipp)


def test_families_stay_in_range():
    rng = np.random.default_rng(3)
    H, names = F.mixed(rng, 500)
    n = H.sum(1)
    assert (H >= 0).all() and n.min() >= 1 and n.max() <= 1 << 24
    assert ((n > 1 << 23) & (n < 1 << 24)).sum() > 1000 and (n == 1 << 24).sum() > 100
