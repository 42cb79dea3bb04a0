"""CPU test of the segmentation kernel's staging alias (vi_device.cuh: unit_layout, vi_unit.cuh: process_unit with SEG):
it gathers the next unit's crop into the staging area from the first close pass on, while the remaining close / open
passes, the hole fill, the centroid labelling, the exclusions and the stores use MB, MC and the workspace (run table,
row scan).  The staging area must lie inside gray and MA and clear of all of those, on every shared-memory layout."""
import pytest

from test_unit_layout import GRIDS, layouts  # noqa: F401  (the compiled layout driver, a module fixture)

LIVE_AFTER_FIRST_CLOSE = ('MB', 'MC', 'ws', 'runs')


@pytest.mark.parametrize('name', sorted(GRIDS))
def test_seg_stage_is_clear_of_the_live_masks(layouts, name):  # noqa: F811
    L = layouts[name]
    assert L['ok']
    if L['arena']:
        pytest.skip('the arena kernel has no asynchronous gather')
    regions = {r[0]: r[1:] for r in L['regions']}
    _, s_off, s_len = regions['stage']
    _, g_off, _ = regions['gray']
    _, ma_off, ma_len = regions['MA']
    assert g_off == s_off == 0 and s_len <= ma_off + ma_len
    for r in LIVE_AFTER_FIRST_CLOSE:
        _, off, size = regions[r]
        assert size == 0 or off >= s_off + s_len, (name, r)
