"""CPU test of the unit kernel's memory layout (vi_device.cuh: unit_layout): a host-only driver compiled with nvcc
prints the layout of a few grids; the values are pinned, and every region is checked for alignment, bounds and
overlaps against the alias table of vi_device.cuh."""
import json
import os
import subprocess

import pytest

from vi_b200 import _build

HERE = os.path.dirname(os.path.abspath(__file__))
OPTIN, STATIC = 232448, 1792      # B200: opt-in shared memory per block; the kernel's static shared memory

# name -> (units, f32 plane, blob_k)
GRIDS = {
    '316x315': (['316x315'], 0, 0),
    '96x96': (['96x96'], 0, 0),
    '150x230': (['150x230'], 0, 0),
    '640x480': (['640x480'], 0, 0),
    '4096x4096': (['4096x4096'], 0, 0),
    'ragged': (['4096x200', '200x8000'], 0, 0),
    '316x315 adaptive blobs': (['316x315'], 1, 1024),
    'small ragged': (['3x5', '40x2', '17x33'], 0, 7),
    'one pixel': (['1x1'], 1, 64),
    'tall': (['200x8192'], 1, 5000),
}

# Layouts the kernel has used since before unit_layout computed them in one place: they must not drift.
PINNED = {
    '316x315': dict(arena=0, gray=99552, n_hist=16, mask=12608, ws=68032, run_cap=3703, total=230624, rank_off=1201920,
                    f32_off=1226496, otsu_off=224416, stage=112160, run_rf=1280, band_cap=6304, dirty_cap=4096,
                    exact_cap=12912, blob_cap=630, blur_off=199088, runs_off=298640, runs_cap=50085, rank_words=2016),
    '96x96': dict(arena=0, gray=9600, n_hist=16, mask=1152, ws=125312, run_cap=6935, total=140672, rank_off=113152, f32_off=130304),
    '150x230': dict(arena=0, gray=35888, n_hist=16, mask=4608, ws=108032, run_cap=5945, total=166960, rank_off=420096, f32_off=439552),
    '640x480': dict(arena=1, gray=309120, n_hist=16, mask=38400, ws=149488, run_cap=8192, total=131072, arena_bytes=650752,
                    rank_off=3697408, f32_off=3736832),
    '4096x4096': dict(arena=1, gray=16793600, n_hist=16, mask=2097152, ws=2890016, run_cap=65534, total=131072,
                      arena_bytes=30169600, rank_off=201417216, f32_off=202688512),
    'ragged': dict(arena=1, gray=1632000, mask=224000, ws=21119360, run_cap=65534, total=131072, arena_bytes=23871488,
                   rank_off=393392384, f32_off=395845632),
    '316x315 adaptive blobs': dict(f32_off=1226496, blob_tail_off=1624832, scratch_bytes=1665792),
}

# The alias table of vi_device.cuh: the regions each region may overlap.  The gray crop, the masks and the workspace
# are disjoint, and so is everything in the per-CTA scratch.
ALIASES = {
    'hist': {'MA', 'MB', 'MC', 'MD', 'ME', 'ws', 'lattice', 'otsu', 'band', 'runs', 'dirty', 'exact', 'blob', 'stage'},
    'lattice': {'MB', 'MC', 'MD', 'ME', 'ws', 'band', 'runs', 'dirty', 'exact', 'blob'},
    'otsu': {'ws', 'runs', 'dirty', 'exact'},
    'band': {'MD', 'ME', 'blob'},
    'runs': {'ws', 'dirty', 'exact'},
    'dirty': {'ws'},
    'exact': {'ws'},
    'blob': {'MC', 'MD'},
    'stage': {'gray', 'MA'},
}
ALLOWED = {frozenset((a, b)) for a, bs in ALIASES.items() for b in bs}


@pytest.fixture(scope='module')
def layouts(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp('layout') / 'unit_layout_dump')
    csrc = os.path.join(os.path.dirname(_build.LIB_PATH), 'csrc')
    cmd = [_build._nvcc(), '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-I', csrc, '-o', exe,
           os.path.join(HERE, 'unit_layout_dump.cu')]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    args = [f'{OPTIN},{STATIC},{f32},{blob_k}:' + ','.join(units) for units, f32, blob_k in GRIDS.values()]
    out = subprocess.run([exe] + args, capture_output=True, text=True, check=True).stdout.splitlines()
    assert len(out) == len(GRIDS)
    return {name: json.loads(line) for name, line in zip(GRIDS, out)}


@pytest.mark.parametrize('name', sorted(PINNED))
def test_layout_values_are_pinned(layouts, name):
    L = layouts[name]
    assert L['ok']
    assert {k: L[k] for k in PINNED[name]} == PINNED[name]


@pytest.mark.parametrize('name', sorted(GRIDS))
def test_layout_invariants(layouts, name):
    L = layouts[name]
    assert L['ok']
    regions = {r[0]: r[1:] for r in L['regions']}
    unit_end = L['arena_bytes'] if L['arena'] else L['total']
    for rname, (space, off, size) in regions.items():
        assert off % 16 == 0, rname
        assert 0 <= off and off + size <= (unit_end if space == 'unit' else L['scratch_bytes']), rname
    assert L['arena'] or L['total'] + STATIC <= OPTIN
    if not L['arena']:
        assert regions['stage'][1] % 128 == 0           # tensor copies land there: 128-byte aligned like the dynamic base
    assert L['lattice_off'] + L['lattice_bytes'] == L['otsu_off']
    if L['arena']:
        assert L['lattice_fits_max']                    # the arena's workspace is sized for the largest unit's lattice
    overlaps = set()
    names = sorted(regions)
    for i, a in enumerate(names):
        for b in names[i + 1:]:
            (sa, oa, na), (sb, ob, nb) = regions[a], regions[b]
            if sa == sb and na > 0 and nb > 0 and oa < ob + nb and ob < oa + na:
                overlaps.add(frozenset((a, b)))
    assert overlaps <= ALLOWED, sorted(tuple(sorted(p)) for p in overlaps - ALLOWED)


def test_layout_leaves_32_bytes_of_shared_memory_at_316x315(layouts):
    assert OPTIN - STATIC - layouts['316x315']['total'] == 32

