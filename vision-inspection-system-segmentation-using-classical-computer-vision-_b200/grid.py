"""Grid generation and grid JSON v2 (host logic of the hot path's inputs).

Mirrors update_grid_preview (indexing_ui.py:2184-2191), export_grid
(:2739-2782) and import_grid (:2844-2889): same nesting order, same schema, the
same tolerance for legacy files (bare list of boxes, dicts without `version` or
`exclusion_alignment`, boxes without `index`, malformed boxes skipped)."""
from __future__ import annotations

import json
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

Rect = Tuple[int, int, int, int]


@dataclass
class Grid:
    boxes: List[Tuple[Rect, int]] = field(default_factory=list)      # ((x,y,w,h), index) in list order
    exclusions: List[dict] = field(default_factory=list)             # unit-local rect / circle dicts
    ref_centroids: Dict[int, Tuple[float, float]] = field(default_factory=dict)   # keyed by list position
    metadata: dict = field(default_factory=dict)

    @property
    def rects(self) -> List[Rect]:
        return [r for r, _ in self.boxes]

    @property
    def indices(self) -> List[int]:
        return [i for _, i in self.boxes]


def generate_grid(base: Rect, units_x, units_y, blocks_x, blocks_y, unit_space_x=0, unit_space_y=0,
                  block_space_x=0, block_space_y=0) -> List[Tuple[Rect, int]]:
    """by -> uy -> bx -> ux nesting: the index runs row-major across all blocks."""
    x0, y0, uw, uh = (int(v) for v in base)
    block_w = units_x * uw + (units_x - 1) * unit_space_x + block_space_x
    block_h = units_y * uh + (units_y - 1) * unit_space_y + block_space_y
    out = []
    for byi in range(blocks_y):
        for uyi in range(units_y):
            y = y0 + byi * block_h + uyi * (uh + unit_space_y)
            for bxi in range(blocks_x):
                for uxi in range(units_x):
                    x = x0 + bxi * block_w + uxi * (uw + unit_space_x)
                    out.append(((int(x), int(y), uw, uh), len(out)))
    return out


def parse_grid(data) -> Grid:
    g = Grid()
    if isinstance(data, dict) and "boxes" in data:
        raw = data["boxes"]
        g.metadata = data.get("metadata", {}) or {}
        g.exclusions = list(data.get("exclusions", []) or [])
        align = data.get("exclusion_alignment", {}) or {}
        if isinstance(align, dict) and align.get("type") == "seg_centroid_xy":
            refc = align.get("ref_centroids", {}) or {}
            if isinstance(refc, dict):
                for k, vv in refc.items():
                    try:
                        g.ref_centroids[int(k)] = (float(vv.get("cx")), float(vv.get("cy")))
                    except Exception:
                        continue
    elif isinstance(data, list):
        raw = data
    else:
        raw = []
    for item in raw:
        try:
            idx = item.get("index", None)
            rect = (int(item["x"]), int(item["y"]), int(item["w"]), int(item["h"]))
        except Exception:
            continue
        g.boxes.append((rect, len(g.boxes) if idx is None else idx))
    return g


def load_grid(path) -> Grid:
    with open(path, "r") as f:
        return parse_grid(json.load(f))


def grid_to_json(grid: Grid) -> dict:
    return {
        "version": 2,
        "metadata": grid.metadata,
        "boxes": [{"index": idx, "x": int(r[0]), "y": int(r[1]), "w": int(r[2]), "h": int(r[3])}
                  for r, idx in grid.boxes],
        "exclusions": list(grid.exclusions),
        "exclusion_alignment": {
            "type": "seg_centroid_xy",
            "ref_centroids": {str(int(k)): {"cx": float(v[0]), "cy": float(v[1])}
                              for k, v in grid.ref_centroids.items()},
        },
    }


def ref_centroids_from_records(records, image=0) -> Dict[int, Tuple[float, float]]:
    """{unit: (cx, cy)} of one image's records (RECORD_DTYPE, [n, units] or [n * units] with the image field): the
    pre-exclusion centroids run_segmentation_all stores from the reference image (indexing_ui.py:2283-2289).  Units
    without a segmented component (NaN) are left out, as the reference leaves them out.  Assign the result to
    `Grid.ref_centroids`; `save_grid` writes it as exclusion_alignment.ref_centroids."""
    import numpy as np
    r = np.asarray(records).reshape(-1)
    r = r[r['image'] == int(image)]
    out = {}
    for rec in r:
        cx, cy = float(rec['cx']), float(rec['cy'])
        if cx == cx and cy == cy:
            out[int(rec['unit'])] = (cx, cy)
    return out


def save_grid(path, grid: Grid):
    with open(path, "w") as f:
        json.dump(grid_to_json(grid), f, indent=2)


def exclusions_to_table(exclusions):
    """dict schema (indexing_ui.py:1811, :1816) -> rows (shape,a,b,c,d) for vi_excl.
    Any shape other than 'rect' is a circle (:2327); malformed entries are skipped (:2336)."""
    rows = []
    for e in exclusions:
        try:
            if e.get("shape") == "rect":
                rows.append((0, int(e.get("x", 0)), int(e.get("y", 0)), int(e.get("w", 0)), int(e.get("h", 0))))
            else:
                rows.append((1, int(e.get("cx", 0)), int(e.get("cy", 0)), int(e.get("r", 0)), 0))
        except Exception:
            continue
    return rows
