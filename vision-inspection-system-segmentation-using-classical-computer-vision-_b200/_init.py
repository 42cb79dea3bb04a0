from . import grid, synth  # noqa: F401
from ._lib import (BLOB_DTYPE, RECORD_DTYPE, STATUS_NG, STATUS_OK, STATUS_ROI_EMPTY, STATUS_SEGMENTED, ViError,  # noqa: F401
                   ViParams, default_params)
from .api import Inspector, default_inspector  # noqa: F401
from .grid import Grid, generate_grid, load_grid, parse_grid, ref_centroids_from_records, save_grid  # noqa: F401

__all__ = ["grid", "synth", "BLOB_DTYPE", "RECORD_DTYPE", "STATUS_NG", "STATUS_OK", "STATUS_ROI_EMPTY", "STATUS_SEGMENTED", "ViError",
           "ViParams", "default_params", "Inspector", "default_inspector", "Grid", "generate_grid", "load_grid", "parse_grid",
           "ref_centroids_from_records", "save_grid"]
