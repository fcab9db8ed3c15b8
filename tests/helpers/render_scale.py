"""The k-scaled cell group of mosaic_build_photomosaic_scaled (include/mosaic_b200.h "scaled compositing"): every tiling parameter of
a step's normal cell times k, flip flags unchanged, the mask upsampled by nearest neighbour. The reference's buildPhotomosaic on a
k-times larger main image with this group and the render library is what the scaled build must produce."""
from dataclasses import replace

import numpy as np


def upsample(a, k):
    """nearest-neighbour upsampling of the first two axes: every pixel a k x k block"""
    return np.repeat(np.repeat(a, k, 0), k, 1)


def scaled_cell(cell, k):
    """oracle.CellShape with size, row / col spacing, alternate spacings and offsets times k and its mask upsampled"""
    return replace(cell, mask=np.ascontiguousarray(upsample(cell.mask, k)), row_spacing=k * cell.row_spacing,
                   col_spacing=k * cell.col_spacing, alt_row_spacing=k * cell.alt_row_spacing, alt_col_spacing=k * cell.alt_col_spacing,
                   alt_row_offset=k * cell.alt_row_offset, alt_col_offset=k * cell.alt_col_offset)


def scaled_group(oracle, group, k):
    """the oracle CellGroup whose normal cells are the k-scaled cells of `group` (the build reads only the normal cells)"""
    g = oracle.CellGroup()
    g.cells = [scaled_cell(c, k) for c in group.cells]
    g.detail_cells = list(group.detail_cells)
    g.detail, g.size_steps = group.detail, group.size_steps
    return g
