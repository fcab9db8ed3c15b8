"""The k-scaled geometry the scaled build is specified against (include/mosaic_b200.h "scaled compositing") is sound: for the
shipped cell shapes, their step cells and k = 1 ... 5, the scaled cell's rects are k times the cell's rects over the padded grid, its
mask flips are the cell's, and its four flipped masks are the cell's upsampled. So the scaled masks tile the plane wherever the
originals do, and a cell covers output pixel (Y, X) exactly when it covers base pixel (Y / k, X / k)."""
import os

import numpy as np
import pytest

from tests.helpers.render_scale import scaled_cell, upsample

CELLS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cells")
NAMES = sorted(f[:-4] for f in os.listdir(CELLS) if f.endswith(".mcs"))


def test_ten_shapes_ship():
    assert len(NAMES) == 10


@pytest.mark.parametrize("name", NAMES)
def test_scaled_geometry(oracle, name):
    base = oracle.load_mcs(os.path.join(CELLS, name + ".mcs"))
    group = oracle.CellGroup.make(base, 100, 2)
    for step, cell in enumerate(group.cells):
        gx, gy = oracle.grid_size(cell, 3 * cell.size + 7, 2 * cell.size + 5)  # an image size that clips the edge cells
        m4 = cell.masks4()
        for k in range(1, 6):
            sc = scaled_cell(cell, k)
            assert sc.size == k * cell.size
            assert np.array_equal(sc.masks4(), np.stack([upsample(m, k) for m in m4])), (name, step, k)
            for y in range(gy):
                for x in range(gx):
                    r = oracle.rect_at(cell, x - oracle.PAD_GRID, y - oracle.PAD_GRID)
                    assert oracle.rect_at(sc, x - oracle.PAD_GRID, y - oracle.PAD_GRID) == tuple(k * v for v in r), (name, step, k, x, y)
                    assert oracle.flip_at(sc, x - oracle.PAD_GRID, y - oracle.PAD_GRID) == \
                        oracle.flip_at(cell, x - oracle.PAD_GRID, y - oracle.PAD_GRID), (name, step, k, x, y)
