"""Python mirror of the reference's generator interface over the C ABI (include/mosaic_b200.h).

Names, argument meaning and error behaviour follow the reference so its fixtures port mechanically
(test/tst_Generator.h:66-137, Benchmark/Benchmark_Generator.h:17-81):

    PhotomosaicGeneratorBase   src/Photomosaic/PhotomosaicGeneratorBase.h:32-112
    CellShape                  src/CellShape/CellShape.h
    CellGroup                  src/CellShape/CellGroup.h
    ColourDifference::Type     src/Photomosaic/ColourDifference.h:13-19
    ColourScheme::Type         src/Photomosaic/ColourScheme.h:10-19

Images are numpy arrays where the reference takes cv::Mat (8U BGR, H x W x 3); the best-fit grid is a list
(one entry per size step) of int64 arrays with -1 where the reference holds std::nullopt.
All compute happens in libmosaic_b200.so on the GPU; nothing here falls back to the CPU.
"""
from __future__ import annotations

import ctypes
import enum

import numpy as np

from ._capi import PROGRESS_FN, CellShapeC, MosaicError, Timings, capi


class ColourDifference(enum.IntEnum):
    RGB_EUCLIDEAN = 0
    CIE76 = 1
    CIEDE2000 = 2


class ColourScheme(enum.IntEnum):
    NONE = 0
    COMPLEMENTARY = 1
    TRIADIC = 2
    COMPOUND = 3
    TETRADIC = 4
    ANALAGOUS = 5


RGB_EUCLIDEAN, CIE76, CIEDE2000 = ColourDifference.RGB_EUCLIDEAN, ColourDifference.CIE76, ColourDifference.CIEDE2000
PAD_GRID = 2  # GridUtility::PAD_GRID


class CellShape:
    """CellShape (src/CellShape/CellShape.h:98-109): a binary square mask plus tiling parameters."""

    def __init__(self, mask_or_size, as_stored: bool = False):
        """as_stored: the mask comes from CellShape::loadFromFile, which keeps the decoded values (no threshold, CellShape.cpp:405-410);
        non-zero = active downstream, and only resized() binarises. Makes no difference for the binary masks the reference writes."""
        self._as_stored = bool(as_stored)
        if isinstance(mask_or_size, (int, np.integer)):
            mask = np.full((int(mask_or_size), int(mask_or_size)), 255, np.uint8)  # CellShape(size_t), CellShape.cpp:66-69
        else:
            mask = np.asarray(mask_or_size)
        if mask.ndim != 2 or mask.shape[0] != mask.shape[1] or mask.dtype != np.uint8:
            raise ValueError("Unsupported mask type")  # std::invalid_argument, CellShape.cpp:133
        self._mask = np.ascontiguousarray(mask) if as_stored else np.where(mask > 127, 255, 0).astype(np.uint8)  # setCellMask threshold
        s = mask.shape[0]
        self.rowSpacing = self.colSpacing = self.alternateRowSpacing = self.alternateColSpacing = s
        self.alternateRowOffset = self.alternateColOffset = 0
        self.alternateColFlipHorizontal = self.alternateColFlipVertical = False
        self.alternateRowFlipHorizontal = self.alternateRowFlipVertical = False
        self.name = ""

    def getSize(self):
        return self._mask.shape[0]

    def getCellMask(self, flippedHorizontal=False, flippedVertical=False):
        m = self._mask
        if flippedHorizontal:
            m = m[:, ::-1]
        if flippedVertical:
            m = m[::-1, :]
        return np.ascontiguousarray(m)

    def _c(self) -> CellShapeC:
        return CellShapeC(self.getSize(), self.rowSpacing, self.colSpacing, self.alternateRowSpacing, self.alternateColSpacing,
                          self.alternateRowOffset, self.alternateColOffset, int(self.alternateColFlipHorizontal),
                          int(self.alternateColFlipVertical), int(self.alternateRowFlipHorizontal),
                          int(self.alternateRowFlipVertical))

    @staticmethod
    def _from_c(c: CellShapeC, mask: np.ndarray, as_stored: bool = False) -> "CellShape":
        s = CellShape(mask, as_stored=as_stored)
        s.rowSpacing, s.colSpacing = c.row_spacing, c.col_spacing
        s.alternateRowSpacing, s.alternateColSpacing = c.alt_row_spacing, c.alt_col_spacing
        s.alternateRowOffset, s.alternateColOffset = c.alt_row_offset, c.alt_col_offset
        s.alternateColFlipHorizontal, s.alternateColFlipVertical = bool(c.alt_col_flip_h), bool(c.alt_col_flip_v)
        s.alternateRowFlipHorizontal, s.alternateRowFlipVertical = bool(c.alt_row_flip_h), bool(c.alt_row_flip_v)
        return s

    def resized(self, size: int) -> "CellShape":
        """CellShape::resized (CellShape.cpp:281-312), computed by the library's host model."""
        if size == self.getSize():
            return self._copy()
        L = capi()
        out = np.empty((size, size), np.uint8)
        # ImageUtility::resizeImage (ImageUtility.cpp:50-51): INTER_AREA when shrinking, INTER_CUBIC when growing
        fn = L.mosaic_host_resize_cubic_u8 if size > self.getSize() else L.mosaic_host_resize_area_u8
        rc = fn(self._mask.ctypes.data, self.getSize(), self.getSize(), 1, out.ctypes.data, size, size)
        if rc:
            raise MosaicError(rc, "resize failed")
        r = CellShape(out)
        ratio = size / self.getSize()
        fl = lambda v: int(np.floor(v * ratio))
        r.rowSpacing, r.colSpacing = max(fl(self.rowSpacing), 1), max(fl(self.colSpacing), 1)
        r.alternateRowSpacing, r.alternateColSpacing = max(fl(self.alternateRowSpacing), 1), max(fl(self.alternateColSpacing), 1)
        r.alternateRowOffset, r.alternateColOffset = fl(self.alternateRowOffset), fl(self.alternateColOffset)
        for a in ("alternateColFlipHorizontal", "alternateColFlipVertical", "alternateRowFlipHorizontal", "alternateRowFlipVertical", "name"):
            setattr(r, a, getattr(self, a))
        return r

    def _copy(self):
        r = CellShape(self._mask, as_stored=self._as_stored)
        r.__dict__.update({k: v for k, v in self.__dict__.items() if k != "_mask"})
        return r


def load_mcs(path: str) -> CellShape:
    """Reads a .mcs cell shape (CellShape::loadFromFile, CellShape.cpp:363-434) with the library's own reader
    (mosaic_mcs_load: QDataStream layout + PNG codec in csrc/containers.cpp, no OpenCV / Qt involved)."""
    L = capi()
    c = CellShapeC()
    name = ctypes.create_string_buffer(1024)
    bpath = str(path).encode()
    rc = L.mosaic_mcs_load(bpath, ctypes.byref(c), None, 0, name, len(name))
    if rc:
        raise MosaicError(rc, L.mosaic_io_last_error().decode())
    mask = np.empty((c.size, c.size), np.uint8)
    rc = L.mosaic_mcs_load(bpath, ctypes.byref(c), mask.ctypes.data, mask.size, name, len(name))
    if rc:
        raise MosaicError(rc, L.mosaic_io_last_error().decode())
    s = CellShape._from_c(c, mask, as_stored=True)
    s.name = name.value.decode()
    return s


class CellGroup:
    """CellGroup (src/CellShape/CellGroup.h): top-level shape + detail (percent) + size steps."""

    def __init__(self):
        self._shape = None
        self._detail = 100
        self._size_steps = 0

    def setCellShape(self, shape: CellShape):
        self._shape = shape

    def setDetail(self, detail: int = 100):
        self._detail = int(detail)

    def getDetail(self) -> float:
        return self._detail / 100.0

    def setSizeSteps(self, steps: int):
        self._size_steps = int(steps)

    def getSizeSteps(self) -> int:
        return self._size_steps

    def getCellSize(self, sizeStep: int = 0, detail: bool = False) -> int:
        return self.getCell(sizeStep, detail).getSize()

    def getCell(self, sizeStep: int = 0, detail: bool = False) -> CellShape:
        """The normal or detail cell of one size step, derived as CellGroup::setDetail / setSizeSteps do (CellGroup.cpp:65-128):
        every step halves the previous step's normal cell (integer division), the detail cell is the step's normal cell
        resized to max(int(size * detail), 1). Host arithmetic of the library (CellShape.resized), no device needed."""
        if self._shape is None:
            raise ValueError("cell group has no shape")
        if not 0 <= sizeStep <= self._size_steps:
            raise IndexError("size step out of range")  # std::out_of_range from cells.at(), CellGroup.cpp:131-145
        cell = self._shape
        size = cell.getSize()
        for _ in range(sizeStep):
            size //= 2
            cell = cell.resized(size)
        return cell.resized(max(int(size * self.getDetail()), 1)) if detail else cell


class PhotomosaicGenerator:
    """The reference's generator object (PhotomosaicGeneratorBase + CUDAPhotomosaicGenerator) on one B200."""

    def __init__(self, device: int = 0):
        self._L = capi()
        h = ctypes.c_void_p()
        rc = self._L.mosaic_create(int(device), ctypes.byref(h))
        if rc:
            raise MosaicError(rc, "mosaic_create failed: no usable CUDA device %d (there is no CPU fallback)" % device)
        self._h = h
        self._cells = None
        self._progress_cb = None
        self._shapes = None
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._L.mosaic_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc:
            raise MosaicError(rc, self._L.mosaic_last_error(self._h).decode())

    # ---- setters (PhotomosaicGeneratorBase.h:40-66)
    def setMainImage(self, img: np.ndarray):
        if img.dtype != np.uint8 or img.ndim != 3 or img.shape[2] != 3:
            raise ValueError("main image must be 8U BGR")
        if img.strides[2] != 1 or img.strides[1] != 3:
            img = np.ascontiguousarray(img)
        self._main_shape = img.shape[:2]
        self._ck(self._L.mosaic_set_main_image(self._h, img.ctypes.data, img.shape[0], img.shape[1], img.strides[0]))

    def setLibrary(self, lib):
        """lib: N x S x S x 3 uint8 array (or a list of S x S x 3 images), already at the cell size."""
        arr = np.ascontiguousarray(np.stack(lib) if isinstance(lib, (list, tuple)) else lib)
        if arr.dtype != np.uint8 or arr.ndim != 4 or arr.shape[3] != 3 or arr.shape[1] != arr.shape[2]:
            raise ValueError("library must be N x S x S x 3 uint8")
        self._n_lib = arr.shape[0]
        self._ck(self._L.mosaic_set_library(self._h, arr.ctypes.data, arr.shape[0], arr.shape[1]))

    def setLibraryPtr(self, ptr: int, n: int, size: int):
        """Same as setLibrary from a raw host pointer (e.g. a pinned torch tensor's data_ptr())."""
        self._n_lib = n
        self._ck(self._L.mosaic_set_library(self._h, ptr, n, size))

    def setMainImagePtr(self, ptr: int, rows: int, cols: int, row_stride: int):
        self._main_shape = (rows, cols)
        self._ck(self._L.mosaic_set_main_image(self._h, ptr, rows, cols, row_stride))

    def setColourDifference(self, t=ColourDifference.RGB_EUCLIDEAN):
        self._ck(self._L.mosaic_set_colour_difference(self._h, int(t)))

    def setColourScheme(self, t=ColourScheme.NONE):
        self._ck(self._L.mosaic_set_colour_scheme(self._h, int(t)))

    def setCellGroup(self, cells: CellGroup):
        if cells._shape is None:
            raise ValueError("cell group has no shape")
        c = cells._shape._c()
        m = cells._shape.getCellMask()
        self._ck(self._L.mosaic_set_cell_group_ex(self._h, ctypes.byref(c), m.ctypes.data, 0, cells._detail, cells._size_steps,
                                                  int(cells._shape._as_stored)))
        self._cells = cells

    def getCellGroup(self) -> CellGroup:
        return self._cells

    def getCellGroupCell(self, step: int, detail: bool) -> CellShape:
        c = CellShapeC()
        self._ck(self._L.mosaic_get_cell_shape(self._h, step, int(detail), ctypes.byref(c), None, 0))
        m = np.empty((c.size, c.size), np.uint8)
        self._ck(self._L.mosaic_get_cell_shape(self._h, step, int(detail), ctypes.byref(c), m.ctypes.data, m.size))
        return CellShape._from_c(c, m)

    def setGridState(self, gridState):
        """gridState: list (per step) of rows x cols arrays; entries < 0 (or None / False) are std::nullopt."""
        for step, g in enumerate(gridState):
            a = np.asarray(g)
            valid = np.ascontiguousarray((a >= 0) if a.dtype != bool else a, dtype=np.uint8)
            self._ck(self._L.mosaic_set_grid_state(self._h, step, valid.shape[0], valid.shape[1], valid.ctypes.data))

    def computeGridState(self):
        """GridGenerator::getGridState(cellGroup, mainImage, rows, cols) on the inputs already set
        (Benchmark_Generator.h:70); returns the state like getBestFits()."""
        self._ck(self._L.mosaic_compute_grid_state(self._h))
        return self.getBestFits()

    def setRepeat(self, repeatRange: int = 0, repeatAddition: int = 0):
        self._ck(self._L.mosaic_set_repeat(self._h, int(repeatRange), int(repeatAddition)))

    def setVariantQuirk(self, faithful: bool = True):
        self._ck(self._L.mosaic_set_variant_quirk(self._h, int(faithful)))

    # ---- run
    def generateBestFits(self) -> bool:
        """Returns True on success, False when cancelled (as the reference); raises MosaicError on errors the
        reference reports through message boxes."""
        rc = self._L.mosaic_generate(self._h)
        if rc == -6:
            return False
        self._ck(rc)
        return True

    def getBestFits(self):
        out = []
        for step in range(self._L.mosaic_get_grid_steps(self._h)):
            r, c = ctypes.c_int(), ctypes.c_int()
            self._ck(self._L.mosaic_get_grid_size(self._h, step, ctypes.byref(r), ctypes.byref(c)))
            g = np.empty((r.value, c.value), np.int64)
            self._ck(self._L.mosaic_get_best_fits(self._h, step, g.ctypes.data, r.value, c.value))
            out.append(g)
        return out

    # ---- mirrored library tiles (no reference counterpart, include/mosaic_b200.h "mirrored library tiles")
    def setTileFlips(self, horizontal: bool = False, vertical: bool = False):
        """Lets the best fit place a library image mirrored horizontally and/or vertically. getBestFits() keeps returning image
        indices; getBestFitFlips() the orientation; getDifferences() has a column per (orientation, image) slot, orientation-major."""
        self._flips = int(bool(horizontal)) | 2 * int(bool(vertical))
        self._ck(self._L.mosaic_set_tile_flips(self._h, self._flips))

    def getBestFitFlips(self):
        """Per step an int8 array: orientation of each cell's tile, flip_h + 2 * flip_v (as mosaic_flip_at), -1 = no best fit."""
        out = []
        for step in range(self._L.mosaic_get_grid_steps(self._h)):
            r, c = ctypes.c_int(), ctypes.c_int()
            self._ck(self._L.mosaic_get_grid_size(self._h, step, ctypes.byref(r), ctypes.byref(c)))
            g = np.empty((r.value, c.value), np.int8)
            rc = self._L.mosaic_get_best_fit_flips(self._h, step, g.ctypes.data, r.value, c.value)
            if rc:
                raise MosaicError(rc, "getBestFitFlips: no best fits on the current grid state")
            out.append(g)
        return out

    # ---- usage limit (no reference counterpart, include/mosaic_b200.h "usage limit")
    def setUsageLimit(self, maxUses: int = 0):
        """Lets each library image be chosen at most maxUses times per generate, over all size steps (1 = no duplicates, 0 = unlimited).
        Cells are decided in step and raster order, each taking the best image that is still allowed; generateBestFits() raises
        MosaicError when maxUses * library size is less than the number of cells."""
        self._ck(self._L.mosaic_set_usage_limit(self._h, int(maxUses)))

    def buildPhotomosaic(self, backgroundColour=(0, 0, 0, 0)) -> np.ndarray:
        """PhotomosaicGeneratorBase::buildPhotomosaic(const cv::Scalar&): H x W x 4 uint8 BGRA mosaic."""
        rows, cols = self._main_shape
        out = np.empty((rows, cols, 4), np.uint8)
        bg = np.asarray(backgroundColour, np.uint8)
        self._ck(self._L.mosaic_build_photomosaic(self._h, bg.ctypes.data, out.ctypes.data, rows, cols, out.strides[0]))
        return out

    def getMaxProgress(self) -> int:
        return self._L.mosaic_get_max_progress(self._h)

    def setProgressCallback(self, fn):
        self._progress_cb = PROGRESS_FN(lambda p, _u: fn(p)) if fn else PROGRESS_FN()
        self._L.mosaic_set_progress_callback(self._h, self._progress_cb, None)

    def cancel(self):
        """slot cancel(): sticky like m_wasCanceled -- generateBestFits() returns False until resetCancel()."""
        self._L.mosaic_cancel(self._h)

    def resetCancel(self):
        self._L.mosaic_reset_cancel(self._h)

    # ---- parity / measurement taps
    def setKeepDifferences(self, keep: bool = True):
        self._ck(self._L.mosaic_set_keep_differences(self._h, int(keep)))

    def getDifferences(self, step: int = 0) -> np.ndarray:
        first, n, k = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int()
        rc = self._L.mosaic_get_candidate_count(self._h, step, ctypes.byref(first), ctypes.byref(n), ctypes.byref(k))
        n_cells = n.value if rc == 0 else self._L.mosaic_get_valid_cell_count(self._h, step)
        n_slots = self._n_lib << bin(getattr(self, "_flips", 0)).count("1")  # O * N columns with tile flips
        out = np.empty((n_cells, n_slots), np.float32)
        self._ck(self._L.mosaic_get_differences(self._h, step, out.ctypes.data, n_cells, n_slots))
        return out

    def setReportMargins(self, report: bool = True):
        self._ck(self._L.mosaic_set_report_margins(self._h, int(report)))

    def getMargins(self, step: int = 0):
        """(best, second-best) penalised score of every valid cell of a step (tie-band reporting)."""
        n = self._L.mosaic_get_valid_cell_count(self._h, step)
        best, second = np.empty(n, np.float32), np.empty(n, np.float32)
        self._ck(self._L.mosaic_get_margins(self._h, step, best.ctypes.data, second.ctypes.data, n))
        return best, second

    def getTimings(self) -> dict:
        t = Timings()
        self._ck(self._L.mosaic_get_timings(self._h, ctypes.byref(t)))
        return {n: getattr(t, n) for n, _ in Timings._fields_}

    # ---- multi-GPU sharding (one process per GPU; exchange done by the caller, see parallel.py)
    def setShard(self, rank: int, world: int):
        self._ck(self._L.mosaic_set_shard(self._h, rank, world))

    def generateCandidates(self):
        self._ck(self._L.mosaic_generate_candidates(self._h))

    def candidateInfo(self, step: int):
        first, n, k = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int()
        self._ck(self._L.mosaic_get_candidate_count(self._h, step, ctypes.byref(first), ctypes.byref(n), ctypes.byref(k)))
        s, i = ctypes.c_void_p(), ctypes.c_void_p()
        self._ck(self._L.mosaic_get_candidates_device(self._h, step, ctypes.byref(s), ctypes.byref(i)))
        return {"first_cell": first.value, "n_cells": n.value, "k": k.value, "scores_ptr": s.value, "indices_ptr": i.value,
                "n_valid": self._L.mosaic_get_valid_cell_count(self._h, step)}

    def selectFromCandidates(self, step: int, scores_ptr: int, indices_ptr: int, k: int):
        self._ck(self._L.mosaic_select_from_candidates(self._h, step, scores_ptr, indices_ptr, k))

    def candidateBlock(self, step: int):
        """This rank's candidates of a step as ONE device block {f32 scores [rows_per_rank][k], i32 indices [rows_per_rank][k]};
        every rank's block has the same size, so a single all-gather assembles the step (parallel.generate_sharded)."""
        ptr, rows, k, nbytes = ctypes.c_void_p(), ctypes.c_int64(), ctypes.c_int(), ctypes.c_size_t()
        self._ck(self._L.mosaic_get_candidate_block(self._h, step, ctypes.byref(ptr), ctypes.byref(rows), ctypes.byref(k),
                                                    ctypes.byref(nbytes)))
        return {"ptr": ptr.value, "rows_per_rank": rows.value, "k": k.value, "bytes": nbytes.value,
                "n_valid": self._L.mosaic_get_valid_cell_count(self._h, step)}

    def selectFromGathered(self, step: int, gathered_ptr: int, k: int, rows_per_rank: int):
        self._ck(self._L.mosaic_select_from_gathered(self._h, step, gathered_ptr, k, rows_per_rank))

    # ---- sharded inputs: a rank uploads only what it computes on
    def shardRows(self, rows: int, cols: int):
        """Main-image rows [lo, hi) this handle's cells read (cell group, grid state and shard set beforehand)."""
        lo, hi = ctypes.c_int(), ctypes.c_int()
        self._ck(self._L.mosaic_get_shard_rows(self._h, rows, cols, ctypes.byref(lo), ctypes.byref(hi)))
        return lo.value, hi.value

    def setMainImageRowsPtr(self, ptr: int, rows: int, cols: int, row_stride: int, row_lo: int, row_hi: int):
        """setMainImage from a pointer to row 0 of the full image, uploading rows [row_lo, row_hi) only."""
        self._main_shape = (rows, cols)
        self._ck(self._L.mosaic_set_main_image_rows(self._h, ptr, rows, cols, row_stride, row_lo, row_hi))

    def setLibraryShardPtr(self, slice_ptr: int, first: int, count: int, n_total: int, size: int, capacity: int):
        """This rank's slice of the library (resized to the detail size on the GPU when detail != 100 %)."""
        self._n_lib = n_total
        self._ck(self._L.mosaic_set_library_shard(self._h, slice_ptr, first, count, n_total, size, capacity))

    def libraryDevice(self):
        ptr, stored, cap = ctypes.c_void_p(), ctypes.c_int(), ctypes.c_int64()
        self._ck(self._L.mosaic_get_library_device(self._h, ctypes.byref(ptr), ctypes.byref(stored), ctypes.byref(cap)))
        return {"ptr": ptr.value, "stored_size": stored.value, "capacity": cap.value}
