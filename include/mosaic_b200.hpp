// mosaic_b200.hpp -- header-only C++ mirror of the reference's generator classes over the C ABI (mosaic_b200.h).
//
// Same method names, argument meaning and error behaviour as
//   PhotomosaicGeneratorBase / CUDAPhotomosaicGenerator   src/Photomosaic/PhotomosaicGeneratorBase.h:32-112,
//                                                          src/Photomosaic/CUDA/CUDAPhotomosaicGenerator.h:27-60
//   CellShape, CellGroup                                   src/CellShape/CellShape.h, CellGroup.h
//   GridUtility::MosaicBestFit                             src/Grid/GridUtility.h:29-31
// so that callers written against the reference (MainWindow.cpp:584-607, tst_Generator.h:66-137,
// Benchmark_Generator.h:17-81) port mechanically. Qt-free and OpenCV-free: images are described by
// mosaicb200::Image (pointer + geometry; a cv::Mat maps onto it as {m.data, m.rows, m.cols, m.step}).
#pragma once
#include <cstdint>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "mosaic_b200.h"

namespace mosaicb200 {

struct Image {  // 8U BGR view
    const uint8_t *data = nullptr;
    int rows = 0, cols = 0;
    size_t step = 0;  // bytes per row
};

namespace ColourDifference {
enum class Type { RGB_EUCLIDEAN = 0, CIE76 = 1, CIEDE2000 = 2, MAX };  // ColourDifference.h:13-19
}
namespace ColourScheme {
enum class Type { NONE = 0, COMPLEMENTARY, TRIADIC, COMPOUND, TETRADIC, ANALAGOUS, MAX };  // ColourScheme.h:10-19
}

namespace GridUtility {
using CellBestFit = std::optional<size_t>;
using StepBestFit = std::vector<std::vector<CellBestFit>>;
using MosaicBestFit = std::vector<StepBestFit>;
constexpr int PAD_GRID = 2;
}  // namespace GridUtility

class CellShape {
public:
    CellShape() = default;
    explicit CellShape(size_t size) : m_mask(size * size, 255) { init(static_cast<int>(size)); }  // default square cell
    CellShape(const uint8_t *mask, int size) : m_mask(mask, mask + static_cast<size_t>(size) * size) { init(size); }

    int getSize() const { return m_c.size; }
    bool empty() const { return m_mask.empty(); }
    void setRowSpacing(int v) { m_c.row_spacing = v; }
    void setColSpacing(int v) { m_c.col_spacing = v; }
    void setAlternateRowSpacing(int v) { m_c.alt_row_spacing = v; }
    void setAlternateColSpacing(int v) { m_c.alt_col_spacing = v; }
    void setAlternateRowOffset(int v) { m_c.alt_row_offset = v; }
    void setAlternateColOffset(int v) { m_c.alt_col_offset = v; }
    void setAlternateColFlipHorizontal(bool v) { m_c.alt_col_flip_h = v; }
    void setAlternateColFlipVertical(bool v) { m_c.alt_col_flip_v = v; }
    void setAlternateRowFlipHorizontal(bool v) { m_c.alt_row_flip_h = v; }
    void setAlternateRowFlipVertical(bool v) { m_c.alt_row_flip_v = v; }
    int getRowSpacing() const { return m_c.row_spacing; }
    int getColSpacing() const { return m_c.col_spacing; }
    const std::vector<uint8_t> &getCellMask() const { return m_mask; }
    const mosaic_cell_shape &c() const { return m_c; }
    void setName(const std::string &name) { m_name = name; }
    const std::string &getName() const { return m_name; }

    // CellShape::loadFromFile / saveToFile (.mcs, CellShape.cpp:321-434); std::invalid_argument like the reference
    void loadFromFile(const std::string &filename)
    {
        mosaic_cell_shape c{};
        char name[1024] = {0};
        if (mosaic_mcs_load(filename.c_str(), &c, nullptr, 0, name, sizeof name) != MOSAIC_OK)
            throw std::invalid_argument(mosaic_io_last_error());
        std::vector<uint8_t> mask(static_cast<size_t>(c.size) * c.size);
        if (mosaic_mcs_load(filename.c_str(), &c, mask.data(), mask.size(), nullptr, 0) != MOSAIC_OK)
            throw std::invalid_argument(mosaic_io_last_error());
        m_mask = std::move(mask);  // as stored: loadFromFile does not threshold (CellShape.cpp:405-410)
        m_asStored = true;
        m_c = c;
        m_name = name;
    }
    // true for a shape that came from loadFromFile: its mask is kept as the file holds it (non-zero = active downstream)
    bool maskAsStored() const { return m_asStored; }
    void saveToFile(const std::string &filename) const
    {
        if (mosaic_mcs_save(filename.c_str(), &m_c, m_mask.data(), m_name.c_str()) != MOSAIC_OK)
            throw std::invalid_argument(mosaic_io_last_error());
    }

private:
    void init(int size)
    {
        m_c = mosaic_cell_shape{size, size, size, size, size, 0, 0, 0, 0, 0, 0};
        for (auto &v : m_mask)
            v = v > 127 ? 255 : 0;  // setCellMask threshold, CellShape.cpp:123
    }
    std::vector<uint8_t> m_mask;
    mosaic_cell_shape m_c{};
    std::string m_name;
    bool m_asStored = false;
};

class CellGroup {
public:
    void setCellShape(const CellShape &s) { m_shape = s; }
    const CellShape &getCellShape() const { return m_shape; }
    void setDetail(int detail = 100) { m_detail = detail; }
    double getDetail() const { return m_detail / 100.0; }
    int getDetailPercent() const { return m_detail; }
    void setSizeSteps(size_t steps) { m_steps = static_cast<int>(steps); }
    size_t getSizeSteps() const { return static_cast<size_t>(m_steps); }

private:
    CellShape m_shape;
    int m_detail = 100, m_steps = 0;
};

// ImageLibrary (src/ImageLibrary/ImageLibrary.h:9-66): the container that feeds setLibrary. addImage's centre crop and
// EXACT resize (ImageLibrary.cpp:62-86) run on the GPU through mosaic_library_ingest; .mil files are read and written by
// the Python layer (mosaicmagnifique_b200/formats.py), not here.
class ImageLibrary {
public:
    explicit ImageLibrary(size_t imageSize, int device = 0) : m_imageSize(imageSize), m_device(device) {}

    void setImageSize(size_t size)  // ImageLibrary.cpp:42-52
    {
        if (size == m_imageSize)
            return;
        m_imageSize = size;
        for (size_t i = 0; i < m_originalImages.size(); ++i)
            m_resizedImages[i] = ingest(Image{m_originalImages[i].data(), m_originalSize[i], m_originalSize[i],
                                              static_cast<size_t>(m_originalSize[i]) * 3});
    }
    size_t getImageSize() const { return m_imageSize; }

    // the reference inserts at an index drawn from std::random_device (ImageLibrary.cpp:75-78); pass the index to choose it
    size_t addImage(const Image &im, const std::string &name = std::string(), size_t index = static_cast<size_t>(-1))
    {
        if (!im.data || im.rows <= 0 || im.cols <= 0)
            throw std::invalid_argument("t_im was empty.");
        if (index > m_names.size())
            index = m_names.size();
        std::vector<uint8_t> img = ingest(im);
        m_names.insert(m_names.begin() + index, name);
        m_originalSize.insert(m_originalSize.begin() + index, static_cast<int>(m_imageSize));
        m_originalImages.insert(m_originalImages.begin() + index, img);  // addImageInternal, ImageLibrary.cpp:240-244
        m_resizedImages.insert(m_resizedImages.begin() + index, std::move(img));
        return index;
    }
    const std::vector<std::string> &getNames() const { return m_names; }
    const std::vector<std::vector<uint8_t>> &getImages() const { return m_resizedImages; }  // each imageSize x imageSize x 3
    void removeAtIndex(size_t i)
    {
        m_names.erase(m_names.begin() + i);
        m_originalSize.erase(m_originalSize.begin() + i);
        m_originalImages.erase(m_originalImages.begin() + i);
        m_resizedImages.erase(m_resizedImages.begin() + i);
    }
    void clear()
    {
        m_names.clear();
        m_originalSize.clear();
        m_originalImages.clear();
        m_resizedImages.clear();
    }
    // ImageLibrary::saveToFile / loadFromFile (.mil, ImageLibrary.cpp:117-236); std::invalid_argument like the reference
    void saveToFile(const std::string &filename) const
    {
        const std::vector<uint8_t> all = packed();
        std::string names;
        for (const auto &n : m_names)
            names.append(n).push_back('\0');
        if (mosaic_mil_save(filename.c_str(), all.data(), static_cast<int64_t>(m_resizedImages.size()), static_cast<int>(m_imageSize),
                            names.c_str()) != MOSAIC_OK)
            throw std::invalid_argument(mosaic_io_last_error());
    }
    void loadFromFile(const std::string &filename)  // appends the file's images; its image size becomes the library's
    {
        int64_t n = 0;
        int size = 0;
        size_t nameBytes = 0;
        if (mosaic_mil_info(filename.c_str(), &n, &size, &nameBytes) != MOSAIC_OK)
            throw std::invalid_argument(mosaic_io_last_error());
        std::vector<uint8_t> images(static_cast<size_t>(n) * size * size * 3);
        std::vector<char> names(nameBytes + 1, 0);
        if (mosaic_mil_load(filename.c_str(), images.data(), images.size(), names.data(), nameBytes) != MOSAIC_OK)
            throw std::invalid_argument(mosaic_io_last_error());
        m_imageSize = static_cast<size_t>(size);
        const size_t per = static_cast<size_t>(size) * size * 3;
        const char *p = names.data();
        for (int64_t i = 0; i < n; ++i) {
            m_names.emplace_back(p);
            p += m_names.back().size() + 1;
            std::vector<uint8_t> img(images.begin() + i * per, images.begin() + (i + 1) * per);
            m_originalSize.push_back(size);
            m_originalImages.push_back(img);
            m_resizedImages.push_back(std::move(img));
        }
    }

    // contiguous [N][size][size][3] block for PhotomosaicGenerator::setLibrary
    std::vector<uint8_t> packed() const
    {
        std::vector<uint8_t> out;
        out.reserve(m_resizedImages.size() * m_imageSize * m_imageSize * 3);
        for (const auto &im : m_resizedImages)
            out.insert(out.end(), im.begin(), im.end());
        return out;
    }

private:
    std::vector<uint8_t> ingest(const Image &im) const
    {
        std::vector<uint8_t> out(m_imageSize * m_imageSize * 3);
        const int rc = mosaic_library_ingest(m_device, im.data, im.rows, im.cols, im.step, static_cast<int>(m_imageSize), out.data());
        if (rc == MOSAIC_ERR_INVALID_ARGUMENT)
            throw std::invalid_argument("t_im was empty.");
        if (rc != MOSAIC_OK)
            throw std::runtime_error("mosaic_library_ingest failed (CUDA)");
        return out;
    }
    size_t m_imageSize;
    int m_device;
    std::vector<std::string> m_names;
    std::vector<int> m_originalSize;
    std::vector<std::vector<uint8_t>> m_originalImages, m_resizedImages;
};

// CUDAPhotomosaicGenerator(const int device): the only back-end; there is no CPU fallback.
class PhotomosaicGenerator {
public:
    explicit PhotomosaicGenerator(int device = 0)
    {
        if (mosaic_create(device, &m_g) != MOSAIC_OK)
            throw std::runtime_error("mosaic_create failed: no usable CUDA device");
    }
    ~PhotomosaicGenerator() { mosaic_destroy(m_g); }
    PhotomosaicGenerator(const PhotomosaicGenerator &) = delete;
    PhotomosaicGenerator &operator=(const PhotomosaicGenerator &) = delete;

    void setMainImage(const Image &img) { ck(mosaic_set_main_image(m_g, img.data, img.rows, img.cols, img.step)); }
    // library: n square images of size x size, 8U BGR, contiguous
    void setLibrary(const uint8_t *bgr, int64_t n, int size) { ck(mosaic_set_library(m_g, bgr, n, size)); }
    void setColourDifference(ColourDifference::Type t = ColourDifference::Type::RGB_EUCLIDEAN)
    {
        if (mosaic_set_colour_difference(m_g, static_cast<int>(t)) != MOSAIC_OK)
            throw std::invalid_argument(mosaic_last_error(m_g));  // ColourDifference.cpp:23
    }
    void setColourScheme(ColourScheme::Type t = ColourScheme::Type::NONE)
    {
        if (mosaic_set_colour_scheme(m_g, static_cast<int>(t)) != MOSAIC_OK)
            throw std::invalid_argument(mosaic_last_error(m_g));
    }
    void setCellGroup(const CellGroup &cg)
    {
        m_cells = cg;
        ck(mosaic_set_cell_group_ex(m_g, &cg.getCellShape().c(), cg.getCellShape().getCellMask().data(), 0, cg.getDetailPercent(),
                                    static_cast<int>(cg.getSizeSteps()), cg.getCellShape().maskAsStored() ? 1 : 0));
    }
    CellGroup &getCellGroup() { return m_cells; }
    void setGridState(const GridUtility::MosaicBestFit &state)
    {
        for (size_t s = 0; s < state.size(); ++s) {
            const int rows = static_cast<int>(state[s].size()), cols = rows ? static_cast<int>(state[s][0].size()) : 0;
            std::vector<uint8_t> valid(static_cast<size_t>(rows) * cols);
            for (int y = 0; y < rows; ++y)
                for (int x = 0; x < cols; ++x)
                    valid[static_cast<size_t>(y) * cols + x] = state[s][y][x].has_value();
            ck(mosaic_set_grid_state(m_g, static_cast<int>(s), rows, cols, valid.data()));
        }
    }
    // GridGenerator::getGridState(cellGroup, mainImage, rows, cols) on the inputs already set
    GridUtility::MosaicBestFit computeGridState()
    {
        ck(mosaic_compute_grid_state(m_g));
        return getBestFits();
    }
    void setRepeat(int range = 0, int addition = 0) { ck(mosaic_set_repeat(m_g, range, addition)); }

    // Returns true if successful, false when cancelled or on a CUDA error (text in lastError()), like the reference.
    bool generateBestFits() { return mosaic_generate(m_g) == MOSAIC_OK; }
    GridUtility::MosaicBestFit getBestFits() const
    {
        GridUtility::MosaicBestFit out(static_cast<size_t>(mosaic_get_grid_steps(m_g)));
        for (size_t s = 0; s < out.size(); ++s) {
            int rows = 0, cols = 0;
            mosaic_get_grid_size(m_g, static_cast<int>(s), &rows, &cols);
            std::vector<int64_t> v(static_cast<size_t>(rows) * cols);
            mosaic_get_best_fits(m_g, static_cast<int>(s), v.data(), rows, cols);
            out[s].assign(rows, std::vector<GridUtility::CellBestFit>(cols));
            for (int y = 0; y < rows; ++y)
                for (int x = 0; x < cols; ++x)
                    if (v[static_cast<size_t>(y) * cols + x] >= 0)
                        out[s][y][x] = static_cast<size_t>(v[static_cast<size_t>(y) * cols + x]);
        }
        return out;
    }
    // ---- mirrored library tiles (no reference counterpart; see mosaic_b200.h "mirrored library tiles"): the best fit may place an
    // image mirrored horizontally and/or vertically. getBestFits() keeps returning image indices; getBestFitFlips() gives, per step,
    // the orientation of every cell's tile (flip_h + 2 * flip_v, -1 = no best fit).
    void setTileFlips(bool horizontal, bool vertical) { ck(mosaic_set_tile_flips(m_g, (horizontal ? 1 : 0) | (vertical ? 2 : 0))); }
    std::vector<std::vector<std::vector<int8_t>>> getBestFitFlips() const
    {
        std::vector<std::vector<std::vector<int8_t>>> out(static_cast<size_t>(mosaic_get_grid_steps(m_g)));
        for (size_t s = 0; s < out.size(); ++s) {
            int rows = 0, cols = 0;
            mosaic_get_grid_size(m_g, static_cast<int>(s), &rows, &cols);
            std::vector<int8_t> v(static_cast<size_t>(rows) * cols);
            if (mosaic_get_best_fit_flips(m_g, static_cast<int>(s), v.data(), rows, cols) != MOSAIC_OK)
                throw std::runtime_error("getBestFitFlips: no best fits on the current grid state");
            out[s].assign(rows, std::vector<int8_t>(cols));
            for (int y = 0; y < rows; ++y)
                for (int x = 0; x < cols; ++x)
                    out[s][y][x] = v[static_cast<size_t>(y) * cols + x];
        }
        return out;
    }
    // ---- usage limit (no reference counterpart; see mosaic_b200.h "usage limit"): each library image is chosen at most maxUses times
    // per generate, over all size steps (1 = no duplicates, 0 = unlimited); generateBestFits() returns false (lastError() says why)
    // when maxUses * library size is less than the number of cells.
    void setUsageLimit(int maxUses) { ck(mosaic_set_usage_limit(m_g, maxUses)); }
    // cv::Mat buildPhotomosaic(const cv::Scalar&): fills a rows x cols BGRA buffer (step = bytes per row)
    void buildPhotomosaic(const uint8_t backgroundBGRA[4], uint8_t *outBGRA, int rows, int cols, size_t step)
    {
        ck(mosaic_build_photomosaic(m_g, backgroundBGRA, outBGRA, rows, cols, step));
    }
    // ---- scaled compositing (no reference counterpart; see mosaic_b200.h "scaled compositing"): the library's images, same order, at
    // side R = k * cell size; buildPhotomosaicScaled then fills a (k * rows) x (k * cols) BGRA buffer (host or device memory)
    void setRenderLibrary(const uint8_t *bgr, int64_t n, int size) { ck(mosaic_set_render_library(m_g, bgr, n, size)); }
    void buildPhotomosaicScaled(const uint8_t backgroundBGRA[4], uint8_t *outBGRA, int rows, int cols, size_t step)
    {
        ck(mosaic_build_photomosaic_scaled(m_g, backgroundBGRA, outBGRA, rows, cols, step));
    }
    int getMaxProgress() { return mosaic_get_max_progress(m_g); }
    // slot cancel(): callable from any thread or from inside the progress callback; the running kernel drains within milliseconds
    // and generateBestFits() returns false. Sticky like the reference's m_wasCanceled until resetCancel().
    void cancel() { mosaic_cancel(m_g); }
    void resetCancel() { mosaic_reset_cancel(m_g); }
    // signal progress(int): fn is called on the generating thread with the reference's cumulative values
    // (grid positions done, weighted 4^(steps - 1 - step), CPUPhotomosaicGenerator.cpp:55, 87-88)
    void setProgressCallback(mosaic_progress_fn fn, void *user) { mosaic_set_progress_callback(m_g, fn, user); }

    // ---- one generator per GPU of a multi-GPU run (no reference counterpart; see mosaic_b200.h "multi-GPU sharding"):
    // setShard + generateCandidates on every rank, one all-gather of candidateBlock() in rank order, selectFromGathered on every rank
    void setShard(int rank, int world) { ck(mosaic_set_shard(m_g, rank, world)); }
    void generateCandidates() { ck(mosaic_generate_candidates(m_g)); }
    struct CandidateBlock {
        void *device = nullptr;   // {float scores [rowsPerRank][k], int32 indices [rowsPerRank][k]}
        int64_t rowsPerRank = 0;
        int k = 0;
        size_t bytes = 0;
    };
    CandidateBlock candidateBlock(int step) const
    {
        CandidateBlock b;
        mosaic_get_candidate_block(m_g, step, &b.device, &b.rowsPerRank, &b.k, &b.bytes);
        return b;
    }
    void selectFromGathered(int step, const void *gatheredBlocks, int k, int64_t rowsPerRank)
    {
        ck(mosaic_select_from_gathered(m_g, step, gatheredBlocks, k, rowsPerRank));
    }
    std::string lastError() const { return mosaic_last_error(m_g); }
    mosaic_timings timings() const
    {
        mosaic_timings t{};
        mosaic_get_timings(m_g, &t);
        return t;
    }
    mosaic_generator *handle() { return m_g; }

private:
    void ck(int rc)
    {
        if (rc != MOSAIC_OK)
            throw std::runtime_error(mosaic_last_error(m_g));
    }
    mosaic_generator *m_g = nullptr;
    CellGroup m_cells;
};

}  // namespace mosaicb200
