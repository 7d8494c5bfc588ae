// hgi.hpp -- C++ host-side mirror of the `hgi` crate's public API (src/lib.rs:16-23) over the C ABI
// in hgi.h.  Header-only; link with -lhgi_b200.  The reference's toolchain (nightly Rust) is not
// available in this environment, so this is the compiled-language host layer north_star asks for:
// same names, argument meaning and error behaviour as the crate, no compute of its own.
//
//   Rust                                              here
//   Linear::from(QuantizationLevel::Medium)           hgi::Linear::from(hgi::QuantizationLevel::Medium)
//   Encoder::new(Crossed, quantizator, levels)        hgi::Encoder<hgi::Crossed, hgi::Linear>(Crossed{}, q, levels)
//   encoder.encode(image) -> Grid                     encoder.encode(image) -> hgi::Grid
//   Decoder::new(Crossed).decode((w,h), levels,&grid) hgi::Decoder<hgi::Crossed>(Crossed{}).decode({w,h}, levels, grid)
//   Archive{metadata, grid}.serialize_to_writer(w)    hgi::Archive{metadata, grid}.serialize_to_writer(os)
//   Archive::deserialize_from_reader(r)               hgi::Archive::deserialize_from_reader(is)
#pragma once
#include <cstdint>
#include <cstring>
#include <istream>
#include <iterator>
#include <memory>
#include <mutex>
#include <ostream>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "hgi.h"

namespace hgi {

// Errors: encode/decode are infallible in the reference (src/encoder.rs:39, src/decoder.rs:18); here a
// failing CUDA call or bad argument surfaces as hgi::Error.  Archive errors correspond to the
// `Result<_, Box<Error>>` of src/archive.rs:31,43 ("incorrect magic number", src/archive.rs:49).
class Error : public std::runtime_error {
public:
    Error(int status, const std::string& where)
        : std::runtime_error(where + ": " + hgi_strerror(status)), status_(status) {}
    int status() const { return status_; }
private:
    int status_;
};

inline void check(int status, const char* where) { if (status != HGI_OK) throw Error(status, where); }

enum class QuantizationLevel : uint32_t { Lossless = 0, Low = 1, Medium = 2, High = 3 };   // src/quantizator.rs:3-8
enum class InterpolationType : uint32_t { Crossed = 0, Line = 1, Previous = 2 };           // src/interpolator.rs:4-9

struct Crossed { static constexpr int id = HGI_INTERP_CROSSED; };   // src/interpolator.rs:30
struct LeftTop { static constexpr int id = HGI_INTERP_LEFTTOP; };   // src/interpolator.rs:15

// `trait Quantizator: From<QuantizationLevel> { quantize(u8)->u8; error()->u8 }` (src/quantizator.rs:12-15)
template <int KIND>
class QuantizatorBase {
public:
    static constexpr int kind = KIND;
    explicit QuantizatorBase(QuantizationLevel level = QuantizationLevel::Lossless) : level_(level)
    {
        check(hgi_quant_table(KIND, (int)level, table_, &error_), "hgi_quant_table");
    }
    static QuantizatorBase from(QuantizationLevel level) { return QuantizatorBase(level); }
    uint8_t quantize(uint8_t value) const { return table_[value]; }
    uint8_t error() const { return error_; }
    QuantizationLevel level() const { return level_; }
private:
    QuantizationLevel level_;
    uint8_t table_[256];
    uint8_t error_ = 0;
};
using NoOp = QuantizatorBase<HGI_QUANT_NOOP>;      // src/quantizator.rs:17-34
using Linear = QuantizatorBase<HGI_QUANT_LINEAR>;  // src/quantizator.rs:36-74

// One per GPU; shared_ptr so encoders/decoders can hold it.
class Context {
public:
    explicit Context(int device = 0) { check(hgi_ctx_create(device, &ctx_), "hgi_ctx_create"); }
    ~Context() { hgi_ctx_destroy(ctx_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    hgi_ctx_t* get() const { return ctx_; }
    void set_path(hgi_path_t path) { check(hgi_ctx_set_path(ctx_, path), "hgi_ctx_set_path"); }
    uint64_t kernel_launches() const { return hgi_ctx_kernel_launches(ctx_); }
    static std::shared_ptr<Context> shared(int device = 0)
    {
        static std::shared_ptr<Context> c = std::make_shared<Context>(device);
        return c;
    }
private:
    hgi_ctx_t* ctx_ = nullptr;
};

// Plane storage: page-locked host memory (hgi_host_alloc), so that the copies of the host-pointer entry points are
// single DMAs instead of driver-staged pageable copies (a 1080p encode call: ~0.1 ms instead of ~0.45 ms).  Freed
// blocks are kept in a small process-wide cache keyed by size, because pinning is expensive and the reference's usage
// -- one Grid / GrayImage of the same size per call (benches/bench.rs:54-110) -- recycles the same few blocks.
// `Bytes(n)` / `resize(n)` leave new bytes uninitialised (every entry point overwrites all of them); `Bytes(n, v)`
// fills.  Falls back to malloc when pinning fails.
class PinnedPool {
public:
    static void* get(size_t bytes, bool* pinned)
    {
        {
            std::lock_guard<std::mutex> lock(mutex());
            auto& c = cache();
            for (size_t i = 0; i < c.size(); ++i)
                if (c[i].bytes == bytes) {
                    void* p = c[i].p;
                    c.erase(c.begin() + (long)i);
                    *pinned = true;
                    return p;
                }
        }
        void* p = hgi_host_alloc(bytes);
        *pinned = p != nullptr;
        return p ? p : ::operator new(bytes ? bytes : 1);
    }
    static void put(void* p, size_t bytes, bool pinned)
    {
        if (!p) return;
        if (!pinned) { ::operator delete(p); return; }
        {
            std::lock_guard<std::mutex> lock(mutex());
            if (cache().size() < 8) { cache().push_back(Block{p, bytes}); return; }
        }
        hgi_host_free(p);
    }
private:
    struct Block { void* p; size_t bytes; };
    struct Cache {
        std::vector<Block> blocks;
        ~Cache() { for (const Block& b : blocks) hgi_host_free(b.p); }
    };
    static std::vector<Block>& cache() { static Cache c; return c.blocks; }
    static std::mutex& mutex() { static std::mutex m; return m; }
};

class Bytes {
public:
    Bytes() = default;
    explicit Bytes(size_t n) { alloc(n); }
    Bytes(size_t n, uint8_t fill) { alloc(n); std::memset(p_, fill, n); }
    Bytes(const Bytes& o) { alloc(o.n_); if (o.n_) std::memcpy(p_, o.p_, o.n_); }
    Bytes(Bytes&& o) noexcept : p_(o.p_), n_(o.n_), pinned_(o.pinned_) { o.p_ = nullptr; o.n_ = 0; }
    Bytes& operator=(Bytes o) noexcept { swap(o); return *this; }
    ~Bytes() { PinnedPool::put(p_, n_, pinned_); }
    void swap(Bytes& o) noexcept { std::swap(p_, o.p_); std::swap(n_, o.n_); std::swap(pinned_, o.pinned_); }
    void resize(size_t n)   // new bytes are uninitialised
    {
        if (n == n_) return;
        Bytes t(n);
        if (p_ && n_) std::memcpy(t.p_, p_, n < n_ ? n : n_);
        swap(t);
    }
    size_t size() const { return n_; }
    bool empty() const { return n_ == 0; }
    uint8_t* data() { return p_; }
    const uint8_t* data() const { return p_; }
    uint8_t& operator[](size_t i) { return p_[i]; }
    uint8_t operator[](size_t i) const { return p_[i]; }
    uint8_t* begin() { return p_; }
    uint8_t* end() { return p_ + n_; }
    const uint8_t* begin() const { return p_; }
    const uint8_t* end() const { return p_ + n_; }
    bool operator==(const Bytes& o) const { return n_ == o.n_ && (n_ == 0 || std::memcmp(p_, o.p_, n_) == 0); }
    bool operator!=(const Bytes& o) const { return !(*this == o); }
private:
    void alloc(size_t n) { n_ = n; p_ = n ? static_cast<uint8_t*>(PinnedPool::get(n, &pinned_)) : nullptr; }
    uint8_t* p_ = nullptr;
    size_t n_ = 0;
    bool pinned_ = false;
};

// `image::GrayImage`: row-major u8, stride == width, zero-filled on construction (image 0.19).
struct GrayImage {
    uint32_t width = 0, height = 0;
    Bytes data;
    GrayImage() = default;
    GrayImage(uint32_t w, uint32_t h) : width(w), height(h), data((size_t)w * h, (uint8_t)0) {}
    struct Uninitialized {};
    GrayImage(uint32_t w, uint32_t h, Uninitialized) : width(w), height(h), data((size_t)w * h) {}
    std::pair<uint32_t, uint32_t> dimensions() const { return {width, height}; }
    uint8_t& at(uint32_t x, uint32_t y) { return data[(size_t)y * width + x]; }
    uint8_t at(uint32_t x, uint32_t y) const { return data[(size_t)y * width + x]; }
};

// src/grid.rs:1-5
struct Grid {
    Bytes buffer;
    size_t width = 0;
    uint8_t get(uint32_t column, uint32_t line) const { return buffer[(size_t)line * width + column]; }
    bool operator==(const Grid& o) const { return width == o.width && buffer == o.buffer; }
};

// `Encoder<I, Q>` (src/encoder.rs:7-24)
template <class I, class Q>
class Encoder {
public:
    Encoder(I, Q quantizator, size_t scale_level, std::shared_ptr<Context> ctx = Context::shared())
        : quantizator_(std::move(quantizator)), scale_level_(scale_level), ctx_(std::move(ctx)) {}

    // `encode(&mut self, input: GrayImage) -> Grid` (src/encoder.rs:39-71).  The reference consumes
    // `input` and uses it as reconstruction scratch; here it is taken by const reference.
    Grid encode(const GrayImage& input, GrayImage* reconstruction = nullptr)
    {
        Grid grid;
        grid.width = input.width;
        grid.buffer.resize(input.data.size());
        if (reconstruction) *reconstruction = GrayImage(input.width, input.height, GrayImage::Uninitialized{});
        const hgi_params_t p{(uint32_t)scale_level_, I::id, Q::kind, (int32_t)quantizator_.level()};
        check(hgi_encode_u8(ctx_->get(), input.data.data(), input.width, input.height, &p, grid.buffer.data(),
                            reconstruction ? reconstruction->data.data() : nullptr), "hgi_encode_u8");
        return grid;
    }
private:
    Q quantizator_;
    size_t scale_level_;
    std::shared_ptr<Context> ctx_;
};

// `Decoder<I>` (src/decoder.rs:6-16)
template <class I>
class Decoder {
public:
    explicit Decoder(I, std::shared_ptr<Context> ctx = Context::shared()) : ctx_(std::move(ctx)) {}

    // `decode(&mut self, (width, height): (u32, u32), levels: usize, grid: &Grid) -> GrayImage` (src/decoder.rs:18-46)
    GrayImage decode(std::pair<uint32_t, uint32_t> dimensions, size_t levels, const Grid& grid)
    {
        GrayImage image(dimensions.first, dimensions.second, GrayImage::Uninitialized{});   // every pixel is written below
        if (grid.buffer.size() != image.data.size()) throw Error(HGI_ERR_INVALID_ARG, "Decoder::decode");
        const hgi_params_t p{(uint32_t)levels, I::id, HGI_QUANT_NOOP, 0};
        check(hgi_decode_u8(ctx_->get(), grid.buffer.data(), image.width, image.height, &p, image.data.data()),
              "hgi_decode_u8");
        return image;
    }

    // Scalable decode (not in the reference): decode(...) at 1/2^scale_log2 resolution -- every 2^k-th pixel of every
    // 2^k-th row -- cut to `region` (scaled coordinates; nullptr = all of it), from the grid rows it depends on only.
    GrayImage decode_region(std::pair<uint32_t, uint32_t> dimensions, size_t levels, const Grid& grid,
                            uint32_t scale_log2, const hgi_rect_t* region = nullptr)
    {
        if (grid.buffer.size() != (size_t)dimensions.first * dimensions.second)
            throw Error(HGI_ERR_INVALID_ARG, "Decoder::decode_region");
        hgi_region_plan_t plan;
        check(hgi_plan_region(dimensions.first, dimensions.second, (uint32_t)levels, scale_log2, region, &plan),
              "hgi_plan_region");
        GrayImage image(region ? region->width : plan.scaled_width, region ? region->height : plan.scaled_height,
                        GrayImage::Uninitialized{});
        const hgi_params_t p{(uint32_t)levels, I::id, HGI_QUANT_NOOP, 0};
        check(hgi_decode_region_u8(ctx_->get(), grid.buffer.data(), dimensions.first, dimensions.second, &p, scale_log2,
                                   region, image.data.data()),
              "hgi_decode_region_u8");
        return image;
    }
private:
    std::shared_ptr<Context> ctx_;
};

// The GPUs of one box behind one handle (hgi_pool_t, SURVEY.md 8e): by image for batches, by row band for one
// huge plane.  Results are byte-identical to a single context.
class Pool {
public:
    // devices: CUDA ordinals (a device may be listed more than once); empty = every sm_100 device of the box
    explicit Pool(const std::vector<int>& devices = {})
    {
        check(hgi_pool_create(devices.empty() ? nullptr : devices.data(), (int)devices.size(), &pool_), "hgi_pool_create");
    }
    ~Pool() { hgi_pool_destroy(pool_); }
    Pool(const Pool&) = delete;
    Pool& operator=(const Pool&) = delete;
    int size() const { return hgi_pool_size(pool_); }
    hgi_pool_t* get() const { return pool_; }

    // `n` planes of width x height back to back in `images`; member k takes the k-th contiguous share
    template <class I, class Q>
    Bytes encode_batch(I, const Q& quantizator, size_t scale_level, const Bytes& images, uint32_t n, uint32_t width, uint32_t height)
    {
        if (images.size() != (size_t)n * width * height) throw Error(HGI_ERR_INVALID_ARG, "Pool::encode_batch");
        Bytes grids(images.size());
        const hgi_params_t p{(uint32_t)scale_level, I::id, Q::kind, (int32_t)quantizator.level()};
        check(hgi_pool_encode_batch_u8(pool_, images.data(), n, width, height, &p, grids.data(), nullptr), "hgi_pool_encode_batch_u8");
        return grids;
    }
    template <class I>
    Bytes decode_batch(I, size_t levels, const Bytes& grids, uint32_t n, uint32_t width, uint32_t height)
    {
        if (grids.size() != (size_t)n * width * height) throw Error(HGI_ERR_INVALID_ARG, "Pool::decode_batch");
        Bytes images(grids.size());
        const hgi_params_t p{(uint32_t)levels, I::id, HGI_QUANT_NOOP, 0};
        check(hgi_pool_decode_batch_u8(pool_, grids.data(), n, width, height, &p, images.data()), "hgi_pool_decode_batch_u8");
        return images;
    }
    // ONE plane cut into row bands (multiples of 2^scale_level rows + 2^scale_level + 1 overlap rows, no exchange)
    template <class I, class Q>
    Grid encode_plane(I, const Q& quantizator, size_t scale_level, const GrayImage& input)
    {
        Grid grid;
        grid.width = input.width;
        grid.buffer.resize(input.data.size());
        const hgi_params_t p{(uint32_t)scale_level, I::id, Q::kind, (int32_t)quantizator.level()};
        check(hgi_pool_encode_plane_u8(pool_, input.data.data(), input.width, input.height, &p, grid.buffer.data()),
              "hgi_pool_encode_plane_u8");
        return grid;
    }
    template <class I>
    GrayImage decode_plane(I, std::pair<uint32_t, uint32_t> dimensions, size_t levels, const Grid& grid)
    {
        GrayImage image(dimensions.first, dimensions.second, GrayImage::Uninitialized{});
        if (grid.buffer.size() != image.data.size()) throw Error(HGI_ERR_INVALID_ARG, "Pool::decode_plane");
        const hgi_params_t p{(uint32_t)levels, I::id, HGI_QUANT_NOOP, 0};
        check(hgi_pool_decode_plane_u8(pool_, grid.buffer.data(), image.width, image.height, &p, image.data.data()),
              "hgi_pool_decode_plane_u8");
        return image;
    }
private:
    hgi_pool_t* pool_ = nullptr;
};

// src/archive.rs:15-22
struct Metadata {
    QuantizationLevel quantization_level = QuantizationLevel::Lossless;
    InterpolationType interpolation = InterpolationType::Crossed;
    uint32_t width = 0, height = 0;
    size_t scale_level = 0;
    bool operator==(const Metadata& o) const
    {
        return quantization_level == o.quantization_level && interpolation == o.interpolation && width == o.width &&
               height == o.height && scale_level == o.scale_level;
    }
};

// src/archive.rs:24-55
struct Archive {
    Metadata metadata;
    Grid grid;
    bool operator==(const Archive& o) const { return metadata == o.metadata && grid == o.grid; }

    // The same container with the fast entropy stage: literals + distance-1 matches, token tables built on the GPU
    // (hgi_rle_histogram_u8), bit-packed on the host (hgi_archive_serialize_rle).  Any inflate reads it.
    void serialize_to_writer_rle(std::ostream& w, const std::shared_ptr<Context>& ctx = Context::shared()) const
    {
        const hgi_metadata_t m{(uint32_t)metadata.quantization_level, (uint32_t)metadata.interpolation,
                               metadata.width, metadata.height, (uint64_t)metadata.scale_level};
        std::vector<uint32_t> table(HGI_RLE_TABLE_SYMBOLS);
        const size_t n = grid.buffer.size();
        check(hgi_rle_histogram_u8(ctx->get(), grid.buffer.data(), n, n ? n : 1, 1, table.data()), "hgi_rle_histogram_u8");
        std::vector<uint8_t> out(hgi_archive_huffman_bound(n, 1));
        size_t len = 0;
        check(hgi_archive_serialize_rle(&m, grid.buffer.data(), n, grid.width, table.data(), 1, n ? n : 1, out.data(), out.size(), &len),
              "hgi_archive_serialize_rle");
        w.write(reinterpret_cast<const char*>(out.data()), (std::streamsize)len);
    }

    void serialize_to_writer(std::ostream& w) const
    {
        const hgi_metadata_t m{(uint32_t)metadata.quantization_level, (uint32_t)metadata.interpolation,
                               metadata.width, metadata.height, (uint64_t)metadata.scale_level};
        std::vector<uint8_t> out(hgi_archive_bound(grid.buffer.size()));
        size_t n = 0;
        check(hgi_archive_serialize(&m, grid.buffer.data(), grid.buffer.size(), grid.width, out.data(), out.size(), &n),
              "hgi_archive_serialize");
        w.write(reinterpret_cast<const char*>(out.data()), (std::streamsize)n);
    }

    static Archive deserialize_from_reader(std::istream& r)
    {
        const std::vector<uint8_t> data((std::istreambuf_iterator<char>(r)), std::istreambuf_iterator<char>());
        hgi_metadata_t m{};
        check(hgi_archive_read_header(data.data(), data.size(), &m), "hgi_archive_read_header");
        size_t glen = 0;
        uint64_t gw = 0;
        const int rc = hgi_archive_read_grid(data.data(), data.size(), nullptr, 0, &glen, &gw);
        if (rc != HGI_OK && rc != HGI_ERR_BUFFER_TOO_SMALL) throw Error(rc, "hgi_archive_read_grid");
        Archive a;
        a.grid.buffer.resize(glen);
        check(hgi_archive_read_grid(data.data(), data.size(), a.grid.buffer.data(), glen, &glen, &gw),
              "hgi_archive_read_grid");
        a.grid.width = (size_t)gw;
        a.metadata = Metadata{(QuantizationLevel)m.quantization_level, (InterpolationType)m.interpolation, m.width,
                              m.height, (size_t)m.scale_level};
        return a;
    }
};

}  // namespace hgi
