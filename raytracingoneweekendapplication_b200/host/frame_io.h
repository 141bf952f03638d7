// frame_io.h — linear-radiance outputs and checkpoint files of the download side.
//
// The reference writes one thing, an RGB8 PNG after sqrt gamma (Camera.txt:74-89,118), and
// restarts from sample 0 whenever it is interrupted.  SURVEY §8f rank 3 asks for the
// obvious extension on the download side of the hot path: keep the linear radiance
// (PFM, and scanline OpenEXR with 32-bit float channels, uncompressed) and make a
// progressive render resumable.  A checkpoint is the raw accumulation buffer of
// rt_accum_download (integer sums, include/rt_b200.h) behind a small header that pins
// what must not change between the two halves of a render.
#ifndef RTB200_FRAME_IO_H
#define RTB200_FRAME_IO_H
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

namespace rtb200 {

// Portable Float Map: "PF\n<w> <h>\n-1.0\n" then rows BOTTOM-UP, little-endian float RGB.
inline bool write_pfm(const char* path, int w, int h, const float* rgb) {
    std::FILE* f = std::fopen(path, "wb");
    if (!f) return false;
    std::fprintf(f, "PF\n%d %d\n-1.0\n", w, h);
    for (int y = h - 1; y >= 0; y--) std::fwrite(rgb + (size_t)y * w * 3, sizeof(float), (size_t)w * 3, f);
    return std::fclose(f) == 0;
}

namespace exr_detail {
inline void put32(std::vector<uint8_t>& o, uint32_t v) { for (int i = 0; i < 4; i++) o.push_back((uint8_t)(v >> (8 * i))); }
inline void put64(std::vector<uint8_t>& o, uint64_t v) { for (int i = 0; i < 8; i++) o.push_back((uint8_t)(v >> (8 * i))); }
inline void puts0(std::vector<uint8_t>& o, const char* s) { while (*s) o.push_back((uint8_t)*s++); o.push_back(0); }
inline void attr(std::vector<uint8_t>& o, const char* name, const char* type, const std::vector<uint8_t>& value) {
    puts0(o, name);
    puts0(o, type);
    put32(o, (uint32_t)value.size());
    o.insert(o.end(), value.begin(), value.end());
}
}  // namespace exr_detail

// OpenEXR 2.0 single-part scanline file, channels B G R (alphabetical, as the format
// requires) of type FLOAT, NO_COMPRESSION, one scanline per chunk, increasing Y.
inline bool write_exr(const char* path, int w, int h, const float* rgb) {
    using namespace exr_detail;
    std::vector<uint8_t> hd;
    put32(hd, 20000630u);  // magic
    put32(hd, 2u);         // version 2, no flags: scanline, single part, short names
    {
        std::vector<uint8_t> ch;
        for (const char* name : {"B", "G", "R"}) {
            puts0(ch, name);
            put32(ch, 2u);  // FLOAT
            ch.push_back(0); ch.push_back(0); ch.push_back(0); ch.push_back(0);  // pLinear + reserved
            put32(ch, 1u);  // xSampling
            put32(ch, 1u);  // ySampling
        }
        ch.push_back(0);
        attr(hd, "channels", "chlist", ch);
    }
    attr(hd, "compression", "compression", {0});
    {
        std::vector<uint8_t> box;
        put32(box, 0); put32(box, 0); put32(box, (uint32_t)(w - 1)); put32(box, (uint32_t)(h - 1));
        attr(hd, "dataWindow", "box2i", box);
        attr(hd, "displayWindow", "box2i", box);
    }
    attr(hd, "lineOrder", "lineOrder", {0});
    {
        std::vector<uint8_t> v;
        float one = 1.0f, zero = 0.0f;
        uint32_t u;
        std::memcpy(&u, &one, 4);
        put32(v, u);
        attr(hd, "pixelAspectRatio", "float", v);
        std::vector<uint8_t> c;
        std::memcpy(&u, &zero, 4);
        put32(c, u); put32(c, u);
        attr(hd, "screenWindowCenter", "v2f", c);
        attr(hd, "screenWindowWidth", "float", v);
    }
    hd.push_back(0);  // end of header
    const uint64_t line_bytes = (uint64_t)w * 3 * 4;
    const uint64_t table_at = hd.size(), data_at = table_at + 8ull * (uint64_t)h;
    for (int y = 0; y < h; y++) put64(hd, data_at + (uint64_t)y * (8 + line_bytes));
    std::FILE* f = std::fopen(path, "wb");
    if (!f) return false;
    std::fwrite(hd.data(), 1, hd.size(), f);
    std::vector<float> line((size_t)w * 3);
    for (int y = 0; y < h; y++) {
        int32_t head[2] = {y, (int32_t)line_bytes};
        std::fwrite(head, 4, 2, f);
        const float* src = rgb + (size_t)y * w * 3;
        for (int c = 0; c < 3; c++)  // planar per scanline: all B, then all G, then all R
            for (int x = 0; x < w; x++) line[(size_t)c * w + x] = src[(size_t)x * 3 + (2 - c)];
        std::fwrite(line.data(), 4, line.size(), f);
    }
    return std::fclose(f) == 0;
}

// ---- checkpoint ------------------------------------------------------------------------
struct checkpoint_header {
    char magic[8];         // "RTB2CKPT"
    uint32_t version;      // 1: the sums; 2: the sums, then the second moments (RT_FLAG_MOMENTS, width * height * 6 uint64)
    int32_t width, height;
    int32_t spp_done;      // samples [0, spp_done) of every pixel are in the sums
    int32_t max_depth;
    uint32_t flags;        // estimator flags of the samples in the file (RT_FLAG_NEE, RT_FLAG_SHADOWED_POINT_LIGHTS): a render
                           // with other flags is another integrand and must not continue from it
    uint64_t seed;
    uint64_t scene_hash;   // FNV-1a over the flattened scene description (0 = not checked)
};

inline uint64_t fnv1a(const void* data, size_t n, uint64_t h = 1469598103934665603ull) {
    const uint8_t* p = (const uint8_t*)data;
    for (size_t i = 0; i < n; i++) { h ^= p[i]; h *= 1099511628211ull; }
    return h;
}

inline bool write_checkpoint(const char* path, const checkpoint_header& hd, const uint64_t* sums, const uint64_t* moments = nullptr) {
    // write-then-rename so that an interruption DURING the save leaves the previous checkpoint intact
    std::string tmp = std::string(path) + ".tmp";
    std::FILE* f = std::fopen(tmp.c_str(), "wb");
    if (!f) return false;
    const size_t n = (size_t)hd.width * hd.height * 4;
    bool ok = std::fwrite(&hd, sizeof hd, 1, f) == 1 && std::fwrite(sums, 8, n, f) == n;
    if (hd.version == 2) ok = ok && moments && std::fwrite(moments, 8, n / 4 * 6, f) == n / 4 * 6;
    ok = (std::fclose(f) == 0) && ok;
    if (!ok) { std::remove(tmp.c_str()); return false; }
    return std::rename(tmp.c_str(), path) == 0;
}

inline bool read_checkpoint(const char* path, checkpoint_header& hd, std::vector<uint64_t>& sums, std::vector<uint64_t>* moments = nullptr) {
    std::FILE* f = std::fopen(path, "rb");
    if (!f) return false;
    bool ok = std::fread(&hd, sizeof hd, 1, f) == 1 && std::memcmp(hd.magic, "RTB2CKPT", 8) == 0 && (hd.version == 1 || hd.version == 2) &&
              hd.width > 0 && hd.height > 0 && hd.spp_done >= 0 && (long long)hd.width * hd.height < (1ll << 31);
    if (ok) {
        // the file must be exactly header + width * height * (32 | 80) bytes BEFORE anything is allocated from its header
        const size_t n = (size_t)hd.width * hd.height * 4, nm = hd.version == 2 ? (size_t)hd.width * hd.height * 6 : 0;
        ok = std::fseek(f, 0, SEEK_END) == 0 && (unsigned long long)std::ftell(f) == sizeof hd + 8ull * (n + nm) && std::fseek(f, (long)sizeof hd, SEEK_SET) == 0;
        if (ok) {
            sums.resize(n);
            ok = std::fread(sums.data(), 8, n, f) == n;
        }
        if (ok && moments) {
            moments->resize(nm);
            ok = std::fread(moments->data(), 8, nm, f) == nm;
        }
    }
    std::fclose(f);
    return ok;
}

}  // namespace rtb200
#endif
