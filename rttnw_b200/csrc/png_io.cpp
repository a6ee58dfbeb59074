// png_io.cpp — minimal PNG reader/writer on top of zlib (libpng is not in the image).
// Reader: what ImageTexture::new needs (src/math/texture.rs:69-75 decodes via the `image`
// crate and converts to RGBA8): 8/16-bit gray, gray+alpha, RGB, RGBA and 8-bit palette,
// non-interlaced. Writer: image::save_buffer(.., ColorType::Rgba8) of src/main.rs:231.
// Also the PFM writer of the linear beauty and the feature buffers (rtx_pfm_write).
#include <zlib.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "scene_api.hpp"

namespace rttnw {

static uint32_t be32(const uint8_t* p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }
static void put32(uint8_t* p, uint32_t v) { p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v; }
static int paeth(int a, int b, int c) {
    int p = a + b - c, pa = std::abs(p - a), pb = std::abs(p - b), pc = std::abs(p - c);
    if (pa <= pb && pa <= pc) return a;
    return pb <= pc ? b : c;
}

bool png_read_rgba8(const char* path, int& width, int& height, std::vector<uint8_t>& rgba, std::string& err) {
    FILE* f = std::fopen(path, "rb");
    if (!f) { err = std::string("cannot open ") + path; return false; }
    std::vector<uint8_t> file;
    uint8_t buf[1 << 16];
    size_t n;
    while ((n = std::fread(buf, 1, sizeof(buf), f)) > 0) file.insert(file.end(), buf, buf + n);
    std::fclose(f);
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
    if (file.size() < 8 || std::memcmp(file.data(), sig, 8) != 0) { err = "not a PNG file"; return false; }
    size_t pos = 8;
    uint32_t w = 0, h = 0;
    int depth = 0, ctype = -1, interlace = 0;
    std::vector<uint8_t> idat, palette, trns;
    bool seen_end = false;
    while (pos + 12 <= file.size() && !seen_end) {
        uint32_t len = be32(&file[pos]);
        const uint8_t* type = &file[pos + 4];
        if (pos + 12 + (size_t)len > file.size()) { err = "truncated PNG chunk"; return false; }
        const uint8_t* data = &file[pos + 8];
        uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), type, 4 + len);
        if (crc != be32(&file[pos + 8 + len])) { err = "PNG chunk CRC mismatch"; return false; }
        if (!std::memcmp(type, "IHDR", 4)) {
            if (len < 13) { err = "bad IHDR"; return false; }
            w = be32(data); h = be32(data + 4);
            depth = data[8]; ctype = data[9]; interlace = data[12];
        } else if (!std::memcmp(type, "PLTE", 4)) {
            palette.assign(data, data + len);
        } else if (!std::memcmp(type, "tRNS", 4)) {
            trns.assign(data, data + len);
        } else if (!std::memcmp(type, "IDAT", 4)) {
            idat.insert(idat.end(), data, data + len);
        } else if (!std::memcmp(type, "IEND", 4)) {
            seen_end = true;
        }
        pos += 12 + (size_t)len;
    }
    if (w == 0 || h == 0 || w > 65535 || h > 65535) { err = "bad PNG dimensions"; return false; }
    if (interlace != 0) { err = "interlaced PNG not supported"; return false; }
    int channels;
    switch (ctype) {
        case 0: channels = 1; break;
        case 2: channels = 3; break;
        case 3: channels = 1; break;
        case 4: channels = 2; break;
        case 6: channels = 4; break;
        default: err = "unsupported PNG colour type"; return false;
    }
    if (!(depth == 8 || (depth == 16 && ctype != 3))) { err = "unsupported PNG bit depth"; return false; }
    size_t bpp = (size_t)channels * (size_t)(depth / 8);
    size_t stride = bpp * w;
    std::vector<uint8_t> raw((stride + 1) * (size_t)h);
    uLongf raw_len = (uLongf)raw.size();
    int zr = uncompress(raw.data(), &raw_len, idat.data(), (uLong)idat.size());
    if (zr != Z_OK || raw_len != raw.size()) { err = "PNG inflate failed"; return false; }
    // undo the per-scanline filters in place
    std::vector<uint8_t> prev(stride, 0);
    for (uint32_t y = 0; y < h; ++y) {
        uint8_t* row = &raw[(stride + 1) * (size_t)y];
        int ft = row[0];
        uint8_t* cur = row + 1;
        for (size_t i = 0; i < stride; ++i) {
            int a = i >= bpp ? cur[i - bpp] : 0, b = prev[i], c = i >= bpp ? prev[i - bpp] : 0;
            int v = cur[i];
            switch (ft) {
                case 0: break;
                case 1: v += a; break;
                case 2: v += b; break;
                case 3: v += (a + b) >> 1; break;
                case 4: v += paeth(a, b, c); break;
                default: err = "bad PNG filter type"; return false;
            }
            cur[i] = (uint8_t)v;
        }
        std::memcpy(prev.data(), cur, stride);
    }
    rgba.resize((size_t)4 * w * h);
    size_t step = (size_t)(depth / 8);  // 16-bit samples: keep the high byte
    for (uint32_t y = 0; y < h; ++y) {
        const uint8_t* cur = &raw[(stride + 1) * (size_t)y + 1];
        uint8_t* out = &rgba[(size_t)4 * w * y];
        for (uint32_t x = 0; x < w; ++x) {
            const uint8_t* p = cur + bpp * x;
            uint8_t r, g, b, a = 255;
            switch (ctype) {
                case 0: r = g = b = p[0]; break;
                case 2: r = p[0]; g = p[step]; b = p[2 * step]; break;
                case 3: {
                    size_t idx = (size_t)p[0] * 3;
                    if (idx + 2 >= palette.size()) { err = "PNG palette index out of range"; return false; }
                    r = palette[idx]; g = palette[idx + 1]; b = palette[idx + 2];
                    if ((size_t)p[0] < trns.size()) a = trns[p[0]];  // per-entry alpha
                    break;
                }
                case 4: r = g = b = p[0]; a = p[step]; break;
                default: r = p[0]; g = p[step]; b = p[2 * step]; a = p[3 * step]; break;
            }
            out[4 * x] = r; out[4 * x + 1] = g; out[4 * x + 2] = b; out[4 * x + 3] = a;
        }
    }
    width = (int)w;
    height = (int)h;
    return true;
}

static void write_chunk(std::vector<uint8_t>& out, const char* type, const uint8_t* data, size_t len) {
    uint8_t hdr[8];
    put32(hdr, (uint32_t)len);
    std::memcpy(hdr + 4, type, 4);
    out.insert(out.end(), hdr, hdr + 8);
    if (len) out.insert(out.end(), data, data + len);
    uint32_t crc = (uint32_t)crc32(0L, Z_NULL, 0);
    crc = (uint32_t)crc32(crc, (const Bytef*)type, 4);
    if (len) crc = (uint32_t)crc32(crc, data, (uInt)len);
    uint8_t c[4];
    put32(c, crc);
    out.insert(out.end(), c, c + 4);
}

bool png_write_rgba8(const char* path, int width, int height, const uint8_t* rgba, std::string& err) {
    if (width <= 0 || height <= 0 || !rgba) { err = "bad image"; return false; }
    size_t stride = (size_t)4 * width;
    std::vector<uint8_t> raw((stride + 1) * (size_t)height);
    for (int y = 0; y < height; ++y) {
        raw[(stride + 1) * (size_t)y] = 0;  // filter: None
        std::memcpy(&raw[(stride + 1) * (size_t)y + 1], rgba + stride * (size_t)y, stride);
    }
    uLongf zlen = compressBound((uLong)raw.size());
    std::vector<uint8_t> z(zlen);
    if (compress2(z.data(), &zlen, raw.data(), (uLong)raw.size(), 6) != Z_OK) { err = "deflate failed"; return false; }
    std::vector<uint8_t> out;
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
    out.insert(out.end(), sig, sig + 8);
    uint8_t ihdr[13];
    put32(ihdr, (uint32_t)width);
    put32(ihdr + 4, (uint32_t)height);
    ihdr[8] = 8; ihdr[9] = 6; ihdr[10] = 0; ihdr[11] = 0; ihdr[12] = 0;
    write_chunk(out, "IHDR", ihdr, 13);
    write_chunk(out, "IDAT", z.data(), zlen);
    write_chunk(out, "IEND", nullptr, 0);
    FILE* f = std::fopen(path, "wb");
    if (!f) { err = std::string("cannot open for writing: ") + path; return false; }
    size_t wr = std::fwrite(out.data(), 1, out.size(), f);
    std::fclose(f);
    if (wr != out.size()) { err = "short write"; return false; }
    return true;
}

// Portable float map: "PF" (RGB) or "Pf" (grey), then "width height", then the scale, negative for little-endian
// samples; the rows follow bottom-up. `data` has row 0 = top, like the accumulators.
bool pfm_write(const char* path, int width, int height, int channels, const float* data, std::string& err) {
    if (width <= 0 || height <= 0 || (channels != 1 && channels != 3) || !data) { err = "bad float map"; return false; }
    const size_t row = (size_t)width * channels;
    char hdr[64];
    int n = std::snprintf(hdr, sizeof(hdr), "%s\n%d %d\n-1.0\n", channels == 3 ? "PF" : "Pf", width, height);
    std::vector<uint8_t> out(hdr, hdr + n);
    out.reserve((size_t)n + row * 4 * (size_t)height);
    for (int y = height - 1; y >= 0; --y) {
        const float* src = data + row * (size_t)y;
        for (size_t i = 0; i < row; ++i) {
            uint32_t u;
            std::memcpy(&u, src + i, 4);
            const uint8_t b[4] = {(uint8_t)u, (uint8_t)(u >> 8), (uint8_t)(u >> 16), (uint8_t)(u >> 24)};
            out.insert(out.end(), b, b + 4);
        }
    }
    FILE* f = std::fopen(path, "wb");
    if (!f) { err = std::string("cannot open for writing: ") + path; return false; }
    size_t wr = std::fwrite(out.data(), 1, out.size(), f);
    bool ok = std::fclose(f) == 0 && wr == out.size();
    if (!ok) { err = "short write"; return false; }
    return true;
}

}  // namespace rttnw
