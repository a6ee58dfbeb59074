// png_io.cpp — minimal PNG reader/writer on top of zlib (libpng is not in the image).
// Reader: what ImageTexture::new needs (src/math/texture.rs:69-75 decodes via the `image`
// crate and converts to RGBA8): 8/16-bit gray, gray+alpha, RGB, RGBA and 8-bit palette,
// non-interlaced. Writer: image::save_buffer(.., ColorType::Rgba8) of src/main.rs:231.
// Also the PFM writer of the linear beauty and the feature buffers (rtx_pfm_write), and the PFM and Radiance .hdr
// readers of environment maps (rtx_pfm_read, rtx_hdr_read).
#include <zlib.h>

#include <algorithm>
#include <cmath>
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

// ---- readers of environment maps ----
static bool slurp(const char* path, std::vector<uint8_t>& file, std::string& err) {
    FILE* f = std::fopen(path, "rb");
    if (!f) { err = std::string("cannot open ") + path; return false; }
    uint8_t buf[1 << 16];
    size_t n;
    while ((n = std::fread(buf, 1, sizeof(buf), f)) > 0) file.insert(file.end(), buf, buf + n);
    std::fclose(f);
    return true;
}
static bool is_space(uint8_t c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r'; }
// The next whitespace-delimited token of at most 63 characters starting at or after pos; false at the end of the file.
static bool next_token(const std::vector<uint8_t>& f, size_t& pos, std::string& tok) {
    while (pos < f.size() && is_space(f[pos])) ++pos;
    tok.clear();
    while (pos < f.size() && !is_space(f[pos]) && tok.size() < 64) tok.push_back((char)f[pos++]);
    return !tok.empty() && tok.size() < 64;
}
static bool parse_dim(const std::string& t, int& v) {
    char* end = nullptr;
    const long long x = std::strtoll(t.c_str(), &end, 10);
    if (*end != 0 || t.empty() || x < 1 || x > 0x7fffffff) return false;
    v = (int)x;
    return true;
}

// "PF" (RGB) or "Pf" (grey), "width height", the scale (negative: little-endian samples, positive: big-endian), one
// whitespace character, then the rows bottom-up.
int pfm_read(const char* path, int& width, int& height, int& channels, std::vector<float>& data, std::string& err) {
    std::vector<uint8_t> f;
    if (!slurp(path, f, err)) return RTX_ERR_IO;
    size_t pos = 0;
    std::string magic, ws, hs, ss;
    if (!next_token(f, pos, magic) || (magic != "PF" && magic != "Pf")) { err = "not a PFM file"; return RTX_ERR_INVALID; }
    if (!next_token(f, pos, ws) || !next_token(f, pos, hs) || !parse_dim(ws, width) || !parse_dim(hs, height)) {
        err = "bad PFM size";
        return RTX_ERR_INVALID;
    }
    char* end = nullptr;
    const double scale = next_token(f, pos, ss) ? std::strtod(ss.c_str(), &end) : 0.0;
    if (!end || *end != 0 || !(scale != 0.0) || !std::isfinite(scale)) { err = "bad PFM scale"; return RTX_ERR_INVALID; }
    if (pos >= f.size() || !is_space(f[pos])) { err = "truncated PFM header"; return RTX_ERR_INVALID; }
    ++pos;
    channels = magic == "PF" ? 3 : 1;
    const uint64_t row = (uint64_t)width * (uint64_t)channels, count = row * (uint64_t)height;
    if (count > (f.size() - pos) / 4) { err = "truncated PFM data"; return RTX_ERR_INVALID; }
    data.resize((size_t)count);
    const bool little = scale < 0.0;
    for (int y = 0; y < height; ++y) {
        const uint8_t* src = f.data() + pos + 4 * row * (uint64_t)(height - 1 - y);  // the file stores the bottom row first
        float* dst = data.data() + row * (uint64_t)y;
        for (uint64_t i = 0; i < row; ++i, src += 4) {
            const uint32_t u = little ? (uint32_t)src[0] | ((uint32_t)src[1] << 8) | ((uint32_t)src[2] << 16) | ((uint32_t)src[3] << 24)
                                      : be32(src);
            std::memcpy(dst + i, &u, 4);
        }
    }
    return RTX_OK;
}

// Radiance RGBE: "#?" header lines up to an empty line (FORMAT must be 32-bit_rle_rgbe when given), the resolution line
// "-Y H +X W" (rows top-first, columns left to right; the other seven orientations are refused), then H scanlines, each
// flat (W x RGBE) or new-style run-length encoded (2, 2, W >> 8, W & 255, then the four components one after the other,
// each as runs: a count byte c > 128 repeats the next byte c - 128 times, 1 <= c <= 128 copies c bytes). A texel is
// m * 2^(e - 136) per channel (m the mantissa byte), black when e = 0: exact in fp32.
int hdr_read(const char* path, int& width, int& height, std::vector<float>& rgb, std::string& err) {
    std::vector<uint8_t> f;
    if (!slurp(path, f, err)) return RTX_ERR_IO;
    if (f.size() < 2 || f[0] != '#' || f[1] != '?') { err = "not a Radiance HDR file"; return RTX_ERR_INVALID; }
    size_t pos = 0;
    auto line = [&](std::string& out) -> bool {  // the next line without its newline; false when the file ends first
        out.clear();
        while (pos < f.size() && f[pos] != '\n') {
            if (out.size() < 256) out.push_back((char)f[pos]);
            ++pos;
        }
        if (pos >= f.size()) return false;
        ++pos;
        return true;
    };
    std::string l;
    for (;;) {
        if (!line(l)) { err = "truncated HDR header"; return RTX_ERR_INVALID; }
        if (l.empty()) break;
        if (l.compare(0, 7, "FORMAT=") == 0 && l != "FORMAT=32-bit_rle_rgbe") { err = "unsupported HDR format " + l; return RTX_ERR_UNSUPPORTED; }
    }
    if (!line(l)) { err = "truncated HDR resolution line"; return RTX_ERR_INVALID; }
    char a0 = 0, a1 = 0, b0 = 0, b1 = 0;
    long long n0 = 0, n1 = 0;
    int used = 0;
    if (std::sscanf(l.c_str(), " %c%c %lld %c%c %lld %n", &a0, &a1, &n0, &b0, &b1, &n1, &used) != 6 || (size_t)used != l.size() ||
        (a0 != '-' && a0 != '+') || (b0 != '-' && b0 != '+') || !((a1 == 'Y' && b1 == 'X') || (a1 == 'X' && b1 == 'Y')) ||
        n0 < 1 || n1 < 1 || n0 > 0x7fffffff || n1 > 0x7fffffff) {
        err = "bad HDR resolution line";
        return RTX_ERR_INVALID;
    }
    if (a0 != '-' || a1 != 'Y' || b0 != '+' || b1 != 'X') { err = "unsupported HDR orientation " + l + " (only -Y H +X W)"; return RTX_ERR_UNSUPPORTED; }
    height = (int)n0;
    width = (int)n1;
    // the fewest bytes a scanline can take (flat, or run-length: 4 + per component 2 bytes per run of at most 127)
    const uint64_t min_scan = std::min<uint64_t>(4 * (uint64_t)width, 4 + 8 * (((uint64_t)width + 126) / 127));
    if (min_scan * (uint64_t)height > f.size() - pos) { err = "truncated HDR data"; return RTX_ERR_INVALID; }
    const size_t W = (size_t)width;
    std::vector<uint8_t> scan(4 * W);
    rgb.resize(3 * W * (size_t)height);
    for (int y = 0; y < height; ++y) {
        const bool rle = W >= 8 && W < 32768 && pos + 4 <= f.size() && f[pos] == 2 && f[pos + 1] == 2 && ((size_t)f[pos + 2] << 8 | f[pos + 3]) == W;
        if (rle) {
            pos += 4;
            for (int c = 0; c < 4; ++c) {
                for (size_t x = 0; x < W;) {
                    if (pos >= f.size()) { err = "truncated HDR scanline"; return RTX_ERR_INVALID; }
                    size_t n = f[pos++];
                    if (n > 128) {
                        n -= 128;
                        if (pos >= f.size() || n > W - x) { err = "bad HDR run"; return RTX_ERR_INVALID; }
                        for (size_t k = 0; k < n; ++k) scan[4 * (x + k) + (size_t)c] = f[pos];
                        ++pos;
                    } else {
                        if (n == 0 || n > W - x || n > f.size() - pos) { err = "bad HDR run"; return RTX_ERR_INVALID; }
                        for (size_t k = 0; k < n; ++k) scan[4 * (x + k) + (size_t)c] = f[pos + k];
                        pos += n;
                    }
                    x += n;
                }
            }
        } else {
            if (4 * W > f.size() - pos) { err = "truncated HDR scanline"; return RTX_ERR_INVALID; }
            std::memcpy(scan.data(), f.data() + pos, 4 * W);
            pos += 4 * W;
        }
        float* out = rgb.data() + 3 * W * (size_t)y;
        for (size_t x = 0; x < W; ++x) {
            const uint8_t* p = &scan[4 * x];
            for (int c = 0; c < 3; ++c) out[3 * x + (size_t)c] = p[3] == 0 ? 0.f : std::ldexp((float)p[c], (int)p[3] - 136);
        }
    }
    return RTX_OK;
}

}  // namespace rttnw
