// pt_png.h -- minimal PNG writer for the texture (replaces cv::imwrite("texture.png", padded),
// /root/reference src/pointsTransfer.cpp:613; OpenCV's C++ headers are absent from this image).
// 8-bit RGBA, filter 0 on every scanline, one zlib stream (deflate level 1: the 8192^2 texture is
// 256 MiB raw).  Input is B G R A as cv::Mat CV_8UC4; cv::imwrite stores such a Mat as RGBA.  The
// height map is written as 16-bit greyscale.
#pragma once
#include <zlib.h>

#include <cstdint>
#include <cstdio>
#include <vector>

namespace ptb {

inline void png_chunk(FILE *f, const char type[4], const uint8_t *data, uint32_t len)
{
    uint8_t hdr[8] = {(uint8_t)(len >> 24), (uint8_t)(len >> 16), (uint8_t)(len >> 8), (uint8_t)len,
                      (uint8_t)type[0], (uint8_t)type[1], (uint8_t)type[2], (uint8_t)type[3]};
    fwrite(hdr, 1, 8, f);
    if (len) fwrite(data, 1, len, f);
    uLong crc = crc32(0L, hdr + 4, 4);
    if (len) crc = crc32(crc, data, len);
    const uint8_t c[4] = {(uint8_t)(crc >> 24), (uint8_t)(crc >> 16), (uint8_t)(crc >> 8), (uint8_t)crc};
    fwrite(c, 1, 4, f);
}

// One PNG of `height` rows of `row_bytes` bytes each, which fill_row(y, dst) writes: filter 0 on
// every scanline, one zlib stream at deflate level 1.
template <typename FillRow>
inline bool write_png_rows(const char *path, int width, int height, uint8_t bit_depth, uint8_t colour_type,
                           size_t row_bytes, FillRow fill_row)
{
    FILE *f = fopen(path, "wb");
    if (!f) return false;
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
    fwrite(sig, 1, 8, f);
    const uint8_t ihdr[13] = {(uint8_t)(width >> 24), (uint8_t)(width >> 16), (uint8_t)(width >> 8), (uint8_t)width,
                              (uint8_t)(height >> 24), (uint8_t)(height >> 16), (uint8_t)(height >> 8), (uint8_t)height,
                              bit_depth, colour_type, 0, 0, 0};
    png_chunk(f, "IHDR", ihdr, 13);
    z_stream z{};
    if (deflateInit(&z, 1) != Z_OK) { fclose(f); return false; }
    std::vector<uint8_t> row(row_bytes + 1), out(1 << 20);
    bool ok = true;
    for (int y = 0; y < height && ok; ++y) {
        row[0] = 0;                                  // filter: none
        fill_row(y, row.data() + 1);
        z.next_in = row.data();
        z.avail_in = (uInt)row.size();
        const int flush = y + 1 == height ? Z_FINISH : Z_NO_FLUSH;
        do {
            z.next_out = out.data();
            z.avail_out = (uInt)out.size();
            const int r = deflate(&z, flush);
            if (r == Z_STREAM_ERROR) { ok = false; break; }
            const size_t have = out.size() - z.avail_out;
            if (have) png_chunk(f, "IDAT", out.data(), (uint32_t)have);
        } while (z.avail_out == 0 || (flush == Z_FINISH && z.avail_in));
    }
    deflateEnd(&z);
    png_chunk(f, "IEND", nullptr, 0);
    ok = ok && fclose(f) == 0;
    return ok;
}

inline bool write_png_bgra(const char *path, const uint8_t *bgra, int width, int height)
{
    // 8 bit, colour type 6 = RGBA
    return write_png_rows(path, width, height, 8, 6, (size_t)width * 4, [&](int y, uint8_t *dst) {
        const uint8_t *src = bgra + (size_t)y * width * 4;
        for (int x = 0; x < width; ++x) {
            dst[4 * x] = src[4 * x + 2];
            dst[4 * x + 1] = src[4 * x + 1];
            dst[4 * x + 2] = src[4 * x];
            dst[4 * x + 3] = src[4 * x + 3];
        }
    });
}

// 16-bit greyscale (colour type 0), samples big-endian as PNG stores them
inline bool write_png_gray16(const char *path, const uint16_t *v, int width, int height)
{
    return write_png_rows(path, width, height, 16, 0, (size_t)width * 2, [&](int y, uint8_t *dst) {
        const uint16_t *src = v + (size_t)y * width;
        for (int x = 0; x < width; ++x) {
            dst[2 * x] = (uint8_t)(src[x] >> 8);
            dst[2 * x + 1] = (uint8_t)src[x];
        }
    });
}

}  // namespace ptb
