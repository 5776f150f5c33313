// png_io.cpp — minimal PNG reader/writer for the host scene layer (system zlib for inflate/deflate).
//
// Covers what the reference's RTexture::LoadTexturePNG accepts (Texture.cpp:97: colour type 2 or 6
// at 8 bits per channel) and what SaveBufferToPNG writes (Texture.cpp:201-283: 8-bit RGB).  The
// reference goes through vendored libpng; here the container format is parsed directly: chunk
// walk, one inflate over the concatenated IDAT payload, then per-scanline filter reversal.
// Adam7-interlaced files are rejected (none of the reference's assets are interlaced).
#include "rt_host.hpp"

#include <stdio.h>
#include <string.h>
#include <math.h>
#include <zlib.h>

namespace rtb200 {

static uint32_t be32(const uint8_t* p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }

static inline int paeth(int a, int b, int c)
{
    int p = a + b - c;
    int pa = p > a ? p - a : a - p;
    int pb = p > b ? p - b : b - p;
    int pc = p > c ? p - c : c - p;
    if (pa <= pb && pa <= pc) return a;
    return pb <= pc ? b : c;
}

bool DecodePng8(const std::string& Filename, int& Width, int& Height, int& Channels,
                std::vector<uint8_t>& Pixels, std::string& Error)
{
    FILE* f = fopen(Filename.c_str(), "rb");
    if (!f) { Error = "File could not be opened for reading: " + Filename; return false; }
    std::vector<uint8_t> file;
    uint8_t buf[1 << 16];
    size_t n;
    while ((n = fread(buf, 1, sizeof buf, f)) > 0) file.insert(file.end(), buf, buf + n);
    fclose(f);

    static const uint8_t sig[8] = { 0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a };
    if (file.size() < 8 || memcmp(file.data(), sig, 8) != 0) { Error = "File is not recognized as a PNG file: " + Filename; return false; }

    std::vector<uint8_t> idat;
    bool have_ihdr = false;
    int bit_depth = 0, color_type = 0, interlace = 0;
    size_t pos = 8;
    while (pos + 12 <= file.size())
    {
        uint32_t len = be32(&file[pos]);
        const uint8_t* type = &file[pos + 4];
        if (pos + 12 + (size_t)len > file.size()) { Error = "truncated PNG chunk: " + Filename; return false; }
        const uint8_t* data = &file[pos + 8];
        if (!memcmp(type, "IHDR", 4) && len >= 13)
        {
            Width = (int)be32(data); Height = (int)be32(data + 4);
            bit_depth = data[8]; color_type = data[9]; interlace = data[12];
            have_ihdr = true;
        }
        else if (!memcmp(type, "IDAT", 4)) idat.insert(idat.end(), data, data + len);
        else if (!memcmp(type, "IEND", 4)) break;
        pos += 12 + (size_t)len;
    }
    if (!have_ihdr || Width <= 0 || Height <= 0) { Error = "missing IHDR: " + Filename; return false; }
    // a header can declare anything: refuse before sizing buffers from it (the atlas caps at 131072 x 65536 anyway)
    if ((unsigned long long)Width * (unsigned long long)Height > (1ull << 28)) { Error = "PNG too large (more than 2^28 pixels): " + Filename; return false; }
    if (!((color_type == 2 || color_type == 6) && bit_depth == 8))
    {
        char msg[128];
        snprintf(msg, sizeof msg, "Not an implemented png format (color type = %d, bit depth = %d): ", color_type, bit_depth);
        Error = msg + Filename;
        return false;
    }
    if (interlace != 0) { Error = "interlaced PNG not supported: " + Filename; return false; }

    Channels = color_type == 2 ? 3 : 4;
    const size_t stride = (size_t)Width * Channels;
    std::vector<uint8_t> raw((stride + 1) * (size_t)Height);
    uLongf raw_len = (uLongf)raw.size();
    int zr = uncompress(raw.data(), &raw_len, idat.data(), (uLong)idat.size());
    if (zr != Z_OK || raw_len != raw.size()) { Error = "Error during read_image: " + Filename; return false; }

    Pixels.resize(stride * (size_t)Height);
    const int bpp = Channels;
    for (int y = 0; y < Height; y++)
    {
        const uint8_t* in = &raw[(stride + 1) * (size_t)y];
        uint8_t* out = &Pixels[stride * (size_t)y];
        const uint8_t* up = y ? out - stride : nullptr;
        const int filter = in[0];
        in++;
        for (size_t i = 0; i < stride; i++)
        {
            int a = i >= (size_t)bpp ? out[i - bpp] : 0;
            int b = up ? up[i] : 0;
            int c = (up && i >= (size_t)bpp) ? up[i - bpp] : 0;
            int v = in[i];
            switch (filter)
            {
            case 0: break;
            case 1: v += a; break;
            case 2: v += b; break;
            case 3: v += (a + b) >> 1; break;
            case 4: v += paeth(a, b, c); break;
            default: Error = "bad PNG filter: " + Filename; return false;
            }
            out[i] = (uint8_t)v;
        }
    }
    return true;
}

std::unique_ptr<RTexture> RTexture::LoadTexturePNG(const std::string& Filename)
{
    int w, h, ch;
    std::vector<uint8_t> px;
    std::string err;
    if (!DecodePng8(Filename, w, h, ch, px, err))
    {
        printf("%s\n", err.c_str());
        return nullptr;
    }
    std::unique_ptr<RTexture> t(new RTexture());
    MakeLut(t->Lut);
    t->Width = w; t->Height = h; t->Channels = ch;
    t->Pixels8 = std::move(px);
    return t;
}

// Linearise once per 8-bit code instead of once per texel: powf((float)c / 255, 2.2f) only
// ever sees 256 inputs, so a table gives the same bits as Texture.cpp:128-131 / ColorBuffer.h:70-78.
void RTexture::MakeLut(float* Out512)
{
    for (int i = 0; i < 256; i++)
    {
        float c = (float)i / 255;
        Out512[i] = powf(c, 2.2f);
        Out512[256 + i] = c;
    }
}

void RTexture::ExpandTo(float* OutRGBA) const
{
    const size_t count = (size_t)Width * Height;
    for (size_t i = 0; i < count; i++)
    {
        const uint8_t* p = &Pixels8[i * Channels];
        float* o = OutRGBA + 4 * i;
        o[0] = Lut[p[0]]; o[1] = Lut[p[1]]; o[2] = Lut[p[2]];
        o[3] = Channels == 4 ? Lut[256 + p[3]] : 1.0f;
    }
}

static void put_chunk(FILE* f, const char* type, const uint8_t* data, uint32_t len)
{
    uint8_t hdr[8] = { (uint8_t)(len >> 24), (uint8_t)(len >> 16), (uint8_t)(len >> 8), (uint8_t)len,
                       (uint8_t)type[0], (uint8_t)type[1], (uint8_t)type[2], (uint8_t)type[3] };
    fwrite(hdr, 1, 8, f);
    if (len) fwrite(data, 1, len, f);
    uLong crc = crc32(0L, hdr + 4, 4);
    if (len) crc = crc32(crc, data, len);
    uint8_t c[4] = { (uint8_t)(crc >> 24), (uint8_t)(crc >> 16), (uint8_t)(crc >> 8), (uint8_t)crc };
    fwrite(c, 1, 4, f);
}

// 8-bit RGB PNG from an ARGB buffer (red = bits 16-23: the non-OSX packing of ColorBuffer.h:34-41).
bool WritePngARGB(const std::string& Filename, const uint32_t* Pixels, int Width, int Height)
{
    FILE* f = fopen(Filename.c_str(), "wb");
    if (!f) return false;
    static const uint8_t sig[8] = { 0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a };
    fwrite(sig, 1, 8, f);
    uint8_t ihdr[13] = { (uint8_t)(Width >> 24), (uint8_t)(Width >> 16), (uint8_t)(Width >> 8), (uint8_t)Width,
                         (uint8_t)(Height >> 24), (uint8_t)(Height >> 16), (uint8_t)(Height >> 8), (uint8_t)Height,
                         8, 2, 0, 0, 0 };
    put_chunk(f, "IHDR", ihdr, 13);
    const size_t stride = (size_t)Width * 3 + 1;
    std::vector<uint8_t> raw(stride * (size_t)Height);
    for (int y = 0; y < Height; y++)
    {
        uint8_t* row = &raw[stride * (size_t)y];
        row[0] = 0;
        for (int x = 0; x < Width; x++)
        {
            uint32_t c = Pixels[(size_t)y * Width + x];
            row[1 + 3 * x] = (uint8_t)(c >> 16);
            row[2 + 3 * x] = (uint8_t)(c >> 8);
            row[3 + 3 * x] = (uint8_t)c;
        }
    }
    uLongf zlen = compressBound((uLong)raw.size());
    std::vector<uint8_t> z(zlen);
    bool ok = compress2(z.data(), &zlen, raw.data(), (uLong)raw.size(), 6) == Z_OK;
    if (ok) put_chunk(f, "IDAT", z.data(), (uint32_t)zlen);
    put_chunk(f, "IEND", nullptr, 0);
    fclose(f);
    return ok;
}

} // namespace rtb200
