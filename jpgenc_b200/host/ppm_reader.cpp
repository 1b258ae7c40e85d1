#include "ppm_reader.hpp"

#include <cctype>
#include <cstdio>
#include <cstring>

#include "../../include/jpgenc_b200.h"

namespace jpgenc {
namespace {

// Token scanner with the reference's rules (PPMFileBuffer::read_word, src/Image.cpp:349-374):
//  - leading whitespace is skipped; a token ends at the first whitespace byte, which is consumed;
//  - '#' discards the rest of the line AND restarts the token at the next line;
//  - at end of file the pending bytes form the last token.
class Scanner {
public:
    Scanner(const uint8_t* p, size_t n, size_t at) : p_(p), n_(n), at_(at) {}
    size_t position() const { return at_; }
    bool exhausted() const { return at_ >= n_; }

    // token bounds [begin, end)
    void token(size_t* begin, size_t* end) {
        int ch = take();
        if (std::isspace(ch)) {
            while (at_ < n_ && std::isspace(p_[at_])) ++at_;
            ch = take();
        }
        size_t start = at_ - 1;
        while (true) {
            if (ch == '#') {
                while (at_ < n_) if (p_[at_++] == '\n') break;
                start = at_;
            } else if (std::isspace(ch)) {
                *begin = start; *end = at_ - 1;
                return;
            } else if (at_ >= n_) {
                *begin = start; *end = at_ < n_ ? at_ : n_;
                return;
            }
            ch = take();
        }
    }

private:
    int take() {
        const int ch = at_ < n_ ? p_[at_] : 0;
        ++at_;
        return ch;
    }
    const uint8_t* p_;
    size_t n_, at_;
};

// std::stoi on the header words: optional sign, digits; anything else is a format error here
bool header_number(const uint8_t* p, size_t b, size_t e, uint32_t* out) {
    if (b >= e) return false;
    uint64_t v = 0;
    size_t i = b;
    if (p[i] == '+') ++i;
    if (i >= e || !std::isdigit(p[i])) return false;
    for (; i < e && std::isdigit(p[i]); ++i) {
        v = v * 10 + (p[i] - '0');
        if (v > 0x7fffffffu) return false;
    }
    *out = static_cast<uint32_t>(v);
    return true;
}

}  // namespace

int parse_ppm_header(const uint8_t* file, size_t n, PpmHeader* h) {
    Scanner sc(file, n, 0);
    size_t b, e;
    sc.token(&b, &e);
    if (e - b != 2 || e > n || file[b] != 'P' || (file[b + 1] != '3' && file[b + 1] != '6')) return JPGENC_ERR_FORMAT;
    h->magic = file[b + 1] - '0';
    sc.token(&b, &e);
    if (e > n || !header_number(file, b, e, &h->width)) return JPGENC_ERR_FORMAT;
    sc.token(&b, &e);
    if (e > n || !header_number(file, b, e, &h->height)) return JPGENC_ERR_FORMAT;
    sc.token(&b, &e);
    if (e > n || !header_number(file, b, e, &h->maxval)) return JPGENC_ERR_FORMAT;
    // the reference asserts max_color < 256 ("Only 1 byte colors supported", src/Image.cpp:462)
    if (h->width == 0 || h->height == 0 || h->maxval == 0 || h->maxval > 255) return JPGENC_ERR_FORMAT;
    h->payload = sc.position();
    return h->payload <= n ? JPGENC_OK : JPGENC_ERR_FORMAT;
}

bool samples_within_maxval(const uint8_t* px, size_t count, uint32_t maxval) {
    if (maxval >= 255) return true;
    uint8_t over = 0;
    for (size_t i = 0; i < count; ++i) over |= static_cast<uint8_t>(px[i] > maxval);
    return over == 0;
}

bool samples_within_maxval(const uint8_t* px, uint32_t w, uint32_t h, size_t pitch, uint32_t bpp, uint32_t maxval) {
    if (maxval >= 255) return true;
    if (bpp == 3 || bpp == 1) {
        for (uint32_t y = 0; y < h; ++y)
            if (!samples_within_maxval(px + y * pitch, static_cast<size_t>(w) * bpp, maxval)) return false;
        return true;
    }
    uint8_t over = 0;
    for (uint32_t y = 0; y < h; ++y) {
        const uint8_t* row = px + y * pitch;
        for (uint32_t x = 0; x < w; ++x)
            over |= static_cast<uint8_t>(row[x * bpp] > maxval) | static_cast<uint8_t>(row[x * bpp + 1] > maxval) |
                    static_cast<uint8_t>(row[x * bpp + 2] > maxval);
    }
    return over == 0;
}

int ppm_samples(const uint8_t* file, size_t n, const PpmHeader& h, std::vector<uint8_t>* storage, const uint8_t** view) {
    const size_t count = static_cast<size_t>(h.width) * h.height * 3;
    if (h.magic == 6) {                                         // loadP6PPM, src/Image.cpp:411-418
        if (h.payload + count > n) return JPGENC_ERR_FORMAT;
        *view = file + h.payload;
        return samples_within_maxval(*view, count, h.maxval) ? JPGENC_OK : JPGENC_ERR_FORMAT;
    }
    storage->resize(count);                                     // loadP3PPM, src/Image.cpp:393-408
    Scanner sc(file, n, h.payload);
    for (size_t i = 0; i < count; ++i) {
        if (sc.exhausted()) return JPGENC_ERR_FORMAT;
        size_t b, e;
        sc.token(&b, &e);
        unsigned v = 0;                                         // fast_atoi: no checks at all (src/Image.cpp:327-333)
        for (size_t k = b; k < e && k < n; ++k) v = v * 10 + (file[k] - '0');
        // a sample above maxval is not an image the 8-bit device path is exact for (the FP32 trust thresholds of K1 assume
        // scaled samples of at most 255): refused, like a truncated file, instead of being encoded differently from the reference
        if (v > h.maxval) return JPGENC_ERR_FORMAT;
        (*storage)[i] = static_cast<uint8_t>(v);
    }
    *view = storage->data();
    return JPGENC_OK;
}

int slurp_file(const std::string& path, std::vector<uint8_t>* out) {
    std::FILE* f = std::fopen(path.c_str(), "rb");
    if (!f) return JPGENC_ERR_IO;
    std::fseek(f, 0, SEEK_END);
    const long sz = std::ftell(f);
    std::fseek(f, 0, SEEK_SET);
    out->resize(sz > 0 ? static_cast<size_t>(sz) : 0);
    const size_t got = out->empty() ? 0 : std::fread(out->data(), 1, out->size(), f);
    std::fclose(f);
    return got == out->size() ? JPGENC_OK : JPGENC_ERR_IO;
}

}  // namespace jpgenc
