// PPM (P3/P6) front end of the encode path: header + sample extraction with the reference's parsing rules
// (src/Image.cpp:334-473).  Only raw 8-bit samples are produced; scaling by 255/maxval and padding to multiples
// of 16 happen on the GPU.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

namespace jpgenc {

struct PpmHeader {
    int magic = 0;                 // 3 or 6
    uint32_t width = 0, height = 0, maxval = 0;
    size_t payload = 0;            // offset of the first sample
};

// 0 on success; JPGENC_ERR_FORMAT when the magic is not P3/P6 or the header is unusable
int parse_ppm_header(const uint8_t* file, size_t n, PpmHeader* h);
// samples -> interleaved u8 RGB.  P6: `*view` points into `file` (no copy); P3: decoded into `storage`.
int ppm_samples(const uint8_t* file, size_t n, const PpmHeader& h, std::vector<uint8_t>* storage, const uint8_t** view);
// false when a sample exceeds maxval (< 255): such a file is refused (JPGENC_ERR_FORMAT) -- the reference would scale the sample past 255,
// which the 8-bit device path is not exact for; jpgenc_encode_planes takes such data as planes of doubles
bool samples_within_maxval(const uint8_t* px, size_t count, uint32_t maxval);
// the same for h rows of w pixels, `pitch` bytes apart, `bpp` bytes per pixel of which the first three are colour (bpp 1: a grey
// pixel or one plane of planar RGB): a 4th byte and the bytes between rows are not samples and are not read
bool samples_within_maxval(const uint8_t* px, uint32_t w, uint32_t h, size_t pitch, uint32_t bpp, uint32_t maxval);
// whole file into memory; JPGENC_ERR_IO when it cannot be opened
int slurp_file(const std::string& path, std::vector<uint8_t>* out);

}  // namespace jpgenc
