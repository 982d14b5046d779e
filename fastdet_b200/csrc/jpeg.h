// jpeg.h — baseline-JPEG front end of perform(): replaces `Image.open(io.BytesIO(data))` + `np.array(img)`
// (reference server/detector.py:128-133), i.e. what libjpeg(-turbo) does behind PIL with its default settings
// (ISLOW integer IDCT, "fancy" triangle chroma upsampling, 16.16 fixed-point YCbCr -> RGB).
//
// Split of the work:
//   host  : marker parse + Huffman entropy decode -> quantised DCT coefficients (int16, natural order), one
//           frame per pool thread (jpeg_parse / jpeg_decode_coefficients, JpegPool)
//   device: de-quantise + IDCT -> component planes (jpeg_idct_kernel), then chroma upsample + colour
//           conversion -> RGB u8 HWC written straight into the batch's input tensor (jpeg_rgb_kernel)
// Streams the device path does not take (progressive, arithmetic, 12-bit, CMYK/RGB-coded, 4:4:0/4:1:1, multi-scan,
// anything malformed) are *reported*, never approximated: the caller sees FD_ERR_JPEG and hands those bytes to the
// reference's own decoder.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

namespace fd {

enum JpegStatus { JPEG_OK = 0, JPEG_NOT_JPEG = 1, JPEG_CORRUPT = 2, JPEG_UNSUPPORTED = 3 };

struct HuffTable {
    bool present;
    uint8_t bits[17];
    uint8_t vals[256];
    uint16_t lut[512];   // 9-bit look-ahead: (length << 8) | symbol, 0 = longer than 9 bits
    int16_t fast_ac[512]; // AC tables: (value << 8) | (run << 4) | (code + magnitude bits) when both fit in 9 bits, else 0
    int maxcode[18];     // largest code of each length, -1 if none
    int valoffset[17];   // vals index of the first code of each length minus that code
};

struct JpegInfo {
    int width, height, ncomp;
    int hs, vs;             // luma sampling factors (chroma is 1x1): 1x1 = 4:4:4, 2x1 = 4:2:2, 2x2 = 4:2:0
    int mcus_x, mcus_y;
    int bw[3], bh[3];       // blocks per component plane, padded to whole MCUs
    int restart_interval;
    uint16_t q[3][64];      // quantisation tables per component, natural (row-major) order
    int dc_tbl[3], ac_tbl[3];
    size_t scan_off;        // first byte of the entropy-coded segment
    HuffTable dc[4], ac[4];
};

// Parses the markers up to and including SOS.  Returns a JpegStatus; `why` gets a short reason.
int jpeg_parse(const uint8_t* d, size_t len, JpegInfo* info, char* why, size_t why_cap);
// int16 coefficients a frame needs: sum over components of bw*bh*64.
size_t jpeg_coef_count(const JpegInfo& info);
// Entropy-decodes the single interleaved scan into out[comp][block row][block col][64] (natural order,
// still quantised).  Strict: any anomaly libjpeg would only warn about is JPEG_CORRUPT here.
int jpeg_decode_coefficients(const uint8_t* d, size_t len, const JpegInfo& info, int16_t* out, char* why, size_t why_cap);

// what the kernels need to know about one frame; uploaded in front of the batch's coefficients
struct alignas(16) JpegFrameDev {
    uint16_t q[3][64];      // read 16 bytes at a time by the IDCT kernel: keep first and aligned
    uint32_t coef_off[3];   // int16 index of each component's first block within the batch coefficient buffer
    uint32_t plane_off[3];  // byte offset of each component plane within the frame's plane area
    uint16_t bw[3], bh[3];
    uint16_t hs, vs;
};

// the descriptor of a frame whose coefficients start at int16 index coef_index of the batch coefficient buffer
void jpeg_frame_desc(const JpegInfo& info, size_t coef_index, JpegFrameDev* out);
// bytes in front of a JPEG batch's coefficients: the descriptors of `frames` frames, rounded up to 256
inline size_t jpeg_head_bytes(int frames) { return (sizeof(JpegFrameDev) * size_t(frames) + 255) / 256 * 256; }
// bytes that hold the coefficients of any frame of this size the device path takes (4:4:4 / 4:2:2 / 4:2:0); a multiple of 512
size_t jpeg_frame_stride(int width, int height);

// coefficients -> u8 component planes [frame][plane_stride]
int launch_jpeg_idct(const int16_t* coefs, const JpegFrameDev* frames, uint8_t* planes, size_t plane_stride, int n,
                     int max_blocks, cudaStream_t s);
// planes -> RGB u8 [n, h, w, 3]
int launch_jpeg_rgb(const uint8_t* planes, size_t plane_stride, const JpegFrameDev* frames, uint8_t* rgb, int n, int h,
                    int w, cudaStream_t s);

// fixed pool of host threads for the entropy decode (one frame per task)
class JpegPool {
public:
    explicit JpegPool(int threads);
    ~JpegPool();
    void run(int tasks, const std::function<void(int)>& fn);  // blocks until every task has run
    int size() const { return static_cast<int>(workers_.size()) + 1; }

private:
    void worker();
    std::vector<std::thread> workers_;
    std::mutex mu_;
    std::condition_variable cv_work_, cv_done_;
    const std::function<void(int)>* fn_ = nullptr;
    int tasks_ = 0, next_ = 0, running_ = 0;
    unsigned long generation_ = 0;
    bool stop_ = false;
};

}  // namespace fd
