// options.h — plan-time options of the library (process-wide, read when execution state for a batch size is built).
//
// They replace the getenv() switches of the first round: a test or tool sets one through the C ABI
// (fd_set_option / fd_get_option, include/fastdet_b200.h), builds a model, and asserts the kernel form each layer took
// through fd_layer_exec_info.  The defaults are the production configuration; nothing reads the environment.
#pragma once

namespace fd {

struct Options {
    int strip = 1;            // 3x3 s1 p1 layers of the CTA-pair kernel: 0 im2col form only, 1 strips where they pay and fill the GPU, 2 wherever legal
    int strip_min_w = 12;     // strips only on maps at least this wide (pad positions cost (W+1)(H+1)/(WH))
    int swap = 1;             // swapped (channels on the MMA's M side) form for 65..128 output channels
    int two_cta = 1;          // CTA-pair (cta_group::2) kernel for Cout > 128, Cin % 64 == 0
    int split_k = 1;          // split long K loops when a launch cannot fill the GPU (small batches)
    int split_k_min_kb = 32;  // ... only with at least this many K blocks
    int split_k_max = 4;      // ... into at most this many parts
    int latency_bn = 1;       // small batches: layers that would fill < 1/4 of the SMs use 128 x 64 / 128 x 128 single-CTA tiles
                              // (1: chosen per layer, 64 / 128: forced, 0: off)
    int b_resident = 1;       // keep a narrow layer's whole filter bank in shared memory
    int stem = 1;             // first two convolutions (3 -> 32 s1, 32 -> 64 s2) of a YOLOv3-shaped graph in one kernel (conv_stem.cu)
    int block = 1;            // a 1x1 (64 -> 32) + 3x3 (32 -> 64) + residual block on a large map in one kernel (conv_block.cu)
    int halo = 1;             // halo-patch kernel for 16/32/64-channel 3x3 layers on large maps
    int halo_skew = 1;        // ... with chunk planes skewed against shared-memory bank conflicts
    int halo_slots = 0;       // ... patch ring depth cap (0: the kernel's maximum)
    int fuse_pool = 1;        // MaxPool(2, 2) after the first convolution / a halo-patch layer runs in that kernel's epilogue
    int pdl = 1;              // programmatic dependent launch between layers
    int graph = 1;            // replay the forward pass as a captured CUDA graph
    int exact_batch = 0;      // one execution state per exact batch size instead of per bucket
    int nms_general = 0;      // force the general (global-memory) Soft-NMS loop
    int jpeg_threads = 0;     // host threads of the JPEG entropy decoder; 0 = all hardware threads (max 64)
    int server_inflight = 2;  // fd_server: micro-batches in flight per lane (2: copy / compute overlap at saturation; 1: a closed loop
                              // of few streams per lane gathers larger batches, see DESIGN.md section 6)
    int detect_overlap = 1;   // synchronous fd_detect: the frame copy in four pieces, overlapped with the first layers
};

Options& options();
// name -> field; returns nullptr for unknown names
int* option_slot(const char* name);

}  // namespace fd
