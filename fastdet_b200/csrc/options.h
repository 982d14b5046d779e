// options.h — plan-time options of the library (process-wide, read when execution state for a batch size is built).
//
// A test or tool sets one through the C ABI (fd_set_option / fd_get_option, include/fastdet_b200.h), builds a model, and
// asserts the kernel form each layer took through fd_layer_exec_info.  The defaults are the production configuration;
// nothing reads the environment.  Each option selects a kernel form that tests compare with another one (strip, stem,
// block, fuse_pool, nms_general) or sizes a host-side resource (jpeg_threads, server_inflight).  fd_set_option also takes
// "segv_backtrace" (capi.cu), which installs a crash handler and is not stored here.
#pragma once

namespace fd {

struct Options {
    int strip = 1;            // 3x3 s1 p1 layers of the CTA-pair kernel: 0 im2col form only, 1 strips where they pay and fill the GPU, 2 wherever legal
    int stem = 1;             // first two convolutions (3 -> 32 s1, 32 -> 64 s2) of a YOLOv3-shaped graph in one kernel (conv_stem.cu)
    int block = 1;            // a 1x1 (64 -> 32) + 3x3 (32 -> 64) + residual block on a large map in one kernel (conv_block.cu)
    int fuse_pool = 1;        // MaxPool(2, 2) after the first convolution / a halo-patch layer runs in that kernel's epilogue
    int nms_general = 0;      // force the general (global-memory) Soft-NMS loop
    int jpeg_threads = 0;     // host threads of the JPEG entropy decoder; 0 = all hardware threads (max 64)
    int server_inflight = 2;  // fd_server: micro-batches in flight per lane (2: copy / compute overlap at saturation; 1: a closed loop
                              // of few streams per lane gathers larger batches, see DESIGN.md section 6)
};

Options& options();
// name -> field; returns nullptr for unknown names
int* option_slot(const char* name);

}  // namespace fd
