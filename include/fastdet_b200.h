/* fastdet_b200.h — C ABI of libfastdet_b200.so: the B200-native replacement for the work
 * `ONNXDetector` hands to ONNX Runtime plus its Python pre/post-processing.
 *
 * Reference interface each entry point replaces (paths relative to the reference repo):
 *   fd_model_create      ort.InferenceSession(path, providers)          server/detector.py:108-121
 *   fd_preprocess        PIL frame -> /255 -> f32 -> NCHW               server/detector.py:131-134
 *   fd_forward           self.model.run(None, {'input': a})             server/detector.py:135
 *   fd_postprocess       process_yolo + soft_nms + pixel scaling        server/detector.py:136-144, 45-59, 148-166
 *   fd_detect            ONNXDetector.perform after image decode        server/detector.py:126-146
 *   fd_detect_jpeg       the whole of ONNXDetector.perform, JPEG bytes in   server/detector.py:126-146 (decode :128-133)
 *   fd_pack_wire         DetectService.process_data's response packing   server/server.py:234-239
 *   fd_heads_fp32 ...    parity hooks (the raw tensors model.run returns, the f32 NCHW input tensor)
 *
 * Conventions: plain C types only; every function returns 0 on success or a negative FD_ERR_* code, with a
 * human-readable reason available from fd_last_error() (thread-local).  `stream` is a cudaStream_t passed as
 * void*; NULL selects the model's own stream.  Calls with a stream are asynchronous on it unless stated.
 * A model belongs to one CUDA device; calls on one model must not overlap in time (the reference's caller
 * is single-threaded, server/server.py:156-163).  There is no CPU fallback: without a CUDA device every
 * compute entry point fails with FD_ERR_CUDA.
 */
#ifndef FASTDET_B200_H_
#define FASTDET_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FD_OK 0
#define FD_ERR_ARG (-1)      /* bad argument */
#define FD_ERR_MODEL (-2)    /* ONNX file malformed or outside the supported operator subset */
#define FD_ERR_HEADS (-3)    /* graph has a number of outputs other than 2 or 3 (reference: KeyError at detector.py:136) */
#define FD_ERR_CUDA (-4)     /* CUDA runtime / driver failure, or no device */
#define FD_ERR_SIZE (-5)     /* frame size not accepted (reference: ValueError('invalid image size'), detector.py:132) */
#define FD_ERR_JPEG (-6)     /* a frame is not a JPEG the device decoder takes (status[] / fd_last_error say which and why);
                                nothing was launched — give those bytes to the reference's own decoder (PIL) instead */

/* per-frame status of the JPEG entry points */
#define FD_JPEG_OK 0
#define FD_JPEG_NOT_JPEG 1    /* no SOI marker: some other image format */
#define FD_JPEG_CORRUPT 2     /* malformed or truncated stream (also everything libjpeg would only warn about) */
#define FD_JPEG_UNSUPPORTED 3 /* valid JPEG outside the device path: progressive, arithmetic, 12-bit, grey/CMYK/RGB-coded,
                                 sampling other than 4:4:4 / 4:2:2 / 4:2:0, non-interleaved scans */
#define FD_JPEG_SIZE 4        /* decodable, but not the network's size (reference: ValueError('invalid image size')) */

#define FD_MAX_HEADS 4
#define FD_MAX_SLOTS 2 /* batches in flight through fd_submit / fd_collect */
#define FD_ABI_VERSION 4

typedef struct fd_model fd_model;

/* One detection, in network-input pixels, (x, y) = top-left corner: the tuple perform() returns
 * (server/detector.py:142-144).  `box` is the insertion-order index of the anchor box (head, row, column,
 * anchor) and has no counterpart in the reference; it makes results traceable to head-tensor cells. */
typedef struct fd_det {
    int32_t klass; /* 1-based class id (detector.py:165 `mi+1`) */
    int32_t box;
    double conf, x, y, w, h;
} fd_det;

typedef struct fd_info {
    int32_t abi_version;
    int32_t device;
    int32_t net_w, net_h, num_classes;
    int32_t n_heads;
    int32_t head_h[FD_MAX_HEADS], head_w[FD_MAX_HEADS], head_c[FD_MAX_HEADS];
    float anchors[FD_MAX_HEADS][3][2]; /* (w, h) in network-input pixels, chosen by n_heads as detector.py:96-106,136 */
    int32_t boxes_per_frame;
    int32_t n_layers;             /* fused layers = kernel launches per forward pass */
    int32_t n_conv;               /* convolutions among them */
    int32_t launches_per_detect;  /* n_layers + postprocess kernels */
    double conv_flops_per_frame;  /* algorithmic: sum 2*Cout*Cin*k*k*Ho*Wo */
    uint64_t num_params;
    uint64_t weight_bytes;        /* packed device weights */
} fd_info;

typedef struct fd_layer_desc {
    int32_t kind; /* 0 first conv (u8 in), 1 conv (tcgen05), 2 maxpool, 3 copy/upsample */
    int32_t c, h, w;                /* output tensor, per frame */
    int32_t cin, ksize, stride, act, has_residual, upsample2x, out_fp32, block_n;
    double flops;                   /* per frame */
    char name[96];                  /* ONNX node name */
    char out_name[96];              /* ONNX tensor name the output corresponds to */
} fd_layer_desc;

/* How one fused layer executes at a given batch size (the kernel form is chosen per batch-size bucket when the
 * execution state is built): lets tests assert that the configuration they check is the one that is timed. */
#define FD_KERNEL_CONV0 0         /* conv0_ws_kernel: normalise + first conv (pre.cu) */
#define FD_KERNEL_TC_SINGLE 1     /* conv_tc_kernel, one CTA per 128 x block_n tile */
#define FD_KERNEL_TC_PAIR 2       /* conv_tc_kernel, CTA pair (cta_group::2), 256 x 256 tiles, im2col / tiled A */
#define FD_KERNEL_TC_PAIR_STRIP 3 /* conv_tc_kernel, CTA pair, strip form (3x3 s1 p1) */
#define FD_KERNEL_TC_SWAPPED 4    /* conv_tc_kernel, channels on the MMA's M side (Cout 65..128) */
#define FD_KERNEL_HALO 5          /* conv_halo_kernel (narrow 3x3 on large maps) */
#define FD_KERNEL_MAXPOOL 6
#define FD_KERNEL_COPY 7
#define FD_KERNEL_STEM 8          /* conv_stem_kernel: normalise + first conv + second (stride-2) conv in one kernel; reported for the second */
#define FD_KERNEL_FUSED_NEXT 9    /* no launch of its own: computed inside the next layer's kernel (FD_KERNEL_STEM / FD_KERNEL_BLOCK) */
#define FD_KERNEL_BLOCK 10        /* conv_block_kernel: 1x1 + 3x3 + residual of one block in one kernel; reported for the 3x3 */
typedef struct fd_layer_exec {
    int32_t kernel;       /* FD_KERNEL_* */
    int32_t bucket;       /* batch-size bucket whose execution state answered (n rounded up) */
    int32_t block_n, split_k, grid, num_stages, kb_per_stage, b_resident;
    int32_t smem_bytes;
    int32_t chunk_frames; /* frames per launch of this layer (the bucket) */
    int32_t launches;     /* launches of this layer per forward pass (0: FD_KERNEL_FUSED_NEXT, else 1) */
    int32_t reserved[5];
} fd_layer_exec;

const char* fd_last_error(void);
int fd_abi_version(void);
/* Plan-time options (process-wide; read when a model's execution state for a batch size is first built, so set them
 * before the first call at that size).  Names and defaults: csrc/options.h.  Unknown names return FD_ERR_ARG. */
int fd_set_option(const char* name, int value);
int fd_get_option(const char* name, int* value);
/* Number of CUDA devices visible; 0 when there is no driver/GPU (never fails). */
int fd_device_count(void);

/* Parse + plan + upload.  net_w/net_h: network input size (the reference hard-wires 416x416, detector.py:66). */
int fd_model_create(const void* onnx_bytes, size_t len, int num_classes, int net_w, int net_h, int device,
                    fd_model** out);
void fd_model_destroy(fd_model* m);
int fd_model_info(const fd_model* m, fd_info* out);
int fd_layer_info(const fd_model* m, int layer, fd_layer_desc* out);
/* Host logic only (also on a plan-only model, device -1): the layer pairs the planner hands to the fused kernels at batch n under
 * the current options.  *stem: 1 when layers 0 + 1 run as one kernel (FD_KERNEL_STEM); *block_layer: the first layer of the pair
 * that runs as FD_KERNEL_BLOCK, or -1. */
int fd_planned_fusions(const fd_model* m, int n, int32_t* stem, int32_t* block_layer);
/* Builds (if needed) the execution state for batch size n and reports the kernel form of `layer` in it. */
int fd_layer_exec_info(fd_model* m, int layer, int n, fd_layer_exec* out);

/* Stage `n` RGB u8 HWC frames for the next fd_forward.  src_w x src_h must equal the network size unless
 * allow_resize != 0, in which case the frames are letterboxed on the device (extension).  on_device: frames
 * is a device pointer on the model's device; otherwise host memory (pinned memory makes the copy async). */
int fd_preprocess(fd_model* m, const uint8_t* frames, int n, int src_w, int src_h, int on_device, int allow_resize,
                  void* stream);
/* Run the conv stack on the staged frames (captured CUDA graph per batch size). */
int fd_forward(fd_model* m, int n, void* stream);
/* Decode + Soft-NMS on the head tensors of the last fd_forward.  Results land in device/pinned buffers owned by
 * the model; fd_fetch copies them out.  threshold is the reference's `threshold` (a Python float). */
int fd_postprocess(fd_model* m, int n, double threshold, int max_det, void* stream);
/* fd_postprocess with one threshold per frame (thresholds[n], host memory; read before the call returns).  Frame f's
 * records are bit for bit those of fd_postprocess at thresholds[f]. */
int fd_postprocess_thresholds(fd_model* m, int n, const double* thresholds, int max_det, void* stream);
/* Synchronise `stream` and copy the results of the last fd_postprocess: counts[n] and out[n][max_det]
 * (max_det as given to fd_postprocess).  total[n] (optional) receives the untruncated kept count. */
int fd_fetch(fd_model* m, int n, fd_det* out, int32_t* counts, int32_t* total, void* stream);
/* preprocess -> forward -> postprocess -> fetch; synchronous; frames in host (or device) memory. */
int fd_detect(fd_model* m, const uint8_t* frames, int n, int src_w, int src_h, int on_device, int allow_resize,
              double threshold, int max_det, fd_det* out, int32_t* counts);

/* Pipelined form of fd_detect for callers that serve a stream of batches (the reference's server loop calls
 * perform() once per UDP payload, server/server.py:225-241; a batching front end calls these instead).
 * fd_submit enqueues copy -> forward -> postprocess -> result copy for ring slot `slot` (0 .. FD_MAX_SLOTS-1) and
 * returns without waiting; the host->device copy runs on its own stream, so it overlaps the previous slot's
 * compute.  `frames` must stay valid (and should be pinned) until fd_collect(slot) returns.  fd_collect blocks
 * until the slot's results are on the host and copies out counts[n] and out[n][max_det]; total may be NULL.
 * Results are identical to fd_detect on the same frames. */
int fd_submit(fd_model* m, int slot, const uint8_t* frames, int n, int src_w, int src_h, int on_device,
              int allow_resize, double threshold, int max_det);
int fd_collect(fd_model* m, int slot, fd_det* out, int32_t* counts, int32_t* total);

/* ---- JPEG in: the first lines of the reference's perform() (server/detector.py:128-133) are
 * `img = Image.open(io.BytesIO(data))`, the size check and `np.array(img)`, i.e. a libjpeg decode on one host core per
 * frame.  These entry points take the JPEG bytes themselves: Huffman decode on a pool of host threads, then
 * de-quantisation, IDCT (libjpeg's ISLOW), fancy chroma upsampling and YCbCr->RGB on the device, bit-identical to
 * libjpeg(-turbo)'s default output, written straight into the batch's input tensor.  Baseline / extended-sequential
 * Huffman, 8-bit, 3-component YCbCr, 4:4:4 / 4:2:2 / 4:2:0, restart intervals.  Anything else is refused with
 * FD_ERR_JPEG before any device work (no approximation, no silent host decode): status[n] (may be NULL) receives one
 * FD_JPEG_* per frame.  A batch whose only problem is the frame size returns FD_ERR_SIZE like fd_detect.
 * allow_resize != 0 (extension, as in fd_preprocess): the frames may have any ONE size (that of the first decodable
 * frame, at most 8192 x 8192); they are decoded at that size and letterboxed to the network's on the device. */
typedef struct fd_jpeg_info {
    int32_t status; /* FD_JPEG_* (size is not checked here) */
    int32_t width, height, components;
    int32_t h_samp, v_samp; /* luma sampling factors */
    int32_t restart_interval;
    int32_t blocks_w[3], blocks_h[3]; /* 8x8 blocks per component plane, padded to whole MCUs */
    int64_t coef_count;               /* int16 coefficients fd_jpeg_coefficients writes */
    uint16_t quant[3][64];            /* per component, row-major (de-zigzagged) */
    char reason[160];
} fd_jpeg_info;
/* Host only (no device needed): parse the headers / entropy-decode one frame into quantised coefficients
 * coefs[component][block row][block col][64], row-major inside a block.  Test and tooling hooks. */
int fd_jpeg_probe(const uint8_t* data, size_t len, fd_jpeg_info* out);
int fd_jpeg_coefficients(const uint8_t* data, size_t len, int16_t* coefs, size_t cap, fd_jpeg_info* out);
/* Decode n JPEGs into the model's input tensor for batch size n (where fd_preprocess puts frames), synchronous; follow
 * with fd_forward(m, n, NULL).  rgb_out (host, may be NULL) receives the decoded frames [n, net_h, net_w, 3]. */
int fd_decode_jpeg(fd_model* m, const uint8_t* const* data, const size_t* lens, int n, int allow_resize, int32_t* status,
                   uint8_t* rgb_out);
/* fd_detect / fd_submit taking JPEG bytes.  The entropy decode runs inside the call on the host pool (while the device
 * works on the other slot); collect with fd_collect. */
int fd_detect_jpeg(fd_model* m, const uint8_t* const* data, const size_t* lens, int n, int allow_resize, double threshold,
                   int max_det, fd_det* out, int32_t* counts, int32_t* status);
int fd_submit_jpeg(fd_model* m, int slot, const uint8_t* const* data, const size_t* lens, int n, int allow_resize,
                   double threshold, int max_det, int32_t* status);

/* Letterbox bookkeeping (host only; extension — the reference rejects frames that are not network-sized).  With
 * allow_resize the frame is scaled to new_w x new_h (aspect kept, the long side filling the network) and centred at
 * (off_x, off_y) on a grey canvas; detections come back in network pixels.  fd_unmap_letterbox rewrites `count` records
 * in place to pixels of the src_w x src_h frame the caller sent: x = (x - off_x) * src_w / new_w, w = w * src_w / new_w,
 * same for y / h (float64). */
int fd_letterbox_geometry(int src_w, int src_h, int net_w, int net_h, int32_t* new_w, int32_t* new_h, int32_t* off_x,
                          int32_t* off_y);
int fd_unmap_letterbox(fd_det* dets, int count, int src_w, int src_h, int net_w, int net_h);

/* Wire-format packer (host only, no device needed): the response payload the reference builds per request in
 * DetectService.process_data (server/server.py:234-239): a 16-byte big-endian header '>4sLLL' = (b"YOLO", reqid, msec,
 * payload length) followed by one 10-byte record '>BBhhhh' = (klass, int(conf*255), int(x), int(y), int(w), int(h)) per
 * detection, int() truncating toward zero.  saturate = 0 mirrors struct.pack: a klass outside 0..255 or a coordinate
 * outside int16 returns FD_ERR_ARG (the reference raises struct.error and its server loop dies); saturate != 0 clamps
 * instead.  *len receives the bytes written; cap must be >= 16 + 10 * count. */
int fd_pack_wire(const fd_det* dets, int count, uint32_t reqid, uint32_t msec, int saturate, uint8_t* out, size_t cap,
                 size_t* len);

/* ---- multi-model, multi-GPU serving (BASELINE config 5) ----------------------------------------------------------
 * The reference keeps one detector object per model spec and shares it between all sessions (server/server.py:295,
 * 311-312), each payload served by one blocking detector.perform() on a single select loop (:156-163, :232).  fd_server
 * is that dict of detectors replicated on every device: one LANE per (device, model) = a model replica with its own
 * streams + a worker thread + a queue of micro-batches (two in flight through fd_submit / fd_collect).  A stream is
 * pinned to device slot (stream_id mod n_devices).  fd_server_perform has the call shape of perform() — one decoded RGB
 * frame in, that frame's records out, blocking — and may be called from any number of threads at once; concurrent calls
 * for the same (device, model) ride in one batch.  fd_server_perform_jpeg takes the payload perform() gets, JPEG bytes with
 * the request's own threshold, and decodes it on the device path of fd_detect_jpeg.  Results are those of fd_detect on the same frame (to the batch-size
 * dependence documented for split-K).  No collective, no cross-device traffic: frames are independent. */
#define FD_SERVER_MAX_MODELS 8
#define FD_SERVER_MAX_DEVICES 16
typedef struct fd_server fd_server;
typedef struct fd_server_model {
    const void* onnx_bytes;
    size_t len;
    int32_t num_classes, net_w, net_h;
} fd_server_model;
typedef struct fd_serve_stats {
    double seconds;
    int64_t frames;
    double frames_per_second;
    double latency_ms_p50, latency_ms_p90, latency_ms_p99, latency_ms_mean, latency_ms_max;
    int64_t batches;    /* batches the lanes ran inside the measured window */
    double mean_batch;  /* frames per batch */
    int64_t detections;
    int32_t streams;
    int32_t reserved;
    int64_t frames_per_device[FD_SERVER_MAX_DEVICES];
    int64_t frames_per_model[FD_SERVER_MAX_MODELS];
} fd_serve_stats;
/* devices[n_devices]: CUDA device ordinals (device slot d serves the streams with stream_id % n_devices == d).
 * max_batch: frames per micro-batch at most; max_det: records kept per frame; max_delay_ms: how long a lane with NOTHING
 * in flight waits for more callers before it runs a partial batch (0: not at all). */
int fd_server_create(const fd_server_model* models, int n_models, const int32_t* devices, int n_devices, int max_batch,
                     int max_det, double max_delay_ms, fd_server** out);
void fd_server_destroy(fd_server* s);
/* Blocking, thread-safe.  frame: host RGB u8 [src_h, src_w, 3] (copied before the call sleeps); src size must be the
 * model's (FD_ERR_SIZE otherwise, reference detector.py:132).  out[max_det], *count: the frame's records.  A micro-batch
 * of RGB frames holds one threshold: a caller with another threshold starts a new batch. */
int fd_server_perform(fd_server* s, int stream_id, int model, const uint8_t* frame, int src_w, int src_h, double threshold,
                      fd_det* out, int max_det, int32_t* count);
/* fd_server_perform for one encoded payload: blocking, thread-safe.  A payload the device decoder does not take returns
 * FD_ERR_JPEG with *status (FD_JPEG_*) and never enters a batch; a decodable frame of another size returns FD_ERR_SIZE.
 * The caller's thread parses the payload and entropy-decodes it straight into the open JPEG micro-batch of its lane; the
 * IDCT, colour conversion, forward pass and post-processing of the batch run on the device.  Callers with different
 * thresholds share a JPEG batch (the thresholds are per frame).  A payload whose entropy data turns out damaged behind a
 * valid header still rides its batch, but its caller gets FD_ERR_JPEG / FD_JPEG_CORRUPT and no records; the other
 * frames of the batch are not affected.  status may be NULL. */
int fd_server_perform_jpeg(fd_server* s, int stream_id, int model, const uint8_t* data, size_t len, double threshold,
                           fd_det* out, int max_det, int32_t* count, int32_t* status);
/* Build every lane's execution state for the batch-size buckets up to `up_to` frames now (in parallel over the lanes), so
 * that no request pays for buffer allocation and graph capture later.  Call before serving. */
int fd_server_warm(fd_server* s, int up_to);
int fd_server_lane_stats(fd_server* s, int device_slot, int model, int64_t* batches, int64_t* frames);
/* Load generator (measurement tool): n_streams caller threads, stream i -> model stream_model[i] and device slot
 * i % n_devices, each sending its next frame (from frames[n_frames][src_h][src_w][3], host) as soon as the previous result
 * is back; statistics over `seconds` after `warmup_seconds`.  Latency = wall time of one fd_server_perform call. */
int fd_server_closed_loop(fd_server* s, int n_streams, const int32_t* stream_model, const uint8_t* frames, int n_frames,
                          int src_w, int src_h, double threshold, double warmup_seconds, double seconds, fd_serve_stats* out);
/* Host-only stand-in backend (tests of routing / batching without a GPU): every frame "detects" one record that says where
 * it was served: klass = the frame's first byte, box = size of the batch it rode in, conf = device slot, x = model, y = ring
 * slot; collect sleeps latency_us.  JPEG payloads go through the real host half (parse, entropy decode into the batch);
 * their record has klass = the frame's first quantised luma DC coefficient and w = the frame's threshold. */
int fd_server_create_fake(int n_models, int n_devices, int net_w, int net_h, int max_batch, double max_delay_ms, int latency_us,
                          fd_server** out);
const char* fd_server_last_error(void);

/* ---- parity / profiling hooks (synchronous; host pointers) ---- */
/* Raw head tensor `head` of the last forward as f32 NCHW [n, C, H, W] — what model.run returns. */
int fd_heads_fp32(fd_model* m, int head, float* dst_nchw, int n);
/* Overwrite head tensor `head` with f32 NCHW data (to test postprocess on exact inputs). */
int fd_set_heads_fp32(fd_model* m, int head, const float* src_nchw, int n);
/* Output of fused layer `layer` of the last forward as f32 NCHW. */
int fd_layer_output_fp32(fd_model* m, int layer, float* dst_nchw, int n);
/* The f32 NCHW tensor the reference feeds to model.run, computed on the device from net-sized u8 frames. */
int fd_normalise_f32(fd_model* m, const uint8_t* frames, int n, float* dst_nchw);
/* Device letterbox of host frames [n, src_h, src_w, 3] to [n, net_h, net_w, 3]. */
int fd_letterbox_u8(fd_model* m, const uint8_t* frames, int n, int src_w, int src_h, uint8_t* dst);
/* Per-layer device time (ms, mean over reps) of the forward pass at batch n: every layer timed alone (reps back-to-back
 * launches; 0 for a layer computed inside the next layer's kernel). */
int fd_time_layers(fd_model* m, int n, int reps, float* ms_per_layer);
/* Device time (ms, mean over reps back-to-back runs) of fd_forward at batch n: the captured graph as serving runs it. */
int fd_time_forward(fd_model* m, int n, int reps, float* ms);

#ifdef __cplusplus
}
#endif
#endif /* FASTDET_B200_H_ */
