/*
 * tic.h — C ABI of the B200-native hot path of the learned patch codec
 * (tf_image_compression): conv analysis transform -> quantise (+histogram) ->
 * deconv synthesis transform -> rm_block_effect post-filter.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types,
 * no exceptions.  Every entry point names the reference interface it replaces
 * (paths relative to the reference repo).  Host-side mirror of the reference's
 * Python API: tf_image_compression_b200/ (see INTEGRATION.md for the binding a
 * reference maintainer would add).
 *
 * Conventions
 *   - all activations / images are NHWC, channel-contiguous (the reference's TF layout);
 *   - `mem` says where the caller's I/O buffers live (TIC_MEM_HOST / TIC_MEM_DEVICE);
 *     device pointers are used in place on the handle's stream, host pointers are
 *     copied through a double-buffered H2D -> compute -> D2H pipeline (pinned host
 *     memory overlaps, pageable memory works but serialises);
 *   - the caller owns every buffer passed in; the handle owns weights, workspaces,
 *     look-up tables and the symbol histogram;
 *   - every function returns TIC_OK (0) or a negative tic_status; the message is
 *     available from tic_last_error().  One handle per device, not thread-safe.
 *   - there is NO CPU fallback: without a CUDA device tic_create fails.
 */
#ifndef TIC_H_
#define TIC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tic_codec tic_codec;

typedef enum tic_status {
  TIC_OK = 0,
  TIC_ERR_INVALID = -1,     /* bad argument / shape (Python shim raises ValueError) */
  TIC_ERR_CUDA = -2,        /* CUDA runtime error (RuntimeError) */
  TIC_ERR_STATE = -3,       /* graph / weights / tables not configured (RuntimeError) */
  TIC_ERR_NOMEM = -4,
  TIC_ERR_UNSUPPORTED = -5
} tic_status;

typedef enum tic_graph_id {
  TIC_GRAPH_ENCODER = 0,    /* model.encoder   (model_0/model.py:34-144) */
  TIC_GRAPH_DECODER = 1,    /* model.decoder   (model_0/model.py:147-263) */
  TIC_GRAPH_POSTFILTER = 2  /* rmbe_model.model (submit/2/rmbe/model.py:113-197) */
} tic_graph_id;

typedef enum tic_layer_kind {
  TIC_CONV = 0,   /* basic_block.my_conv2d           (basic_block/basic_block.py:27-47) */
  TIC_DECONV = 1  /* basic_block.my_conv2d_transpose (basic_block/basic_block.py:50-71) */
} tic_layer_kind;

typedef enum tic_act { TIC_ACT_IDENTITY = 0, TIC_ACT_RELU = 1 } tic_act;
typedef enum tic_mem { TIC_MEM_HOST = 0, TIC_MEM_DEVICE = 1 } tic_mem;
typedef enum tic_dtype { TIC_U8 = 0, TIC_F32 = 1 } tic_dtype;

typedef enum tic_compute_mode {
  TIC_COMPUTE_FP32 = 0,       /* fp32 FMA on CUDA cores: the exact path */
  TIC_COMPUTE_TENSOR_3XTF32 = 1, /* tcgen05 implicit GEMM, error-compensated 3xTF32 split, fp32 accumulate in TMEM */
  TIC_COMPUTE_TENSOR_TF32 = 2,   /* tcgen05 implicit GEMM, single-pass TF32 (fast; symbol mismatch ~1e-4, documented) */
  TIC_COMPUTE_TENSOR_F16X3 = 3   /* tcgen05 implicit GEMM on fp16 (hi, lo) pairs, three products, activations kept as two fp16
                                    planes; fp32-class accuracy, |activation| must stay below 65504 */
} tic_compute_mode;

/* One 3x3 layer.  A res_block (basic_block/basic_block.py:74-93) is two conv layers:
 * the first has res_begin = 1 (its INPUT is remembered), the second has res_end = 1
 * (remembered tensor is added AFTER its activation: x + relu(conv1(relu(conv0(x))))). */
typedef struct tic_layer_desc {
  int32_t kind;      /* tic_layer_kind */
  int32_t cin;
  int32_t cout;
  int32_t stride;    /* conv: 1 or 2 (TF SAME padding); deconv: 2 (output = 2x input) */
  int32_t act;       /* tic_act */
  int32_t res_begin;
  int32_t res_end;
} tic_layer_desc;

/* ---- lifetime ------------------------------------------------------------ */
/* Replaces tf.Session() creation in encode.py:215-234 / decode.py:269-289. */
int tic_create(tic_codec** out, int device);
void tic_destroy(tic_codec* h);
const char* tic_last_error(const tic_codec* h);
/* Message of the last failed tic_create (no handle exists yet). */
const char* tic_create_error(void);
/* Run on the caller's CUDA stream (cudaStream_t as void*); default: a private stream. */
int tic_set_stream(tic_codec* h, void* cuda_stream);
int tic_set_compute_mode(tic_codec* h, int mode);
/* Synchronises the handle's stream and returns its sticky status: TIC_OK, or TIC_ERR_UNSUPPORTED once a
 * TIC_COMPUTE_TENSOR_F16X3 run produced an activation outside the fp16 range (|x| >= 65504: every kernel that writes
 * fp16 pair planes checks).  Host-buffer calls return the status themselves; device-buffer calls are asynchronous, so
 * the status shows at the next hot-path call or here.  tic_set_compute_mode clears it. */
int tic_check_status(tic_codec* h);
/* Patches pushed through the layer stack per launch sequence (workspace size).
 * Given in units of 128x128 patches; scaled by (128/P)^2 for other patch sizes. */
int tic_set_chunk_patches(tic_codec* h, int chunk);

/* ---- graph + parameters -------------------------------------------------- */
/* Replaces the graph build model.encoder(...) / model.decoder(...) / rmbe_model.model(...)
 * at encode.py:147, decode.py:167, submit/2/rmbe/rmbe.py:40. */
int tic_set_graph(tic_codec* h, int graph, const tic_layer_desc* layers, int n_layers);
/* Replaces utils.restore_params (utils/utils.py:84-93) for one layer scope.
 * kernel: host fp32 in the TF variable layout — conv [3,3,cin,cout] (HWIO),
 * deconv [3,3,cout,cin] (basic_block.py:53); bias: host fp32 [cout]. */
int tic_load_weights(tic_codec* h, int graph, int layer, const float* kernel, const float* bias);
/* channel_normalization_params.npz 'mean'/'std' (model_0/model.py:26-28,44,251), fp32 [3]. */
int tic_set_norm(tic_codec* h, int graph, const float* mean3, const float* std3);
/* quan_scale from config.json and the q-entry inverse-sigmoid table
 * lut[s] = log(p/(1-p)), p = (s+1e-6)/(q-1+1e-5)  (model_0/model.py:153, basic_block.py:152-155). */
int tic_set_quantizer(tic_codec* h, int quan_scale, const float* inv_sigmoid_lut);
/* Bottleneck shape (h_b, w_b, c_b) the encoder graph produces for patch size P. */
int tic_bottleneck_shape(tic_codec* h, int P, int* hb, int* wb, int* cb);

/* ---- hot path ------------------------------------------------------------ */
/* model.encoder on a batch of patches (encode.py:157-165): patches [n,P,P,3] (u8 or f32,
 * 0..255) -> symbols [n,h_b,w_b,c_b] (u8, or integer-valued f32 as the reference returns).
 * Also accumulates the symbol histogram (get_encoded_distribution.py:113-126). */
int tic_encode_patches(tic_codec* h, const void* patches, int in_dtype, int64_t n, int P,
                       void* symbols, int out_dtype, int mem);
/* crop_image_input_patches (utils/utils.py:96-133) + encoder, fused: n_images u8 images
 * [n_images,H,W,3] are reflect-padded to a multiple of P by index arithmetic inside the
 * first layer's loads; symbols come back patch-major per image (encode.py:171-182):
 * [n_images, gh*gw, h_b, w_b, c_b] u8. */
int tic_encode_images(tic_codec* h, const uint8_t* images, int64_t n_images, int H, int W, int P,
                      uint8_t* symbols, int mem);
/* model.decoder on a batch of symbol patches (decode.py:204-220): symbols [n,h_b,w_b,c_b] u8
 * -> recon [n,P,P,3] f32 in [0,255]. */
int tic_decode_patches(tic_codec* h, const uint8_t* symbols, int64_t n, int hb, int wb,
                       float* recon, int mem);
/* decoder + concat_patches (utils/utils.py:136-167) (+ np.around -> uint8, decode.py:249), fused:
 * the last layer scatters straight into [n_images,H,W,3]; out_dtype TIC_U8 rounds half-to-even,
 * TIC_F32 keeps the float image (input of rmbe, submit/2/decoder.py:183-184). */
int tic_decode_images(tic_codec* h, const uint8_t* symbols, int64_t n_images, int H, int W, int P,
                      void* images, int out_dtype, int mem);
/* test.py:95-146 (compress_and_uncompress): encoder and decoder built in ONE graph, image in ->
 * reconstruction out, no bitstream in between.  images [n_images,H,W,3] u8 -> symbols
 * [n_images, gh*gw, h_b, w_b, c_b] u8 (may be NULL with host buffers: not copied back) and recon
 * [n_images,H,W,3] (TIC_U8 rounded half-to-even | TIC_F32).  Results are identical to
 * tic_encode_images followed by tic_decode_images; with host buffers the H2D of chunk i+1, the
 * kernels of chunk i and the D2H of chunk i-1 overlap, so both PCIe directions are busy at once. */
int tic_roundtrip_images(tic_codec* h, const uint8_t* images, int64_t n_images, int H, int W, int P,
                         uint8_t* symbols, void* recon, int out_dtype, int mem);
/* rmbe_model.model on [n,128,128,3] f32 tiles (submit/2/rmbe/model.py:113-197). */
int tic_postfilter_patches(tic_codec* h, const float* tiles, int64_t n, int P, float* out, int mem);
/* rmbe.rmbe(image) (submit/2/rmbe/rmbe.py:15-111): two in-place passes of 128x128 tiles offset
 * by 64 (vertical seams, then horizontal seams) over f32 images [n_images,H,W,3]. */
int tic_postfilter_images(tic_codec* h, float* images, int64_t n_images, int H, int W, int mem);
/* Layers [0, n_layers) of a graph on plain f32 NHWC activations, without the fused prologue /
 * epilogue: in [n,h0,w0,cin of layer 0] -> out [n,h,w,cout of layer n_layers-1].  What a
 * sess.run on an intermediate tensor of the reference graph returns (e.g. the commented-out
 * tf.Print probes, model_0/model.py:157,222,248); used by the layer-by-layer parity tests. */
int tic_run_layers(tic_codec* h, int graph, const float* in, int64_t n, int h0, int w0, int n_layers,
                   float* out, int mem);
/* np.around -> uint8 of a float image (decode.py:249), device or host buffers. */
int tic_round_u8(tic_codec* h, const float* src, uint8_t* dst, int64_t count, int mem);

/* ---- symbol statistics --------------------------------------------------- */
/* freq[q] accumulated by every tic_encode_* since the last reset
 * (get_encoded_distribution.py:113-126).  counts: host uint64[q]. */
int tic_hist_reset(tic_codec* h);
int tic_hist_read(tic_codec* h, uint64_t* counts, int q);
/* Device address of the uint64[256] histogram (for an in-place NCCL all-reduce of the
 * dataset-wide table across ranks; the only collective on the path). */
int tic_hist_device_ptr(tic_codec* h, void** dev_ptr);
/* Per-position symbol sums over patches (cal_encoded_distribution.py:111-128):
 * sums[h_b*w_b*c_b] (uint64) += sum_n symbols[n, pos].  symbols u8 [n, npos]. */
int tic_position_sums(tic_codec* h, const uint8_t* symbols, int64_t n, int64_t npos,
                      uint64_t* sums, int mem);
/* The same per sess.run batch: sums[b][pos] = sum over patches [b*batch, (b+1)*batch) (overwritten, not accumulated),
 * b < ceil(n / batch).  The reference folds one batch of 64 at a time into a float64 running mean
 * (cal_encoded_distribution.py:111-128); exact integer batch sums let the host repeat that arithmetic bit for bit. */
int tic_position_sums_batched(tic_codec* h, const uint8_t* symbols, int64_t n, int64_t npos, int64_t batch,
                              uint64_t* sums, int mem);

/* ---- GPU entropy stage (SURVEY.md §8f rank 4) ----------------------------- */
/* The per-image static-model range coder of encode.py:171-202 (RangeEncoder(path).encode(seq, cum_freq); close()) on
 * the device: n_streams streams of stream_len uint8 symbols each (one image's patch-major symbol sequence,
 * encode.py:171-182, exactly what tic_encode_images leaves in HBM), one table for all (encode.py:76-91).  Stream i is
 * written to out + i * out_stride (tic_entropy_bound(stream_len) bytes always suffice), out_bytes[i] = its stored
 * length.  The bytes are IDENTICAL to what the host coder (include/tic_rangecoder.h) writes to its file for the same
 * symbols and table: both compile include/tic_rc_core.h.  Tables: 1..256 symbols, total <= 65536.
 * mem = TIC_MEM_DEVICE: symbols / out / out_bytes are device buffers, asynchronous on the handle's stream (errors —
 * a symbol outside the table or of zero probability — surface through tic_check_status); cum_freq is always a host
 * array.  mem = TIC_MEM_HOST: staged, synchronous, only the stored bytes are copied back. */
int64_t tic_entropy_bound(int64_t stream_len);
int tic_entropy_encode(tic_codec* h, const uint8_t* symbols, int64_t n_streams, int64_t stream_len, const uint32_t* cum_freq,
                       int n_cum, uint8_t* out, int64_t out_stride, int64_t* out_bytes, int mem);
/* RangeDecoder(path).decode(n, cum_freq) (decode.py:79-101, 182) for n_streams files at once: stream i = in_bytes[i]
 * stored bytes at in + i * in_stride (in_stride a multiple of 16, device buffers 16-byte aligned; bytes past the stored
 * length read as zero, like the host decoder past EOF) -> symbols[i * stream_len ...]. */
int tic_entropy_decode(tic_codec* h, const uint8_t* in, int64_t n_streams, int64_t in_stride, const int64_t* in_bytes,
                       const uint32_t* cum_freq, int n_cum, uint8_t* symbols, int64_t stream_len, int mem);

/* ---- rate-distortion evaluation ------------------------------------------ */
/* encode.py -> decode.py -> processing_utils/evaluate.py (scipt_bash/encode_decode_evaluate.sh) without files:
 * images [n_images,H,W,3] u8 -> code_bytes[i] = stored length of image i's range-coded stream (== tic_entropy_encode's
 * out_bytes == the size of the file entry.compress writes), sq_err[i] = sum over H*W*3 of (recon - image)^2 with recon
 * the u8 reconstruction tic_decode_images(TIC_U8) returns; recon may be NULL (not written).  cum_freq: host array, as in
 * tic_entropy_encode.  mem applies to images, code_bytes, sq_err and recon.
 * Chunks of whole images run encoder -> range coder (lengths only) -> decoder -> squared error on the device; symbols,
 * reconstructions and squared errors stay in HBM.  Host buffers: the H2D of chunk i+1 overlaps the kernels of chunk i
 * (as in tic_roundtrip_images), the per-image results come back once at the end, errors are returned.  Device buffers:
 * asynchronous on the handle's stream; a symbol outside the table or of zero probability surfaces at tic_check_status.
 * The symbol histogram accumulates as on every encoder call.  n_images == 0 writes nothing. */
int tic_evaluate_images(tic_codec* h, const uint8_t* images, int64_t n_images, int H, int W, int P,
                        const uint32_t* cum_freq, int n_cum, int64_t* code_bytes, uint64_t* sq_err,
                        uint8_t* recon, int mem);

/* ---- introspection (measurement) ----------------------------------------- */
/* Kernels launched by this handle since creation (bench.py's gpu_launches). */
int64_t tic_launch_count(const tic_codec* h);
/* Device time (ms) of the last tic_* hot-path call, measured with CUDA events on the
 * handle's stream around the kernel sequence (excludes H2D/D2H of host-mode calls). */
float tic_last_kernel_ms(const tic_codec* h);
/* Per-layer device timing: when enabled, every layer launch is bracketed by CUDA events on the
 * handle's stream.  tic_profile_read returns, for `graph`, the accumulated milliseconds and launch
 * counts per layer since the last tic_profile_reset (arrays of n_layers entries). */
int tic_profile_enable(tic_codec* h, int on);
int tic_profile_reset(tic_codec* h);
int tic_profile_read(tic_codec* h, int graph, float* ms, int64_t* launches, int n_layers);
/* CRC-32C (Castagnoli, reflected, init/xorout 0xffffffff) of a host buffer: the checksum of the TF-V2 checkpoint
 * bundle that utils.restore_params reads (utils/utils.py:84-93; tf_image_compression_b200/checkpoint.py). */
uint32_t tic_crc32c(const void* data, uint64_t n);
const char* tic_version(void);

#ifdef __cplusplus
}
#endif
#endif /* TIC_H_ */
