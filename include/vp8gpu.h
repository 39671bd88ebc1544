/* vp8gpu.h -- C ABI of the B200-native VP8 pixel pipeline.
 *
 * This is the drop-in boundary for the hot path of excamera/alfalfa's src/decoder
 * (SURVEY.md section 8b).  Alfalfa has no FFI of its own: its boundary is the C++
 * class API, so every entry point below names the reference interface it stands in for
 * (paths relative to /root/reference/src).  Plain pointers and sizes only; no C++ or
 * torch types cross this line.  The C++ mirror of the reference classes that sits on
 * top of this ABI is alfalfa_b200/host/alfalfa_gpu.hh; INTEGRATION.md shows the
 * reference-side binding.
 *
 * Layering (top to bottom):
 *   vp8gpu_decoder_*   = Decoder           (decoder/decoder.hh:244-300)
 *   vp8gpu_parse_*     = DecoderState::parse_and_apply (decoder/decoder_state.hh:73-167)
 *   vp8gpu_decode_parsed = Frame::decode + Frame::loopfilter (decoder/frame.cc:139-250),
 *                        the narrowest seam: parsed records in, pixels out
 *   vp8gpu_frame_*     = RasterHandle / MutableRasterHandle (decoder/raster_handle.hh)
 *
 * Every function returns an int status (VP8GPU_OK or a negative VP8GPU_ERR_*), never
 * throws, and never falls back to a CPU implementation: if the CUDA device or the
 * kernels are unavailable the call fails with VP8GPU_ERR_CUDA.
 */
#ifndef VP8GPU_H
#define VP8GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes: one per reference exception class (util/exception.hh:76-98) ---- */
#define VP8GPU_OK                0
#define VP8GPU_ERR_INVALID      -1 /* Invalid: malformed bitstream                     */
#define VP8GPU_ERR_UNSUPPORTED  -2 /* Unsupported: legal VP8 the reference also rejects */
#define VP8GPU_ERR_LOGIC        -3 /* LogicError / bad argument                        */
#define VP8GPU_ERR_CUDA         -4 /* CUDA runtime failure (no device, launch error)   */
#define VP8GPU_ERR_NOMEM        -5 /* pool exhausted / allocation failure              */

/* ---- prediction modes: numbering of decoder/modemv_data.hh:41-50 ---- */
enum {
  VP8GPU_DC_PRED = 0, VP8GPU_V_PRED, VP8GPU_H_PRED, VP8GPU_TM_PRED, VP8GPU_B_PRED,
  VP8GPU_NEARESTMV, VP8GPU_NEARMV, VP8GPU_ZEROMV, VP8GPU_NEWMV, VP8GPU_SPLITMV
};
enum {
  VP8GPU_B_DC_PRED = 0, VP8GPU_B_TM_PRED, VP8GPU_B_VE_PRED, VP8GPU_B_HE_PRED, VP8GPU_B_LD_PRED,
  VP8GPU_B_RD_PRED, VP8GPU_B_VR_PRED, VP8GPU_B_VL_PRED, VP8GPU_B_HD_PRED, VP8GPU_B_HU_PRED
};
/* reference_frame of decoder/modemv_data.hh:52 */
enum { VP8GPU_REF_CURRENT = 0, VP8GPU_REF_LAST, VP8GPU_REF_GOLDEN, VP8GPU_REF_ALTREF };

/* ---- the parsed-frame records that cross the seam (host -> HBM) ----
 *
 * One frame = one vp8gpu_frame_desc + mb_cols*mb_rows vp8gpu_mb records (raster order) +
 * a token stream + the split-MV side array.  This is what the CPU entropy front end
 * emits instead of the reference's TwoD<Macroblock>/Block object graph
 * (decoder/frame.hh:56-61, block.hh:128-146).
 */

/* One non-zero quantised coefficient, exactly as decoded by tokens.cc:50-135 (NOT
 * dequantised, NOT transformed; the GPU back end does that):
 *   bits  0..15  value (int16, two's complement)
 *   bits 16..19  coefficient position in raster order inside the 4x4 block
 *                (= zigzag[index], tokens.hh:60)
 *   bits 20..24  block: 0..15 Y (raster order), 16..19 U, 20..23 V, 24 Y2
 */
typedef uint32_t vp8gpu_token;
#define VP8GPU_TOKEN(blk, pos, val) \
  ((uint32_t)(uint16_t)(val) | ((uint32_t)(pos) << 16) | ((uint32_t)(blk) << 20))
#define VP8GPU_BLK_U  16
#define VP8GPU_BLK_V  20
#define VP8GPU_BLK_Y2 24

#define VP8GPU_MB_HAS_Y2 1u /* Y2Block::coded(): y_mode is neither B_PRED nor SPLITMV */
#define VP8GPU_MB_SKIP   2u /* mb_skip_coeff (macroblock.cc:57-58).  Only present while the token
                               partitions of the frame are still to be decoded on the device
                               (vp8gpu_decode_ivf); that kernel clears it, so records seen through
                               vp8gpu_parse_frame / vp8gpu_decode_parsed never carry it */

/* 32 bytes per macroblock. */
typedef struct vp8gpu_mb {
  uint32_t tok_off;    /* first token of this MB in the frame's token stream          */
  uint16_t tok_cnt;    /* number of tokens; 0 <=> Macroblock::has_nonzero_ == false    */
  uint8_t  y_mode;     /* VP8GPU_DC_PRED .. VP8GPU_SPLITMV                             */
  uint8_t  uv_mode;    /* VP8GPU_DC_PRED .. VP8GPU_TM_PRED (intra MBs)                 */
  uint8_t  ref_frame;  /* VP8GPU_REF_*; CURRENT = intra-coded                          */
  uint8_t  segment_id; /* 0..3, row of vp8gpu_frame_desc.quant                         */
  uint8_t  lf_level;   /* loop-filter level after segment/ref/mode adjustment and the
                          single clamp of loopfilter.cc:85 (0..63); 0 = MB not filtered */
  uint8_t  flags;      /* VP8GPU_MB_*                                                  */
  int16_t  mv_x, mv_y; /* base motion vector (Y_.at(3,3)), 1/8-pel units, luma even   */
  uint32_t split_idx;  /* SPLITMV: entry in the split-MV side array                    */
  uint32_t reserved;
  uint64_t b_modes;    /* B_PRED: 16 x 4-bit VP8GPU_B_*; sub-block i in bits 4i..4i+3  */
} vp8gpu_mb;

/* 16 luma motion vectors of a SPLITMV macroblock, raster order, (x, y) pairs. */
typedef struct vp8gpu_split_mvs { int16_t mv[16][2]; } vp8gpu_split_mvs;

/* Dequantisation factors of one segment, already resolved from QuantIndices the way
 * Quantizer::Quantizer does (decoder/quantization.cc:83-93). */
typedef struct vp8gpu_quant {
  uint16_t y_dc, y_ac, y2_dc, y2_ac, uv_dc, uv_ac;
} vp8gpu_quant;

typedef struct vp8gpu_frame_desc {
  uint16_t width, height;       /* display size                                        */
  uint16_t mb_cols, mb_rows;    /* ceil(width/16), ceil(height/16)                     */
  uint8_t  key_frame;
  uint8_t  show_frame;
  uint8_t  loop_filter_level;   /* frame header value; 0 disables the whole pass
                                   (frame.cc:144)                                      */
  uint8_t  sharpness;           /* 0..7                                                */
  uint8_t  pad0[4];
  vp8gpu_quant quant[4];        /* per segment (all four equal when segmentation off)  */
  uint32_t n_tokens;
  uint32_t n_split;             /* entries in the split-MV side array                  */
  /* reference-buffer update (frame.cc:272-307), applied by the host after decoding */
  uint8_t  refresh_last, refresh_golden, refresh_alternate;
  uint8_t  copy_to_golden;      /* 0 none, 1 last, 2 alternate                         */
  uint8_t  copy_to_alternate;   /* 0 none, 1 last, 2 golden                            */
  uint8_t  pad1[3];
} vp8gpu_frame_desc;

/* ---- context, device frames ---- */

typedef struct vp8gpu_ctx vp8gpu_ctx;
typedef int32_t vp8gpu_frame_id; /* handle of a ref-counted device raster, >= 0 */

/* Create a context on CUDA device `device` for rasters of display size width x height.
 * `max_frames` bounds the device frame pool (each frame is 1.5 * W16 * H16 bytes, planar
 * Y/U/V, MB-aligned like VP8Raster, vp8_raster.hh:53 / prediction.cc:87-90); 0 = default.
 * Unlike the reference's process-global pools (raster_handle.cc:74-83) a context is
 * independent of every other context, so several frame sizes can coexist. */
int vp8gpu_ctx_create(int device, int width, int height, int max_frames, vp8gpu_ctx** out);
void vp8gpu_ctx_destroy(vp8gpu_ctx* ctx);
const char* vp8gpu_last_error(const vp8gpu_ctx* ctx); /* text of the last failure */

/* MutableRasterHandle(width,height) (raster_handle.cc:145): a writable frame, refcount 1.
 * Contents are undefined until written by upload or decode. */
int vp8gpu_frame_alloc(vp8gpu_ctx* ctx, vp8gpu_frame_id* out);
/* RasterHandle copy / destruction (shared_ptr semantics, raster_handle.hh:95-123). */
int vp8gpu_frame_retain(vp8gpu_ctx* ctx, vp8gpu_frame_id id);
int vp8gpu_frame_release(vp8gpu_ctx* ctx, vp8gpu_frame_id id);
/* Copy the MB-aligned planes host<->device. Strides in bytes; the planes are
 * 16*mb_cols x 16*mb_rows (Y) and half that (U, V).  download blocks until done. */
int vp8gpu_frame_upload(vp8gpu_ctx* ctx, vp8gpu_frame_id id, const uint8_t* y, size_t y_stride,
                        const uint8_t* u, const uint8_t* v, size_t uv_stride);
int vp8gpu_frame_download(vp8gpu_ctx* ctx, vp8gpu_frame_id id, uint8_t* y, size_t y_stride,
                          uint8_t* u, uint8_t* v, size_t uv_stride);
/* BaseRaster::dump (util/raster.cc:85-114): the display rectangle as packed planar
 * Y, U, V into `dst` (size width*height + 2*ceil(w/2)*ceil(h/2)). Blocks until done. */
int vp8gpu_frame_download_display(vp8gpu_ctx* ctx, vp8gpu_frame_id id, uint8_t* dst, size_t dst_size);
/* Same copy, asynchronous: queued behind the frame's producer; `dst` should be pinned
 * (vp8gpu_host_alloc).  vp8gpu_ctx_sync waits for everything queued so far. */
int vp8gpu_frame_download_display_async(vp8gpu_ctx* ctx, vp8gpu_frame_id id, uint8_t* dst, size_t dst_size);
/* RasterHandle::hash() (raster_handle.hh:60-75): 64-bit content hash of the MB-aligned pixels,
 * computed on the device (our own function, not boost::hash_range). Blocks until decoded. */
int vp8gpu_frame_hash(vp8gpu_ctx* ctx, vp8gpu_frame_id id, uint64_t* out);
/* BaseRaster::quality (util/raster.cc:63-66): SSIM of the macroblock-aligned luma planes, x264's
 * pixel_ssim_wxh / window count as util/ssim.cc computes it (8x8 windows at a 4-pixel step). */
int vp8gpu_frame_ssim(vp8gpu_ctx* ctx, vp8gpu_frame_id a, vp8gpu_frame_id b, double* out);
/* The whole raster (macroblock-aligned planes in the context's pitched layout, vp8gpu_frame_bytes bytes)
 * to / from a buffer that may live on the host or on this device (e.g. a tensor about to be
 * broadcast over NCCL): how reference rasters (References, decoder.hh:123-141) travel between GPUs.
 * Synchronous. */
size_t vp8gpu_frame_bytes(const vp8gpu_ctx* ctx);
int vp8gpu_frame_export(vp8gpu_ctx* ctx, vp8gpu_frame_id id, void* dst, size_t bytes);
int vp8gpu_frame_import(vp8gpu_ctx* ctx, vp8gpu_frame_id id, const void* src, size_t bytes);
int vp8gpu_ctx_sync(vp8gpu_ctx* ctx);
int vp8gpu_host_alloc(void** out, size_t bytes); /* pinned host memory */
void vp8gpu_host_free(void* p);

/* ---- the seam: Frame::decode + Frame::loopfilter on parsed records ----
 *
 * Replaces the two calls at decoder/decoder.cc:109-111 (and encoder/encoder.cc:155-156).
 * refs[] = {last, golden, alternative} as in References (decoder.hh:123-141); ignored
 * for key frames.  `out` must be a frame from vp8gpu_frame_alloc that nobody else reads.
 * The call is asynchronous with respect to the host (work is queued on `lane`, a small
 * integer naming one of the context's CUDA streams; use one lane per decoder instance so
 * independent decoders overlap on the device).  Host buffers are consumed before return.
 */
int vp8gpu_decode_parsed(vp8gpu_ctx* ctx, int lane, const vp8gpu_frame_desc* desc,
                         const vp8gpu_mb* mbs, const vp8gpu_token* tokens,
                         const vp8gpu_split_mvs* split, const vp8gpu_frame_id refs[3],
                         vp8gpu_frame_id out);

/* Batched form of the seam: n independent frames (different decoders / GOPs / streams)
 * in one set of kernel launches.  All arrays have n entries. */
typedef struct vp8gpu_job {
  const vp8gpu_frame_desc* desc;
  const vp8gpu_mb* mbs;
  const vp8gpu_token* tokens;
  const vp8gpu_split_mvs* split;
  vp8gpu_frame_id refs[3];
  vp8gpu_frame_id out;
} vp8gpu_job;
int vp8gpu_decode_batch(vp8gpu_ctx* ctx, int lane, const vp8gpu_job* jobs, int n);

/* Device-resident batch: records are uploaded once, then the kernels can be run any
 * number of times (used by bench.py for the HBM-resident `value` measurement and by
 * profilers).  `kernel_ms`, if not NULL, receives the device time of this run measured
 * with CUDA events on the launching stream. */
typedef struct vp8gpu_resident_batch vp8gpu_resident_batch;
int vp8gpu_batch_upload(vp8gpu_ctx* ctx, const vp8gpu_job* jobs, int n, vp8gpu_resident_batch** out);
int vp8gpu_batch_run(vp8gpu_ctx* ctx, int lane, vp8gpu_resident_batch* b, float* kernel_ms);
void vp8gpu_batch_free(vp8gpu_ctx* ctx, vp8gpu_resident_batch* b);
/* Run n resident batches back to back on one lane (e.g. the 30 frame positions of a set of
 * GOPs) without host synchronisation in between; *total_ms = device time from the first launch
 * to the last kernel's end (CUDA events on the launching stream). */
int vp8gpu_batches_run(vp8gpu_ctx* ctx, int lane, vp8gpu_resident_batch* const* batches, int n, float* total_ms);
/* Run one resident batch with a CUDA event between the kernels:
 * kernel_ms[0..2] = k_inter, k_intra, k_loopfilter device time (0 for a kernel that did not run). */
int vp8gpu_batch_run_timed(vp8gpu_ctx* ctx, int lane, vp8gpu_resident_batch* b, float kernel_ms[3]);
/* kernels launched by this context since creation (bench.py's gpu_launches) */
uint64_t vp8gpu_launch_count(const vp8gpu_ctx* ctx);
/* rasters of the context's pool that are currently handed out (RasterHandle count of the reference's pool,
 * raster_handle.cc:103-122); after an error every raster a call took must have come back */
int vp8gpu_frames_in_use(const vp8gpu_ctx* ctx);

/* ---- CPU entropy front end: DecoderState::parse_and_apply ----
 *
 * vp8gpu_state is DecoderState (decoder.hh:190-225): probability tables, segmentation
 * (incl. the persistent segment map) and loop-filter adjustments.  It is a plain value:
 * clone is a deep copy, equal/hash follow DecoderState::operator== / hash.
 */
typedef struct vp8gpu_state vp8gpu_state;
int vp8gpu_state_create(int width, int height, vp8gpu_state** out);
int vp8gpu_state_clone(const vp8gpu_state* s, vp8gpu_state** out);
void vp8gpu_state_destroy(vp8gpu_state* s);
int vp8gpu_state_equal(const vp8gpu_state* a, const vp8gpu_state* b);
uint64_t vp8gpu_state_hash(const vp8gpu_state* s);
/* DecoderState::serialize / deserialize (decoder.cc:283-330): the DECODER_STATE record of the reference's
 * tag-length-value format (enc_state_serializer.hh), byte-compatible with the reference.  serialize returns
 * the size needed and writes only if cap suffices.  Together with vp8gpu_frame_export / _import this moves a Decoder between processes
 * or GPUs (alfalfa_b200/multigpu.py broadcast_decoder: NCCL broadcast of the reference rasters). */
size_t vp8gpu_state_serialize(const vp8gpu_state* s, uint8_t* out, size_t cap);
int vp8gpu_state_deserialize(const uint8_t* data, size_t len, vp8gpu_state** out);

/* A parsed frame (KeyFrame / InterFrame, frame.hh:126-127) in flat form. The arrays are
 * owned by the vp8gpu_parsed object and stay valid until it is destroyed or reused. */
typedef struct vp8gpu_parsed vp8gpu_parsed;
int vp8gpu_parsed_create(vp8gpu_parsed** out);
void vp8gpu_parsed_destroy(vp8gpu_parsed* p);
const vp8gpu_frame_desc* vp8gpu_parsed_desc(const vp8gpu_parsed* p);
const vp8gpu_mb* vp8gpu_parsed_mbs(const vp8gpu_parsed* p);
const vp8gpu_token* vp8gpu_parsed_tokens(const vp8gpu_parsed* p);
const vp8gpu_split_mvs* vp8gpu_parsed_split(const vp8gpu_parsed* p);

/* Decoder::decompress_frame + parse_frame<KeyFrame|InterFrame> (decoder.cc:83-98):
 * parse one compressed VP8 frame, update `state` exactly as parse_and_apply does, and
 * fill `out`.  Errors: INVALID (truncated / bad start code / bad partition sizes),
 * UNSUPPORTED (version != 0, scaling, colour space / clamping bits, simple filter,
 * size != state size), mirroring uncompressed_chunk.cc:34-130 and frame_header.hh:213-295.
 * On INVALID / UNSUPPORTED `state` is unchanged; after VP8GPU_ERR_NOMEM it must be discarded. */
int vp8gpu_parse_frame(vp8gpu_state* state, const uint8_t* data, size_t len, vp8gpu_parsed* out);

/* Frame::serialize( probability_tables ) of a parsed frame (encoder/serializer.cc:388-405), the inverse of
 * vp8gpu_parse_frame.  The reference's Frame object keeps its header and every macroblock's labels, so its
 * serialize() reproduces the input byte for byte (gate: src/tests/roundtrip.cc:93-112, tests/roundtrip-verify.test);
 * here a vp8gpu_parsed keeps them when vp8gpu_parsed_keep_labels( p, 1 ) was called before the parse: the header
 * decisions as coded, mb_skip_coeff of every macroblock, SPLITMV layouts and sub-vector labels.  Modes, vectors
 * and the DCT partitions are re-written from the flat records with the decoder's contexts.
 * vp8gpu_parsed_serialize: VP8GPU_ERR_LOGIC if the labels were not kept, VP8GPU_ERR_NOMEM if cap is too small
 * (*size = needed). */
int vp8gpu_parsed_keep_labels(vp8gpu_parsed* p, int on);
int vp8gpu_parsed_serialize(const vp8gpu_parsed* p, uint8_t* out, size_t cap, size_t* size);

/* Same contract and same output as vp8gpu_parse_frame, with the front end split the B200 way: the
 * host decodes the first partition (frame header, macroblock modes, motion vectors: macroblock.cc:
 * 44-456), the device decodes the DCT partitions (Frame::parse_tokens, frame.cc:122-137;
 * tokens.cc:50-135) and the completed records are copied back into `out`.  Synchronous; the
 * building block behind VP8GPU_OPT_DEVICE_TOKENS, exported so the records can be checked. */
int vp8gpu_parse_frame_device(vp8gpu_ctx* ctx, vp8gpu_state* state, const uint8_t* data, size_t len,
                              vp8gpu_parsed* out);

/* Context options.  VP8GPU_OPT_DEVICE_TOKENS (default 1): vp8gpu_decode_ivf decodes the DCT
 * partitions on the device (one thread per frame, many frames in flight) instead of on the host
 * workers; 0 = the host workers parse everything.  Output is identical either way. */
#define VP8GPU_OPT_DEVICE_TOKENS 1
int vp8gpu_ctx_set_option(vp8gpu_ctx* ctx, int option, int value);

/* ---- Decoder (decoder.hh:244-300): DecoderState + References, explicit state passing ---- */
typedef struct vp8gpu_decoder vp8gpu_decoder;
/* Decoder(width,height): references start as one shared all-zero raster. */
int vp8gpu_decoder_create(vp8gpu_ctx* ctx, vp8gpu_decoder** out);
/* Decoder(DecoderState, References): takes a copy of `state` and a reference on each frame. */
int vp8gpu_decoder_create_from(vp8gpu_ctx* ctx, const vp8gpu_state* state,
                               const vp8gpu_frame_id refs[3], vp8gpu_decoder** out);
/* Copy construction: O(1) in pixels, the clone shares the three reference rasters. */
int vp8gpu_decoder_clone(const vp8gpu_decoder* d, vp8gpu_decoder** out);
void vp8gpu_decoder_destroy(vp8gpu_decoder* d);
/* Decoder::get_frame_output (decoder.cc:125-135): parse + decode one compressed frame.
 * *shown = show_frame; *out = the decoded raster with one reference owned by the caller
 * (release it with vp8gpu_frame_release).  Asynchronous on the decoder's lane. */
int vp8gpu_decoder_decode(vp8gpu_decoder* d, const uint8_t* data, size_t len, int* shown,
                          vp8gpu_frame_id* out);
/* Decoder::decode_frame (decoder.cc:101-118) for an already parsed frame; `parsed` must
 * have been produced by vp8gpu_parse_frame on this decoder's state (vp8gpu_decoder_state). */
int vp8gpu_decoder_decode_parsed(vp8gpu_decoder* d, const vp8gpu_parsed* parsed, int* shown,
                                 vp8gpu_frame_id* out);
/* on != 0: vp8gpu_decoder_decode leaves the DCT partitions to the device (same stream as the pixel
 * kernels, so this trades latency for host time); default off.  Output is identical. */
int vp8gpu_decoder_set_device_tokens(vp8gpu_decoder* d, int on);
vp8gpu_state* vp8gpu_decoder_state(vp8gpu_decoder* d);            /* get_state (borrowed) */
int vp8gpu_decoder_references(const vp8gpu_decoder* d, vp8gpu_frame_id refs[3]); /* borrowed */
int vp8gpu_decoder_lane(const vp8gpu_decoder* d);
/* Decoder::get_hash (decoder.hh:279-292, DecoderHash): one value over the state and the contents of the
 * three reference rasters (hashed on the device; the value is this library's, not boost's) -- equal
 * decoders hash equally, which is what the reference uses it for (frame-graph bookkeeping, minihash
 * fields of IVF frames).  minihash = its 32-bit fold. */
int vp8gpu_decoder_hash(vp8gpu_decoder* d, uint64_t* out);
/* Decoder::serialize / Decoder::deserialize (decoder.cc:54-81) in the reference's own tag-length-value
 * format (decoder/enc_state_serializer.hh:43-190): DECODER { DECODER_STATE { size, PROB_TABLE, optional
 * SEGM_ABS|SEGM_REL, optional FILT_ADJ } REFERENCES { display size, REF_LAST { Y, U, V planes of the
 * macroblock-aligned raster } } }.  Blobs are interchangeable with the reference's (xc-enc -O / -I state files,
 * EncoderStateDeserializer::build<Decoder>): as there, only the LAST reference travels and a deserialised
 * Decoder has golden = alternative = last.  serialize: VP8GPU_ERR_NOMEM if cap is too small (*size = needed).
 * vp8gpu_state_serialize / _deserialize carry the DECODER_STATE record alone. */
int vp8gpu_decoder_serialize(vp8gpu_decoder* d, uint8_t* out, size_t cap, size_t* size);
int vp8gpu_decoder_deserialize(vp8gpu_ctx* ctx, const uint8_t* data, size_t len, vp8gpu_decoder** out);
/* Decoder::operator== (decoder.cc:153): state equal and the three rasters pixel-equal. */
int vp8gpu_decoder_equal(vp8gpu_decoder* a, vp8gpu_decoder* b, int* equal);

/* ---- the exchange step: reference rasters between GPUs (SURVEY.md 8e; References, decoder.hh:123-141) ----
 * GOPs and streams shard across GPUs without any exchange.  A GOP that continues on another GPU (a long
 * single-GOP stream split across ranks, BASELINE.json configs[3]) needs the producer's reference rasters: they
 * are broadcast device to device with NCCL over NVLink, queued on the context's lane stream between the kernels
 * that wrote them and the kernels that will read them (no host synchronisation, no staging).  One communicator
 * per context and rank set, created collectively like ncclCommInitRank: rank 0 makes the 128-byte id
 * (vp8gpu_comm_unique_id) and hands it to the other ranks by whatever channel the caller has.  NCCL itself is
 * resolved at run time; without it these calls return VP8GPU_ERR_UNSUPPORTED.
 *   vp8gpu_comm_broadcast_frames  collective; ids[i] on the root = the rasters to send, on the other ranks =
 *                                 rasters from vp8gpu_frame_alloc that receive them (same order everywhere)
 *   vp8gpu_comm_broadcast_bytes   collective, synchronous: a small host buffer (vp8gpu_state_serialize output) */
typedef struct vp8gpu_comm vp8gpu_comm;
int vp8gpu_comm_unique_id(uint8_t out[128]);
int vp8gpu_comm_create(vp8gpu_ctx* ctx, int rank, int nranks, const uint8_t unique_id[128], vp8gpu_comm** out);
void vp8gpu_comm_destroy(vp8gpu_comm* comm);
int vp8gpu_comm_broadcast_frames(vp8gpu_comm* comm, int root, int lane, const vp8gpu_frame_id* ids, int n);
int vp8gpu_comm_broadcast_bytes(vp8gpu_comm* comm, int root, void* buf, size_t bytes);
int vp8gpu_comm_rank(const vp8gpu_comm* comm);
int vp8gpu_comm_size(const vp8gpu_comm* comm);

/* ---- whole-stream helper (decoder/player.cc:60-143, FilePlayer) ----
 * Decode every frame of an in-memory IVF with `threads` host workers, one GOP (key frame
 * to next key frame) per task, each worker driving its own Decoder on its own lane.  The
 * display rectangles of the shown frames are written, in stream order, to `dst`
 * (may be NULL to leave the frames on the device).  *n_shown / *n_decoded are outputs. */
int vp8gpu_decode_ivf(vp8gpu_ctx* ctx, const uint8_t* ivf, size_t len, int threads, uint8_t* dst,
                      size_t dst_size, uint32_t* n_decoded, uint32_t* n_shown);

/* ---- encoder side: bitstream writer (Frame::serialize, encoder/serializer.cc:388-829) ----
 * Turns flat records (modes / vectors / quantised-coefficient tokens, as produced by the device
 * encode kernels or by vp8gpu_parse_frame) into one compressed VP8 frame: frame tag, header, mode
 * partition, one DCT partition.  Written subset: no segmentation, no loop-filter deltas, LAST
 * reference only.  Returns VP8GPU_ERR_UNSUPPORTED if a record is outside that subset and
 * VP8GPU_ERR_NOMEM if `cap` is too small (*size then holds the needed size). */
typedef struct vp8gpu_encode_header {
  uint16_t width, height;
  uint8_t key_frame, show_frame;
  uint8_t y_ac_qi;            /* 0..127, all quantiser deltas zero */
  uint8_t loop_filter_level;  /* 0..63 */
  uint8_t sharpness;          /* 0..7 */
  uint8_t optimize_token_probs;
  uint8_t pad[2];
} vp8gpu_encode_header;
int vp8gpu_serialize_frame(const vp8gpu_encode_header* hdr, const vp8gpu_mb* mbs, const vp8gpu_token* tokens,
                           const vp8gpu_split_mvs* split, uint8_t* out, size_t cap, size_t* size);

/* The rest of the frame header (frame_header.hh:37-131, 213-325) for vp8gpu_serialize_frame_ex: with it
 * the writer covers the whole format -- segmentation (records' segment_id), loop-filter deltas,
 * quantiser deltas, 1..8 DCT partitions, LAST / GOLDEN / ALTREF references with sign bias (records'
 * ref_frame), reference refresh / copy flags, persistent coefficient probabilities.  Used to synthesise
 * feature-complete test streams (tools/make_feature_stream.py); what they decode to is defined by the
 * reference decoder. */
typedef struct vp8gpu_encode_features {
  uint8_t log2_partitions;                 /* 0..3 */
  uint8_t segmentation_enabled, update_mb_segmentation_map, update_segment_feature_data, segment_feature_absolute;
  int8_t  segment_quant[4], segment_lf[4];
  uint8_t segment_tree_probs[3];           /* 255 = not sent */
  uint8_t lf_delta_enabled, lf_delta_update;
  int8_t  ref_lf_delta[4], mode_lf_delta[4];
  int8_t  y_dc_delta, y2_dc_delta, y2_ac_delta, uv_dc_delta, uv_ac_delta; /* -15..15 */
  uint8_t refresh_golden, refresh_alternate, refresh_last, refresh_entropy_probs;
  uint8_t copy_to_golden, copy_to_alternate;   /* 0 none, 1 last frame, 2 the other buffer */
  uint8_t sign_bias_golden, sign_bias_alternate;
  uint8_t pad[3];
  uint8_t* saved_coef_probs;  /* 1056 bytes of stream state (DecoderState's coefficient probabilities),
                                 read and, with refresh_entropy_probs, updated; NULL = stateless */
} vp8gpu_encode_features;
int vp8gpu_serialize_frame_ex(const vp8gpu_encode_header* hdr, const vp8gpu_encode_features* features,
                              const vp8gpu_mb* mbs, const vp8gpu_token* tokens, const vp8gpu_split_mvs* split,
                              uint8_t* out, size_t cap, size_t* size);

/* ---- Encoder (encoder/encoder.hh:345-382), first slice ----
 * Explicit state: the encoder owns its LAST reference (the reconstruction of the previous frame);
 * the first frame is a key frame, later frames are inter frames (encoder.cc:559-590).  Source planes
 * are the display-size Y, U, V planes on the host; they are edge-extended to macroblock size like
 * the reference's input reader does.  The emitted frame is a standard VP8 frame. */
typedef struct vp8gpu_encoder vp8gpu_encoder;
int vp8gpu_encoder_create(vp8gpu_ctx* ctx, vp8gpu_encoder** out);
void vp8gpu_encoder_destroy(vp8gpu_encoder* enc);
/* Encoder( const Encoder & ) (encoder/encoder.cc:92-102): an independent copy that shares the (immutable,
 * reference-counted) reference rasters; Salsify copies its encoder twice per frame and encodes on both
 * copies concurrently (salsify/salsify-sender.cc:492-518). */
int vp8gpu_encoder_clone(const vp8gpu_encoder* src, vp8gpu_encoder** out);
/* Encoder( const Decoder &, two_pass, quality ) (encoder/encoder.hh:350-351): continue a stream from a
 * decoder's state and references; the next frame is an inter frame. */
int vp8gpu_encoder_create_from_decoder(vp8gpu_ctx* ctx, vp8gpu_decoder* dec, vp8gpu_encoder** out);
/* Encoder::export_decoder (encoder/encoder.hh:378): a new Decoder in the state a receiver is in after the
 * frames emitted so far (DecoderState + the three references, shared); the caller destroys it. */
int vp8gpu_encoder_export_decoder(vp8gpu_encoder* enc, vp8gpu_decoder** out);
/* Encoder::minihash (encoder/encoder.hh:382) = export_decoder().minihash() */
int vp8gpu_encoder_minihash(vp8gpu_encoder* enc, uint32_t* out);
/* Which bitstream writer the encoder uses.  0 (default): the reference Encoder's own header rules (every
 * changed token probability is sent, explicit zero loop-filter deltas, one DCT partition): the emitted frames
 * are byte-identical to the reference encoder's.  1: compact -- only the probability updates that pay, eight
 * DCT partitions written on eight host threads (same decisions and reconstruction, fewer bytes, faster). */
int vp8gpu_encoder_set_writer(vp8gpu_encoder* enc, int mode);
/* Encoder( ..., two_pass, ... ) (encoder/encoder.hh:347-351): with on != 0 a key frame is coded twice, the second pass
 * with trellis quantisation (Encoder::trellis_quantize, check_reset_y2, encoder/encoder.cc:198-408) priced by the token
 * costs of the default tables; inter frames are coded once either way, as in the reference. */
int vp8gpu_encoder_set_two_pass(vp8gpu_encoder* enc, int on);
/* Encoder( ..., quality ) (encoder/encoder.hh:56-60, 346-351), in the reference enum's order.  REALTIME (the default) is
 * Salsify's setting: inter frames never try B_PRED, NEWMV is searched at every fourth macroblock column and row, and
 * every frame remembers its quantiser and loop-filter level to narrow the next frame's searches (encoder.cc:164-167).
 * BEST is ExCamera's xc-enc default: inter frames try B_PRED at every macroblock, NEWMV is searched everywhere, and
 * nothing is remembered -- every target-size search bisects over [4, 127], every loop-filter search walks up from 0.
 * It applies to every encode_*, estimate and re-encoding call; the emitted frames are byte-identical to the reference
 * encoder's at the same setting.  Valid until the encoder writes its first frame (a clone inherits the setting and
 * whether it may still change); VP8GPU_ERR_LOGIC after that and for other values. */
#define VP8GPU_QUALITY_BEST     0
#define VP8GPU_QUALITY_REALTIME 1
int vp8gpu_encoder_set_quality(vp8gpu_encoder* enc, int quality);
/* Encoder::encode_with_quantizer (encoder.cc:559-590) */
int vp8gpu_encoder_encode_with_quantizer(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u,
                                         const uint8_t* v, size_t uv_stride, int y_ac_qi, uint8_t* out, size_t cap,
                                         size_t* size);
/* Encoder::encode_with_target_size (encoder.cc:592-629): smallest quantiser index in the searched
 * range whose frame fits `target_size` bytes; *chosen_qi (optional) receives it.  The probes of the bisection
 * (Encoder::estimate_frame_size at up to 33 quantiser indices) are coded in one kernel launch and the search walks the
 * finished results in the reference's order; likewise the trials of the loop-filter search of every encode_* call
 * (encoder.cc:460-508).  The emitted bytes do not depend on that (VP8GPU_ENC_SPECULATE=0 in the environment, read once
 * per process, runs both searches candidate by candidate). */
int vp8gpu_encoder_encode_with_target_size(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u,
                                           const uint8_t* v, size_t uv_stride, size_t target_size, uint8_t* out,
                                           size_t cap, size_t* size, int* chosen_qi);
/* Encoder::encode_with_minimum_ssim (encoder.cc:510-557, 577-590) as it is meant: the coarsest quantiser index whose
 * reconstruction still reaches `minimum_ssim` (luma SSIM against the source after the loop filter).  NOT byte-compatible
 * with the reference here, on purpose: its search calls encode_raster( raster, quant_indices, true ) -- the `true` lands on
 * update_state, compute_ssim stays false (encoder.hh:336-337) -- so every candidate reports SSIM 0, the bisection walks
 * down to index 0 and the frame is coded at the finest quantiser whatever was asked for (oracle/_ref/ref_encode with
 * REF_MIN_SSIM shows it). */
int vp8gpu_encoder_encode_with_minimum_ssim(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u,
                                            const uint8_t* v, size_t uv_stride, double minimum_ssim, uint8_t* out,
                                            size_t cap, size_t* size, int* chosen_qi);
/* Encoder::estimate_frame_size (encoder.hh:376, size_estimation.cc): the size in bytes the frame would
 * have at quantiser index y_ac_qi, estimated like the reference does: every fourth macroblock column and
 * row is coded as a (width / 4) x (height / 4) frame with the current probability tables and its size
 * multiplied by 16 (size_estimation.cc:36-181).  Does not change the encoder's state. */
int vp8gpu_encoder_estimate_frame_size(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u,
                                       const uint8_t* v, size_t uv_stride, int y_ac_qi, size_t* size);
/* ---- re-encoding (encoder/reencode.cc; ExCamera's "xc-enc --reencode", frontend/xc-enc.cc:262-327) ----
 * The chunk's frames as they were coded independently ("prediction frames") are parsed by their own decoder
 * state with vp8gpu_parsed_keep_labels on (the reference keeps them as KeyFrame / InterFrame objects); the Encoder
 * was built from the Decoder a receiver has when the chunk starts (vp8gpu_encoder_create_from_decoder).
 *
 * vp8gpu_encoder_update_residues = Encoder::update_residues + write_frame (reencode.cc:131-313, encoder.cc:146-170):
 * the prediction frame's header, modes, vectors and reference choices are kept; the residues are recomputed on the
 * device against THIS encoder's references so that the frame decodes as close as possible to the target planes
 * (display size, host); the emitted frame is then decoded like any receiver would to advance the Encoder.
 * y_ac_qi < 0 keeps the frame's own quantiser index (its deltas are always kept); last_frame != 0 makes the frame
 * refresh all three references (reencode.cc:269-275).  VP8GPU_ERR_UNSUPPORTED for frames with segmentation (the
 * reference writes a frame there that does not decode to its own reconstruction). */
int vp8gpu_encoder_update_residues(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u,
                                   const uint8_t* v, size_t uv_stride, const vp8gpu_parsed* prediction_frame, int y_ac_qi,
                                   int last_frame, uint8_t* out, size_t cap, size_t* size);
/* Encoder::reencode_as_interframe + write_frame (reencode.cc:39-129, 343-351): the chunk's initial key frame is coded
 * again as an inter frame predicted from this encoder's LAST (the reference's inter-frame decision loop on the
 * device), at the key frame's quantiser indices with y_ac_qi replaced, with its sharpness, refreshing all three
 * references.  VP8GPU_ERR_UNSUPPORTED for a key frame with segmentation (like the reference, reencode.cc:49-51). */
int vp8gpu_encoder_reencode_as_interframe(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u,
                                          const uint8_t* v, size_t uv_stride, const vp8gpu_parsed* key_frame, int y_ac_qi,
                                          uint8_t* out, size_t cap, size_t* size);
/* Encoder::write_frame( KeyFrame ) (encoder.cc:146-176) as Encoder::reencode uses it for a key frame that is
 * kept (reencode.cc:363-365): the frame's own bytes are emitted and the Encoder moves past it. */
int vp8gpu_encoder_write_frame(vp8gpu_encoder* enc, const vp8gpu_parsed* frame, uint8_t* out, size_t cap, size_t* size);
/* header().quant_indices.y_ac_qi of a frame parsed with vp8gpu_parsed_keep_labels (Encoder::reencode blends the
 * quantisers of neighbouring prediction frames, reencode.cc:334-361); -1 without kept labels */
int vp8gpu_parsed_y_ac_qi(const vp8gpu_parsed* p);

/* EncoderStats (encoder.hh:118-127) of the last frame, at either quality; any pointer may be NULL. */
int vp8gpu_encoder_stats(const vp8gpu_encoder* enc, double* ssim, int* loop_filter_level, int* y_ac_qi);
/* Diagnostic: where the host spent the last encode_with_quantizer / encode_with_target_size call, wall-clock
 * milliseconds per phase (each phase ends with the device work it queued being finished, so device time is inside):
 * [0] source upload, [1] size estimates: kernel launch(es) + wait, [2] size estimates: download + serialise the probes
 * the search visited, [3] the full pass (decisions, transforms, reconstruction) incl. download of records and tokens,
 * [4] loop-filter search (the frame writer runs next to it), [5] the frame writer's own work (host thread, next to [4]; its wait for
 * the level is not counted), [6] state update (parse of the emitted frame's first partition, reference hand-over), [7] the whole
 * call.  n <= 8 values are written. */
int vp8gpu_encoder_timeline(const vp8gpu_encoder* enc, double* ms, int n);
/* the reconstruction of the last encoded frame = the decoder's LAST reference after decoding it
 * (Encoder::export_decoder, encoder.hh:378); the caller releases the returned raster */
int vp8gpu_encoder_reconstruction(vp8gpu_encoder* enc, vp8gpu_frame_id* out);

/* Host-side time accounting of the last vp8gpu_decode_ivf call, seconds summed over threads:
 * [0] parsing, [1] workers waiting for the dispatcher, [2] workers waiting for DMA, [3] dispatcher
 * in submit, [4] dispatcher queueing downloads, [5] dispatcher idle, [6] batches, [7] frames. */
void vp8gpu_decode_ivf_stats(const vp8gpu_ctx* ctx, double out[8]);

#ifdef __cplusplus
}
#endif
#endif /* VP8GPU_H */
