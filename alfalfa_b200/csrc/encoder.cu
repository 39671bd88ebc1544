// encoder.cu -- host side of the encoder path: Encoder (encoder/encoder.hh:345-382) on the device.
//
// SURVEY.md 8a row a16 + 8 f3: encode_with_quantizer / encode_with_target_size / encode_with_minimum_ssim /
// estimate_frame_size, the two-pass key frame, and re-encoding (update_residues, reencode_as_interframe,
// write_frame).  The per-macroblock decisions are the reference's (k_enc_rd in kernels.cu: rdcost, B_PRED trial,
// motion-vector census + diamond search, chroma by distortion, trellis in the second pass); this file is the
// frame-level policy around them, statement for statement the reference's: the bisection over y_ac_qi on sampled
// size estimates (encoder.cc:592-629, size_estimation.cc), the SSIM-driven loop-filter search (encoder.cc:460-508),
// the writer's header rules (serializer.h RefWriterState) -- the emitted frames are byte-identical to the reference
// encoder's (tests/test_gpu_encoder.py) -- and the closed loop: the emitted frame decodes (reference decoder,
// oracle, this library) to exactly the reconstruction the encoder keeps as its LAST reference, which is what
// Encoder::export_decoder (encoder.hh:378) promises.
//
// What differs from the reference is only the ORDER IN TIME of independent work: the candidates of the two
// searches do not depend on each other (a size estimate is a function of the source, the references and y_ac_qi;
// a loop-filter trial of the reconstruction and the level), and a wavefront kernel lasts as long for one frame as
// for thirty (DESIGN.md section 3), so the candidates a search can still visit are coded in ONE launch
// (estimate_batch_launch, filter_batch) and the search then walks over finished results in the reference's order.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <condition_variable>
#include <mutex>
#include <utility>
#include <vector>

#include "../../include/vp8gpu.h"
#include "enc_costs.h"
#include "engine.hpp"
#include "hostpool.h"
#include "parser.h"
#include "serializer.h"
#include "vp8_enc_tables.h"
#include "vp8_tables.h"

using vp8::Engine;

// shared with capi.cc
extern "C" Engine* vp8gpu_ctx_engine(vp8gpu_ctx* ctx);
extern "C" int vp8gpu_ctx_next_lane(vp8gpu_ctx* ctx);
extern "C" const vp8::ParsedFrame* vp8gpu_parsed_frame(const vp8gpu_parsed* p);
extern "C" int vp8gpu_decoder_decode_known_tokens(vp8gpu_decoder* d, const uint8_t* data, size_t len, const vp8gpu_mb* enc_mbs,
                                                  const vp8gpu_token* enc_tokens, uint32_t n_tok, int* shown, vp8gpu_frame_id* out);

struct vp8gpu_encoder {
  vp8gpu_ctx* ctx = nullptr;
  Engine* e = nullptr;
  int lane = 0;
  bool has_state = false;
  int refs[3] = {-1, -1, -1};  // References: last, golden, alternative (the encoder only ever predicts from LAST
                               // and only refreshes LAST, encode_inter.cc:245,587-589; the others stay the key frame)
  int src = -1;                // device raster holding the (edge-extended) source frame
  int quality = VP8GPU_QUALITY_REALTIME;  // encode_quality_ (encoder.hh:133)
  bool quality_fixed = false;  // a frame has been written (by this Encoder or the one it was copied from)
  int last_qi = -1;            // last_y_ac_qi_: what the target-size search remembers (REALTIME_QUALITY only, encoder.cc:164-167)
  int last_lf = -1;            // loop_filter_level_ (encoder.hh:144): -1 = not initialised; what the loop-filter search remembers
  int stat_qi = -1, stat_lf = -1;  // quantiser and loop-filter level of the last frame, at either quality (vp8gpu_encoder_stats)
  bool mv_costs_filled = false;  // Costs::fill_mv_component_costs has run (encode_inter.cc:601: at the start of the first full
                                 // inter-frame pass of this Encoder or of the one it was copied from; reencode.cc:85)
  bool mv_sad_filled = false;    // Costs::fill_mv_sad_costs has run (encode_inter.cc:602 only)
  uint32_t rd_rate = 300, rd_dist = 1;  // RATE_MULTIPLIER / DISTORTION_MULTIPLIER (encoder.hh:152-153) as the last
                                        // update_rd_multipliers left them; a copy starts from the defaults again
  int lf_sharpness = 0;          // sharpness_level of the frame being built (0 for the Encoder's own frames)
  uint8_t tab_mv_probs[38];      // the motion-vector probabilities the rate tables on the device were built from
  bool two_pass = false;         // Encoder( ..., two_pass, ... ) (encoder.hh:347): key frames get a second, trellis pass
  uint8_t* d_trellis = nullptr;  // TrellisTables | y2_prev[n_mbs] on the device (two-pass only)
  double last_ssim = -1.0;     // encode_stats_.ssim of the last frame
  vp8::State* dec_state = nullptr;  // DecoderState a decoder has after the frames emitted so far (export_decoder)
  // device scratch: EncJob | DevJob | sync ints | mbs | tokens | rate tables
  uint8_t* dev = nullptr;
  size_t off_encjob = 0, off_sync = 0, off_mbs = 0, off_tokens = 0, off_tab = 0, dev_bytes = 0;
  uint32_t tok_cap = 0;
  uint8_t* d_split = nullptr;  // update_residues: the prediction frame's split-MV side array on the device
  size_t split_cap = 0;
  // pinned host buffers
  uint8_t* h_hdr = nullptr;      // EncJob + DevJob
  vp8gpu_mb* h_mbs = nullptr;
  vp8gpu_token* h_tokens = nullptr;
  uint8_t* h_src = nullptr;      // padded planes
  uint32_t* h_count = nullptr;
  uint64_t stat_frames = 0;
  int pending_out = -1;          // output raster of a pass that has been launched but not collected
  vp8::ParsedFrame* scratch = nullptr;  // for re-parsing the emitted frame into dec_state
  // Bitstream writer.  0 (default): the reference Encoder's own header rules and one DCT partition
  // (serializer.h RefWriterState) -- byte-identical output; 1: compact -- only token-probability updates that
  // pay, no zero loop-filter deltas, eight DCT partitions written on eight host threads.
  int writer = 0;
  double tl[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // vp8gpu_encoder_timeline: milliseconds per phase of the last encode call
  // speculative size estimates (estimate_batch_launch): EncJob[kEstMax] | ticket, token counters, row progress |
  // records, token pools and reconstruction rasters of every candidate -- private to this Encoder, allocated on
  // the first target-size search
  uint8_t* d_est = nullptr;
  uint8_t* h_est = nullptr;      // pinned: EncJob[kEstMax] | token counts
  size_t est_off_sync = 0, est_off_mbs = 0, est_off_tokens = 0, est_off_out = 0, est_out_stride = 0;
  uint32_t est_tok_cap = 0;      // tokens per candidate
  int est_n = 0;                 // candidates of the batch whose results are on the device now (0: none)
  int est_qi[33];
  uint32_t est_rate[33], est_dist[33];
  // header state of the reference's four frame objects: key_frame_, inter_frame_, subsampled_*_ (encoder.hh:128-142)
  vp8::EncodeFeatures::RefWriterState ref_key, ref_inter, ref_sub_key, ref_sub_inter;
};

namespace {
double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
struct Phase {  // adds the time between construction and destruction to one slot of the timeline
  double* slot;
  double t0;
  explicit Phase(double* s) : slot(s), t0(now_ms()) {}
  ~Phase() { *slot += now_ms() - t0; }
};
constexpr int kEstMax = 33;   // size estimates per launch: a whole search range of last_y_ac_qi +- 16 (encoder.cc:604-611)
constexpr int kLfMax = 8;     // loop-filter trials per launch (steady state: the last level +- 1, encoder.cc:466-471; a first frame walks up from 0)
constexpr size_t kHdrBytes = 512 + 512 * kLfMax;  // pinned / device header area: EncJob | DevJob[kLfMax]
static_assert(sizeof(vp8::EncJob) <= 512 && sizeof(vp8::DevJob) <= 512, "header area slots");
size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
int clamp_q(int q) { return q < 0 ? 0 : (q > 127 ? 127 : q); }
vp8gpu_quant make_quant(int qi) {  // Quantizer::Quantizer, quantization.cc:83-93 (all deltas zero)
  vp8gpu_quant q;
  q.y_ac = k_ac_q[clamp_q(qi)];
  q.y_dc = k_dc_q[clamp_q(qi)];
  q.y2_ac = static_cast<uint16_t>(k_ac_q[clamp_q(qi)] * 155 / 100);
  q.y2_dc = static_cast<uint16_t>(k_dc_q[clamp_q(qi)] * 2);
  q.uv_ac = k_ac_q[clamp_q(qi)];
  q.uv_dc = k_dc_q[clamp_q(qi)];
  if (q.y2_ac < 8) q.y2_ac = 8;
  if (q.uv_dc > 132) q.uv_dc = 132;
  return q;
}
#define CUE(call)                                                       \
  do {                                                                  \
    cudaError_t e__ = (call);                                           \
    if (e__ != cudaSuccess) return enc->e->cuda_fail(e__, #call);       \
  } while (0)

// macroblock grid of a pass: the whole frame, or the frame Encoder::estimate_size codes -- a
// (width / 4) x (height / 4) frame whose macroblock (c, r) is source macroblock (4c, 4r) (size_estimation.cc:36-99)
void pass_dims(const vp8gpu_encoder* enc, int sub, int* w, int* h, int* cols, int* rows) {
  *w = sub == 1 ? enc->e->width() : (uint16_t)(enc->e->width() / sub);
  *h = sub == 1 ? enc->e->height() : (uint16_t)(enc->e->height() / sub);
  *cols = (*w + 15) / 16;
  *rows = (*h + 15) / 16;
}

// launch half of a pass: everything up to the asynchronous download of the token count and the records
// reenc != nullptr: a pass of Encoder::reencode_as_interframe (reencode.cc:39-129) -- the quantiser comes with the
// call (a key frame's indices with another y_ac_qi), update_rd_multipliers and fill_mv_sad_costs are NOT run
// trellis: the second pass of a two-pass key frame (k_enc_rd<true>; enc->d_trellis holds the tables and the first
// pass's Y2 flags)
int encode_launch(vp8gpu_encoder* enc, bool key, int qi, int sub, const vp8gpu_quant* reenc = nullptr, bool trellis = false) {
  Engine* e = enc->e;
  const vp8::Geom& g = e->geom();
  int pw, ph, cols, rows;
  pass_dims(enc, sub, &pw, &ph, &cols, &rows);
  if (cols < 1 || rows < 1) return e->fail(VP8GPU_ERR_UNSUPPORTED, "frame too small for the sampled size estimate");
  const size_t n_mbs = (size_t)cols * rows;
  if (int rc = e->ensure_lane(enc->lane)) return rc;
  cudaStream_t s = e->stream(enc->lane);
  int out = -1;
  int rc = e->frame_alloc(&out);
  if (rc != VP8GPU_OK) return rc;
  int ids[3] = {enc->src, out, enc->refs[0]};
  rc = e->acquire_frames(enc->lane, ids, key ? 2 : 3, 2u);  // only `out` is written
  if (rc != VP8GPU_OK) {
    e->frame_release(out);
    return rc;
  }
  if (!key && sub == 1 && memcmp(enc->tab_mv_probs, enc->dec_state->mv_probs, 38) != 0) {
    // Costs::fill_mv_component_costs( the stream's probabilities ) at the start of a full inter-frame pass
    // (encode_inter.cc:601, reencode.cc:85): only an Encoder built from a Decoder that had seen motion-vector
    // probability updates ever gets here; sampled passes keep whatever the last full pass filled in
    vp8::EncTables* t = new vp8::EncTables();
    vp8::build_enc_tables(*t, &enc->dec_state->mv_probs[0][0]);
    cudaError_t ce = cudaStreamSynchronize(s);  // nothing of this encoder may still be reading the tables
    if (ce == cudaSuccess) ce = cudaMemcpy(enc->dev + enc->off_tab, t, sizeof(vp8::EncTables), cudaMemcpyHostToDevice);
    delete t;
    if (ce != cudaSuccess) {
      e->frame_release(out);
      return e->cuda_fail(ce, "rate tables upload");
    }
    memcpy(enc->tab_mv_probs, enc->dec_state->mv_probs, 38);
  }
  vp8::EncJob* ej = reinterpret_cast<vp8::EncJob*>(enc->h_hdr);
  memset(enc->h_hdr, 0, 512);
  int* d_sync = reinterpret_cast<int*>(enc->dev + enc->off_sync);
  ej->src = e->frame_dev(enc->src);
  ej->ref = key ? nullptr : e->frame_dev(enc->refs[0]);
  ej->out = e->frame_dev(out);
  ej->mbs = reinterpret_cast<vp8gpu_mb*>(enc->dev + enc->off_mbs);
  ej->tokens = reinterpret_cast<vp8gpu_token*>(enc->dev + enc->off_tokens);
  ej->tok_counter = reinterpret_cast<uint32_t*>(d_sync + 96);
  ej->tok_cap = enc->tok_cap;
  ej->progress = d_sync + 128;
  ej->tab = reinterpret_cast<const vp8::EncTables*>(enc->dev + enc->off_tab);
  ej->q = reenc ? *reenc : make_quant(qi);
  if (!reenc) vp8::rd_multipliers(ej->q.y_ac, &enc->rd_rate, &enc->rd_dist);
  ej->rate_mult = enc->rd_rate;
  ej->dist_mult = enc->rd_dist;
  ej->cols = (uint16_t)cols;
  ej->rows = (uint16_t)rows;
  ej->sub = (uint8_t)sub;
  ej->key_frame = key;
  ej->lf_level = 1;  // records carry "filtered"; the level itself is chosen afterwards (choose_loop_filter)
  ej->sad_per_bit = k_sad_per_bit16[clamp_q(qi)];
  ej->realtime = enc->quality == VP8GPU_QUALITY_REALTIME;
  if (!key && sub == 1) {  // encode_raster<InterFrame> / reencode_as_interframe fill the tables before they use them
    enc->mv_costs_filled = true;
    if (!reenc) enc->mv_sad_filled = true;
  }
  ej->mv_costs_zero = !key && !enc->mv_costs_filled;
  ej->mv_sad_zero = !key && !enc->mv_sad_filled;
  if (trellis) {
    ej->trellis = reinterpret_cast<const vp8::TrellisTables*>(enc->d_trellis);
    ej->y2_prev = enc->d_trellis + align_up(sizeof(vp8::TrellisTables), 256);
  }
  auto fail = [&](int code) {
    e->frame_release(out);
    return code;
  };
#define CUF(call)                                                        \
  do {                                                                   \
    cudaError_t e__ = (call);                                            \
    if (e__ != cudaSuccess) return fail(e->cuda_fail(e__, #call));       \
  } while (0)
  CUF(cudaMemcpyAsync(enc->dev + enc->off_encjob, enc->h_hdr, 512, cudaMemcpyHostToDevice, s));
  CUF(cudaMemsetAsync(d_sync, 0, sizeof(int) * (128 + 2 * (size_t)g.mb_rows), s));
  const vp8::EncJob* d_ej = reinterpret_cast<const vp8::EncJob*>(enc->dev + enc->off_encjob);
  if (int ce = trellis ? vp8::launch_enc_rd_trellis(d_ej, rows, g, d_sync + 0, s) : vp8::launch_enc_rd(d_ej, 1, rows, g, d_sync + 0, s))
    return fail(e->cuda_fail((cudaError_t)ce, "k_enc_rd"));
  e->count_launches(1);
  e->mark_frames(enc->lane, ids, key ? 2 : 3, 2u);
  // results back: token count first, then the records
  CUF(cudaMemcpyAsync(enc->h_count, ej->tok_counter, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CUF(cudaMemcpyAsync(enc->h_mbs, ej->mbs, n_mbs * sizeof(vp8gpu_mb), cudaMemcpyDeviceToHost, s));
  enc->pending_out = out;
  return VP8GPU_OK;
#undef CUF
}

// collect half: wait for the pass, fetch the tokens.  *out_frame = the reconstruction BEFORE the loop
// filter (the caller releases it or keeps it as LAST).
int encode_collect(vp8gpu_encoder* enc, int* out_frame) {
  Engine* e = enc->e;
  cudaStream_t s = e->stream(enc->lane);
  const int out = enc->pending_out;
  enc->pending_out = -1;
  if (out < 0) return e->fail(VP8GPU_ERR_LOGIC, "encode_collect without a launched pass");
  auto fail = [&](int code) {
    e->frame_release(out);
    return code;
  };
  cudaError_t ce = cudaStreamSynchronize(s);
  if (ce != cudaSuccess) return fail(e->cuda_fail(ce, "encoder pass"));
  const uint32_t n_tok = *enc->h_count;
  if (n_tok > enc->tok_cap) return fail(e->fail(VP8GPU_ERR_NOMEM, "encoder token pool overflow"));
  if (n_tok) {
    ce = cudaMemcpyAsync(enc->h_tokens, enc->dev + enc->off_tokens, (size_t)n_tok * sizeof(vp8gpu_token), cudaMemcpyDeviceToHost, s);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
    if (ce != cudaSuccess) return fail(e->cuda_fail(ce, "encoder token download"));
  }
  *out_frame = out;
  return VP8GPU_OK;
}

// One encoding pass at quantiser index qi over the whole frame (sub = 1) or the 1/16 sample (sub = 4):
// decisions, transforms, reconstruction on the device; records and tokens back on the host.
int encode_core(vp8gpu_encoder* enc, bool key, int qi, int sub, int* out_frame, const vp8gpu_quant* reenc = nullptr, bool trellis = false) {
  const int rc = encode_launch(enc, key, qi, sub, reenc, trellis);
  return rc == VP8GPU_OK ? encode_collect(enc, out_frame) : rc;
}

// The compressed frame of the last encode_core pass.  final: the frame that is emitted -- token
// probabilities optimised and saved (refresh_entropy_probs, encode_intra.cc:402, encode_inter.cc:587) in
// `probs`; otherwise a size estimate priced with the current tables, which are left alone
// (size_estimation.cc:92,167: no optimize_probability_tables).
// A loop-filter level that is still being searched for while the frame is written (EncodeFeatures::late_loop_filter_level)
struct LateLevel {
  std::mutex m;
  std::condition_variable cv;
  bool ready = false;
  int level = 0;
  double waited_ms = 0;  // how long the writer stood still for the level (timeline)
  void set(int v) {
    {
      std::lock_guard<std::mutex> lk(m);
      level = v;
      ready = true;
    }
    cv.notify_all();
  }
  static int wait(void* p) {
    LateLevel* l = static_cast<LateLevel*>(p);
    const double t0 = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
    std::unique_lock<std::mutex> lk(l->m);
    l->cv.wait(lk, [l] { return l->ready; });
    l->waited_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count() - t0;
    return l->level;
  }
};

int encode_bytes(vp8gpu_encoder* enc, bool key, int qi, int lf_level, int sub, bool final, uint8_t* probs, std::vector<uint8_t>& bytes,
                 LateLevel* late = nullptr) {
  Engine* e = enc->e;
  int pw, ph, cols, rows;
  pass_dims(enc, sub, &pw, &ph, &cols, &rows);
  vp8::EncodeHeader h;
  h.key_frame = key;
  h.show_frame = true;
  h.width = pw;
  h.height = ph;
  h.y_ac_qi = qi;
  h.loop_filter_level = lf_level;
  h.sharpness = 0;
  h.optimize_token_probs = final;
  vp8::EncodeFeatures ft;
  if (enc->writer == 0) {
    ft.ref_writer = final ? (key ? &enc->ref_key : &enc->ref_inter) : (key ? &enc->ref_sub_key : &enc->ref_sub_inter);
    ft.ref_estimate = !final;
    ft.log2_partitions = 0;
  } else {
    // Eight DCT partitions for the emitted frame (row r -> partition r % 8, frame.cc:131-136): the writer records
    // and codes them on eight host threads, which is most of the host time of a pass (the reference writes one
    // partition; seven more cost 21 bytes of partition sizes).  Estimates are small: one partition.
    ft.log2_partitions = (final && rows >= 16) ? 3 : 0;
    if (const char* v = getenv("VP8GPU_ENC_LOG2_PARTS")) ft.log2_partitions = atoi(v) & 3;  // tuning knob
  }
  ft.refresh_entropy_probs = true;
  uint8_t scratch_probs[1056];
  if (final) {
    ft.saved_coef_probs = probs;
  } else {
    // estimate_size<KeyFrame> starts from a fresh DecoderState (default tables), <InterFrame> from the current one
    memcpy(scratch_probs, key ? k_coef_default_probs : probs, 1056);
    ft.saved_coef_probs = scratch_probs;
  }
  if (!key) {
    // macroblock headers of an inter frame are coded with the stream's saved mode / vector probabilities
    // (Frame::serialize( probability_tables ), encoder.cc:169): the defaults unless this Encoder was built from a
    // Decoder that had seen updates (a key frame resets them; estimate_size<KeyFrame> starts from a fresh state)
    ft.ymode_probs = enc->dec_state->ymode_probs;
    ft.uvmode_probs = enc->dec_state->uvmode_probs;
    ft.mv_probs = enc->dec_state->mv_probs;
  }
  if (late) {
    ft.late_loop_filter_level = &LateLevel::wait;
    ft.late_ctx = late;
  }
  bytes = vp8::serialize_frame(h, enc->h_mbs, enc->h_tokens, nullptr, &ft);
  if (bytes.empty()) return e->fail(VP8GPU_ERR_LOGIC, "serializer rejected the device records");
  return VP8GPU_OK;
}

// one loop-filter pass over `frame` with every macroblock at `level` (in place)
int filter_frame(vp8gpu_encoder* enc, int frame, bool key, int level) {
  Engine* e = enc->e;
  const vp8::Geom& g = e->geom();
  cudaStream_t s = e->stream(enc->lane);
  if (level <= 0) return VP8GPU_OK;  // a frame-level 0 disables the filter (frame.cc:144)
  vp8::DevJob* dj = reinterpret_cast<vp8::DevJob*>(enc->h_hdr + 512);
  memset(dj, 0, 512);
  int* d_sync = reinterpret_cast<int*>(enc->dev + enc->off_sync);
  dj->mbs = reinterpret_cast<const vp8gpu_mb*>(enc->dev + enc->off_mbs);
  dj->tokens = reinterpret_cast<const vp8gpu_token*>(enc->dev + enc->off_tokens);
  dj->out = e->frame_dev(frame);
  dj->lf_progress = d_sync + 128 + g.mb_rows;
  dj->intra_progress = d_sync + 128;
  dj->key_frame = key;
  dj->sharpness = (uint8_t)enc->lf_sharpness;
  dj->lf_enabled = 1;
  dj->lf_force = (uint8_t)level;
  int ids[1] = {frame};
  int rc = e->acquire_frames(enc->lane, ids, 1);
  if (rc != VP8GPU_OK) return rc;
  CUE(cudaMemcpyAsync(enc->dev + enc->off_encjob + 512, dj, 512, cudaMemcpyHostToDevice, s));
  CUE(cudaMemsetAsync(d_sync + 32, 0, sizeof(int), s));                                     // ticket
  CUE(cudaMemsetAsync(d_sync + 128 + g.mb_rows, 0, sizeof(int) * (size_t)g.mb_rows, s));    // row progress
  const vp8::DevJob* d_dj = reinterpret_cast<const vp8::DevJob*>(enc->dev + enc->off_encjob + 512);
  if (int ce = vp8::launch_loopfilter(d_dj, 1, g, d_sync + 32, e->next_epoch(2), s)) return e->cuda_fail((cudaError_t)ce, "k_loopfilter");
  e->count_launches(1);
  e->mark_frames(enc->lane, ids, 1);
  // the pinned descriptor is rewritten by the next call: wait until it has been read
  CUE(cudaStreamSynchronize(s));
  return VP8GPU_OK;
}

// n loop-filter passes in ONE launch: frames[i] filtered in place with every macroblock at levels[i] (> 0).  The
// trials of the loop-filter search are independent of each other and k_loopfilter takes a job array (ticket t ->
// row t / n of job t % n), so n trials last about as long as one.
int filter_batch(vp8gpu_encoder* enc, const int* frames, const int* levels, int n, bool key) {
  Engine* e = enc->e;
  const vp8::Geom& g = e->geom();
  cudaStream_t s = e->stream(enc->lane);
  if (n <= 0) return VP8GPU_OK;
  if (n > kLfMax) return e->fail(VP8GPU_ERR_LOGIC, "filter_batch: too many trials");
  vp8::DevJob* dj = reinterpret_cast<vp8::DevJob*>(enc->h_hdr + 512);
  memset(dj, 0, sizeof(vp8::DevJob) * n);
  int* d_sync = reinterpret_cast<int*>(enc->dev + enc->off_sync);
  for (int i = 0; i < n; i++) {
    dj[i].mbs = reinterpret_cast<const vp8gpu_mb*>(enc->dev + enc->off_mbs);
    dj[i].tokens = reinterpret_cast<const vp8gpu_token*>(enc->dev + enc->off_tokens);
    dj[i].out = e->frame_dev(frames[i]);
    dj[i].lf_progress = d_sync + 128 + (size_t)(1 + i) * g.mb_rows;
    dj[i].intra_progress = d_sync + 128;
    dj[i].key_frame = key;
    dj[i].sharpness = (uint8_t)enc->lf_sharpness;
    dj[i].lf_enabled = 1;
    dj[i].lf_force = (uint8_t)levels[i];
  }
  int rc = e->acquire_frames(enc->lane, frames, n);
  if (rc != VP8GPU_OK) return rc;
  CUE(cudaMemcpyAsync(enc->dev + enc->off_encjob + 512, dj, sizeof(vp8::DevJob) * n, cudaMemcpyHostToDevice, s));
  CUE(cudaMemsetAsync(d_sync + 32, 0, sizeof(int), s));                                         // ticket
  CUE(cudaMemsetAsync(d_sync + 128 + g.mb_rows, 0, sizeof(int) * (size_t)n * g.mb_rows, s));    // row progress
  const vp8::DevJob* d_dj = reinterpret_cast<const vp8::DevJob*>(enc->dev + enc->off_encjob + 512);
  if (int ce = vp8::launch_loopfilter(d_dj, n, g, d_sync + 32, e->next_epoch(2), s)) return e->cuda_fail((cudaError_t)ce, "k_loopfilter");
  e->count_launches(1);
  e->mark_frames(enc->lane, frames, n);
  // the pinned descriptors are rewritten by the next call: wait until they have been read
  CUE(cudaStreamSynchronize(s));
  return VP8GPU_OK;
}

// VP8GPU_ENC_SPECULATE=0: the searches of the encoder run candidate by candidate (one launch each), as in round 1;
// the results are the same either way (tests/test_gpu_encoder.py runs both)
bool enc_speculate() {
  static const bool on = [] {
    const char* v = getenv("VP8GPU_ENC_SPECULATE");
    return !(v && v[0] == '0');
  }();
  return on;
}

// Encoder::apply_best_loopfilter_settings (encoder.cc:460-508): try loop-filter levels in ascending
// order -- all of 0..63 for the first frame, the previous level +-1 afterwards -- on a copy of the
// reconstruction, keep going while the luma SSIM against the source improves, then filter the
// reconstruction itself at the best level.  *recon may be replaced by another raster holding that result.
//
// The trials are independent, so up to kLfMax of them run in one k_loopfilter launch on copies; the walk over
// their SSIMs is the reference's (ascending, stop at the first level that does not improve), and the copy
// that was filtered at the best level IS the filtered reconstruction: it takes the place of *recon instead of a
// further pass.  Steady state: one launch instead of three or four dependent ones.
int choose_loop_filter(vp8gpu_encoder* enc, int* recon, bool key, int* level_out, double* ssim_out) {
  Engine* e = enc->e;
  int lo = 0, hi = 63;
  if (enc->last_lf >= 0) {
    lo = enc->last_lf > 0 ? enc->last_lf - 1 : 0;
    hi = enc->last_lf + 1 > 63 ? 63 : enc->last_lf + 1;
  }
  int temps[kLfMax], n_temps = 0;
  const int want = enc_speculate() ? (hi - lo + 1 < kLfMax ? hi - lo + 1 : kLfMax) : 1;
  for (; n_temps < want; n_temps++)
    if (e->frame_alloc(&temps[n_temps]) != VP8GPU_OK) break;  // a small pool: fewer trials per launch
  if (n_temps == 0) return e->fail(VP8GPU_ERR_NOMEM, "loop-filter search: no raster for a trial");
  int best = 0, keep = -1;  // keep: the trial raster that holds the reconstruction filtered at `best`
  double best_ssim = -1.0;
  int rc = VP8GPU_OK;
  bool stop = false, found = false;
  for (int level = lo; level <= hi && !stop && rc == VP8GPU_OK;) {
    int use[kLfMax], lv[kLfMax], n = 0, nf = 0, fr[kLfMax], fl[kLfMax];
    for (int i = 0; i < n_temps && level + n <= hi; i++) {
      if (temps[i] == keep && n_temps > 1) continue;  // holds the best result so far (a single trial raster is reused)
      use[n] = temps[i];
      lv[n] = level + n;
      n++;
    }
    if (n_temps == 1) keep = -1;
    for (int i = 0; i < n && rc == VP8GPU_OK; i++) {
      rc = e->frame_copy(use[i], *recon, enc->lane);
      if (lv[i] > 0) fr[nf] = use[i], fl[nf] = lv[i], nf++;  // a frame-level 0 disables the filter (frame.cc:144)
    }
    if (rc == VP8GPU_OK) rc = filter_batch(enc, fr, fl, nf, key);
    for (int i = 0; i < n && rc == VP8GPU_OK; i++) {
      double q = 0;
      rc = e->frames_ssim(use[i], enc->src, enc->lane, &q);
      if (rc != VP8GPU_OK) break;
      if (q > best_ssim) {
        best_ssim = q;
        best = lv[i];
        keep = use[i];
        found = true;
      } else {
        stop = true;
        break;
      }
    }
    level += n;
  }
  // a single trial raster is overwritten by the trial that ends the search: filter the reconstruction itself then
  if (rc == VP8GPU_OK && keep < 0 && found) rc = filter_frame(enc, *recon, key, best);
  for (int i = 0; i < n_temps; i++)
    if (temps[i] != keep || rc != VP8GPU_OK) e->frame_release(temps[i]);
  if (rc != VP8GPU_OK) return rc;
  if (keep >= 0) {
    e->frame_release(*recon);
    *recon = keep;
  }
  *level_out = best;
  *ssim_out = best_ssim;
  return VP8GPU_OK;
}

// source planes (display size) -> MB-aligned raster on the device, edges replicated like the
// reference's input reader (input/yuv4mpeg.cc:231-271)
int upload_source(vp8gpu_encoder* enc, const uint8_t* y, size_t ys, const uint8_t* u, const uint8_t* v, size_t cs) {
  Engine* e = enc->e;
  const vp8::Geom& g = e->geom();
  const int w = e->width(), h = e->height(), cw = (w + 1) / 2, ch = (h + 1) / 2;
  uint8_t* py = enc->h_src;
  uint8_t* pu = py + (size_t)g.W * g.H;
  uint8_t* pv = pu + (size_t)(g.W / 2) * (g.H / 2);
  // the copy into pinned memory is on every call's critical path: the luma rows in four slices on the host pool
  auto luma_rows = [&](int r0, int r1) {
    for (int r = r0; r < r1; r++) {
      const uint8_t* srow = y + (size_t)(r < h ? r : h - 1) * ys;
      uint8_t* drow = py + (size_t)r * g.W;
      memcpy(drow, srow, w);
      if (g.W > w) memset(drow + w, srow[w - 1], g.W - w);
    }
  };
  auto chroma_rows = [&]() {
    for (int pl = 0; pl < 2; pl++) {
      const uint8_t* sp = pl ? v : u;
      uint8_t* dp = pl ? pv : pu;
      for (int r = 0; r < g.H / 2; r++) {
        const uint8_t* srow = sp + (size_t)(r < ch ? r : ch - 1) * cs;
        uint8_t* drow = dp + (size_t)r * (g.W / 2);
        memcpy(drow, srow, cw);
        if (g.W / 2 > cw) memset(drow + cw, srow[cw - 1], g.W / 2 - cw);
      }
    }
  };
  if ((size_t)g.W * g.H >= (size_t)640 * 480) {
    vp8::HostPool::Group grp;
    const int q = g.H / 4;
    for (int k = 1; k < 4; k++) grp.run([&luma_rows, k, q, &g] { luma_rows(k * q, k == 3 ? g.H : (k + 1) * q); });
    grp.run(chroma_rows);
    luma_rows(0, q);
    grp.wait();
  } else {
    luma_rows(0, g.H);
    chroma_rows();
  }
  return e->frame_upload(enc->src, py, g.W, pu, pv, g.W / 2);
}

}  // namespace

// layout of the size-estimate scratch (estimate_batch_launch); returns its size
static size_t est_layout(vp8gpu_encoder* enc) {
  const vp8::Geom& g = enc->e->geom();
  int pw, ph, cols, rows;
  pass_dims(enc, 4, &pw, &ph, &cols, &rows);
  const size_t n_mbs = (size_t)cols * rows;
  enc->est_tok_cap = (uint32_t)(n_mbs * 400);
  size_t off = align_up(sizeof(vp8::EncJob) * kEstMax, 256);
  enc->est_off_sync = off;
  off = align_up(off + sizeof(int) * (128 + (size_t)kEstMax * rows), 256);
  enc->est_off_mbs = off;
  off = align_up(off + (size_t)kEstMax * n_mbs * sizeof(vp8gpu_mb), 256);
  enc->est_off_tokens = off;
  off = align_up(off + (size_t)kEstMax * enc->est_tok_cap * sizeof(vp8gpu_token), 256);
  enc->est_off_out = off;
  enc->est_out_stride = align_up(g.frame_bytes, 256);
  return off + (size_t)kEstMax * enc->est_out_stride;
}

// ---- buffer sets of destroyed Encoders, kept per context -----------------------------------------------------
// Salsify copies its Encoder twice per frame and drops the copies again (salsify-sender.cc:492-518); an Encoder
// here owns ~20 MB of pinned host memory and ~20 MB (+ the size-estimate scratch) of device memory at 1080p, and
// cudaHostAlloc / cudaMalloc / cudaFree of those cost milliseconds and serialise on the driver.  A destroyed
// Encoder therefore hands its buffers to its context, the next create / clone of that context takes them over.
struct EncBufferSet {
  uint8_t *dev, *d_split, *d_trellis, *d_est, *h_est, *h_hdr, *h_src;
  vp8gpu_mb* h_mbs;
  vp8gpu_token* h_tokens;
  uint32_t* h_count;
  size_t split_cap;
  uint8_t tab_mv_probs[38];
};
static std::mutex g_enc_pool_mu;
static std::vector<std::pair<Engine*, EncBufferSet>> g_enc_pool;
constexpr size_t kEncPoolPerEngine = 4;

static void enc_buffers_free(const EncBufferSet& b) {
  if (b.dev) cudaFree(b.dev);
  if (b.d_split) cudaFree(b.d_split);
  if (b.d_trellis) cudaFree(b.d_trellis);
  if (b.d_est) cudaFree(b.d_est);
  if (b.h_est) cudaFreeHost(b.h_est);
  if (b.h_hdr) cudaFreeHost(b.h_hdr);
  if (b.h_mbs) cudaFreeHost(b.h_mbs);
  if (b.h_tokens) cudaFreeHost(b.h_tokens);
  if (b.h_src) cudaFreeHost(b.h_src);
  if (b.h_count) cudaFreeHost(b.h_count);
}
// capi.cc vp8gpu_ctx_destroy: the context's buffer sets die with it
extern "C" void vp8gpu_encoder_pool_purge(Engine* e) {
  std::vector<EncBufferSet> dead;
  {
    std::lock_guard<std::mutex> lk(g_enc_pool_mu);
    for (size_t i = 0; i < g_enc_pool.size();) {
      if (g_enc_pool[i].first == e) {
        dead.push_back(g_enc_pool[i].second);
        g_enc_pool.erase(g_enc_pool.begin() + i);
      } else {
        i++;
      }
    }
  }
  for (const EncBufferSet& b : dead) enc_buffers_free(b);
}

// common part of create / clone / create_from: buffers on device and host, the rate tables
static int encoder_alloc(vp8gpu_ctx* ctx, vp8gpu_encoder** out) {
  vp8gpu_encoder* enc = new vp8gpu_encoder();
  enc->ctx = ctx;
  enc->e = vp8gpu_ctx_engine(ctx);
  enc->lane = vp8gpu_ctx_next_lane(ctx);
  Engine* e = enc->e;
  const vp8::Geom& g = e->geom();
  const size_t n_mbs = (size_t)g.mb_cols * g.mb_rows;
  enc->tok_cap = (uint32_t)(n_mbs * 400);
  size_t off = 0;
  enc->off_encjob = off;
  off = align_up(off + kHdrBytes, 256);
  enc->off_sync = off;
  off = align_up(off + sizeof(int) * (128 + (1 + (size_t)kLfMax) * g.mb_rows), 256);
  enc->off_mbs = off;
  off = align_up(off + n_mbs * sizeof(vp8gpu_mb), 256);
  enc->off_tab = off;
  off = align_up(off + sizeof(vp8::EncTables), 256);
  enc->off_tokens = off;
  off = align_up(off + (size_t)enc->tok_cap * sizeof(vp8gpu_token), 256);
  enc->dev_bytes = off;
  cudaSetDevice(e->device());
  bool pooled = false;
  {
    std::lock_guard<std::mutex> lk(g_enc_pool_mu);
    for (size_t i = g_enc_pool.size(); i-- > 0;)
      if (g_enc_pool[i].first == e) {
        const EncBufferSet b = g_enc_pool[i].second;
        g_enc_pool.erase(g_enc_pool.begin() + i);
        enc->dev = b.dev, enc->d_split = b.d_split, enc->d_trellis = b.d_trellis, enc->d_est = b.d_est, enc->h_est = b.h_est;
        enc->h_hdr = b.h_hdr, enc->h_src = b.h_src, enc->h_mbs = b.h_mbs, enc->h_tokens = b.h_tokens, enc->h_count = b.h_count;
        enc->split_cap = b.split_cap;
        memcpy(enc->tab_mv_probs, b.tab_mv_probs, 38);
        pooled = true;
        break;
      }
  }
  if (pooled) {
    // same context = same geometry = same layout; what depends on the Encoder's history is only the rate tables
    if (enc->d_est) est_layout(enc);
    if (e->frame_alloc(&enc->src) != VP8GPU_OK) {
      vp8gpu_encoder_destroy(enc);
      return e->fail(VP8GPU_ERR_NOMEM, "encoder allocation failed");
    }
  } else if (cudaMalloc(&enc->dev, enc->dev_bytes) != cudaSuccess || cudaHostAlloc(&enc->h_hdr, kHdrBytes, cudaHostAllocDefault) != cudaSuccess ||
      cudaHostAlloc(&enc->h_mbs, n_mbs * sizeof(vp8gpu_mb), cudaHostAllocDefault) != cudaSuccess ||
      cudaHostAlloc(&enc->h_tokens, (size_t)enc->tok_cap * sizeof(vp8gpu_token), cudaHostAllocDefault) != cudaSuccess ||
      cudaHostAlloc(&enc->h_src, (size_t)g.W * g.H * 3 / 2, cudaHostAllocDefault) != cudaSuccess ||
      cudaHostAlloc(&enc->h_count, 64, cudaHostAllocDefault) != cudaSuccess || e->frame_alloc(&enc->src) != VP8GPU_OK) {
    vp8gpu_encoder_destroy(enc);
    return e->fail(VP8GPU_ERR_NOMEM, "encoder allocation failed");
  }
  static const vp8::EncTables* tables = [] {
    vp8::EncTables* t = new vp8::EncTables();
    vp8::build_enc_tables(*t);
    return t;
  }();
  if ((!pooled || memcmp(enc->tab_mv_probs, k_mv_default_probs, 38) != 0) &&
      cudaMemcpy(enc->dev + enc->off_tab, tables, sizeof(vp8::EncTables), cudaMemcpyHostToDevice) != cudaSuccess) {
    vp8gpu_encoder_destroy(enc);
    return e->fail(VP8GPU_ERR_CUDA, "encoder rate tables upload failed");
  }
  memcpy(enc->tab_mv_probs, k_mv_default_probs, 38);
  enc->dec_state = new vp8::State(e->width(), e->height());
  enc->scratch = new vp8::ParsedFrame();
  *out = enc;
  return VP8GPU_OK;
}

extern "C" {

int vp8gpu_encoder_create(vp8gpu_ctx* ctx, vp8gpu_encoder** out) {
  if (!ctx || !out) return VP8GPU_ERR_LOGIC;
  return encoder_alloc(ctx, out);
}

// Encoder( const Encoder & ) (encoder.cc:92-102): an independent copy that shares the reference rasters
// (immutable, reference counted); the two can then encode concurrently (salsify-sender.cc:492-518).
int vp8gpu_encoder_clone(const vp8gpu_encoder* src, vp8gpu_encoder** out) {
  if (!src || !out) return VP8GPU_ERR_LOGIC;
  vp8gpu_encoder* enc = nullptr;
  int rc = encoder_alloc(src->ctx, &enc);
  if (rc != VP8GPU_OK) return rc;
  enc->has_state = src->has_state;
  enc->two_pass = src->two_pass;
  enc->quality = src->quality;  // encode_quality_( encoder.encode_quality_ ), encoder.cc:98
  enc->quality_fixed = src->quality_fixed;
  enc->writer = src->writer;  // (the copy's frame objects, i.e. the writer's header state, start fresh: encoder.cc:92-102)
  enc->last_qi = src->last_qi;
  enc->last_lf = src->last_lf;
  enc->stat_qi = src->stat_qi;
  enc->stat_lf = src->stat_lf;
  enc->mv_costs_filled = src->mv_costs_filled;  // costs_( encoder.costs_ ), encoder.cc:96
  enc->mv_sad_filled = src->mv_sad_filled;
  enc->last_ssim = src->last_ssim;
  *enc->dec_state = *src->dec_state;
  for (int k = 0; k < 3; k++) {
    enc->refs[k] = src->refs[k];
    if (enc->refs[k] >= 0) enc->e->frame_retain(enc->refs[k]);
  }
  *out = enc;
  return VP8GPU_OK;
}

// Encoder( const Decoder &, two_pass, quality ) (encoder.hh:350-351): continue a stream from a decoder's
// state and references (the next frame is an inter frame predicted from the decoder's LAST)
int vp8gpu_encoder_create_from_decoder(vp8gpu_ctx* ctx, vp8gpu_decoder* dec, vp8gpu_encoder** out) {
  if (!ctx || !dec || !out) return VP8GPU_ERR_LOGIC;
  vp8gpu_frame_id refs[3];
  const vp8gpu_state* st = vp8gpu_decoder_state(dec);
  int rc = vp8gpu_decoder_references(dec, refs);
  if (rc != VP8GPU_OK || !st) return VP8GPU_ERR_LOGIC;
  vp8gpu_encoder* enc = nullptr;
  rc = encoder_alloc(ctx, &enc);
  if (rc != VP8GPU_OK) return rc;
  uint8_t blob[16384];
  const size_t n = vp8gpu_state_serialize(st, blob, sizeof(blob));
  std::vector<uint8_t> big;
  const uint8_t* bp = blob;
  if (n > sizeof(blob)) {  // a segmentation map makes the blob larger
    big.resize(n);
    vp8gpu_state_serialize(st, big.data(), big.size());
    bp = big.data();
  }
  if (!vp8::State::deserialize(bp, n, *enc->dec_state)) {
    vp8gpu_encoder_destroy(enc);
    return vp8gpu_ctx_engine(ctx)->fail(VP8GPU_ERR_LOGIC, "encoder_create_from_decoder: bad decoder state");
  }
  for (int k = 0; k < 3; k++) {
    enc->refs[k] = refs[k];
    if (refs[k] >= 0) enc->e->frame_retain(refs[k]);
  }
  enc->has_state = true;
  *out = enc;
  return VP8GPU_OK;
}

void vp8gpu_encoder_destroy(vp8gpu_encoder* enc) {
  if (!enc) return;
  cudaSetDevice(enc->e->device());
  if (enc->e->stream(enc->lane)) cudaStreamSynchronize(enc->e->stream(enc->lane));
  for (int k = 0; k < 3; k++)
    if (enc->refs[k] >= 0) enc->e->frame_release(enc->refs[k]);
  if (enc->src >= 0) enc->e->frame_release(enc->src);
  EncBufferSet b;
  b.dev = enc->dev, b.d_split = enc->d_split, b.d_trellis = enc->d_trellis, b.d_est = enc->d_est, b.h_est = enc->h_est;
  b.h_hdr = enc->h_hdr, b.h_src = enc->h_src, b.h_mbs = enc->h_mbs, b.h_tokens = enc->h_tokens, b.h_count = enc->h_count;
  b.split_cap = enc->split_cap;
  memcpy(b.tab_mv_probs, enc->tab_mv_probs, 38);
  bool kept = false;
  if (b.dev && b.h_hdr && b.h_mbs && b.h_tokens && b.h_src && b.h_count) {  // a complete set (not a failed allocation)
    std::lock_guard<std::mutex> lk(g_enc_pool_mu);
    size_t have = 0;
    for (const auto& x : g_enc_pool) have += x.first == enc->e;
    if (have < kEncPoolPerEngine) {
      g_enc_pool.emplace_back(enc->e, b);
      kept = true;
    }
  }
  if (!kept) enc_buffers_free(b);
  delete enc->dec_state;
  delete enc->scratch;
  delete enc;
}

static int apply_emitted_frame(vp8gpu_encoder* enc, const uint8_t* data, size_t len, const vp8gpu_mb* mbs = nullptr,
                               const vp8gpu_token* tokens = nullptr, uint32_t n_tok = 0);
// The tail of Encoder::write_frame (encoder.cc:164-167): at REALTIME_QUALITY the frame's loop-filter level and quantiser
// narrow the next frame's searches; at BEST_QUALITY every search starts from scratch.  vp8gpu_encoder_stats reports
// them either way.
static void remember_frame(vp8gpu_encoder* enc, int qi, int lf) {
  enc->stat_qi = qi;
  enc->stat_lf = lf;
  enc->quality_fixed = true;
  if (enc->quality == VP8GPU_QUALITY_REALTIME) {
    enc->last_qi = qi;
    enc->last_lf = lf;
  }
}
static int finish_frame(vp8gpu_encoder* enc, bool key, const std::vector<uint8_t>& bytes, int out_frame, int qi, int lf, double ssim,
                        uint8_t* out, size_t cap, size_t* size) {
  Engine* e = enc->e;
  *size = bytes.size();
  if (!out || cap < bytes.size()) {
    e->frame_release(out_frame);
    return e->fail(VP8GPU_ERR_NOMEM, "output buffer too small");
  }
  memcpy(out, bytes.data(), bytes.size());
  if (!key && enc->dec_state->seg_enabled) {
    // An Encoder built from a Decoder whose stream uses segmentation: the frame carries no segmentation update, so
    // a receiver keeps dequantising and filtering by segment while k_enc_rd reconstructed with the frame's one
    // quantiser.  The reference is immune because write_frame always decodes what it wrote (encoder.cc:153-158);
    // do the same here instead of keeping the kernel's reconstruction.
    e->frame_release(out_frame);
    const int rc = apply_emitted_frame(enc, bytes.data(), bytes.size(), enc->h_mbs, enc->h_tokens, *enc->h_count);
    if (rc != VP8GPU_OK) return rc;
    remember_frame(enc, qi, lf);
    enc->last_ssim = ssim;
    return VP8GPU_OK;
  }
  // Encoder::write_frame -> update_decoder_state (encoder.cc:146-151): the state a decoder is in after this
  // frame, obtained the way a decoder obtains it -- by parsing the frame (first partition only)
  const int prc = vp8::parse_frame(*enc->dec_state, bytes.data(), bytes.size(), *enc->scratch, true);
  if (prc != VP8GPU_OK) {
    e->frame_release(out_frame);
    return e->fail(VP8GPU_ERR_LOGIC, "the emitted frame does not parse");
  }
  // Frame::copy_to (frame.cc:272-307): a key frame replaces all three references, an inter frame of this
  // encoder (refresh_last only) replaces LAST
  for (int k = 0; k < (key ? 3 : 1); k++) {
    if (enc->refs[k] >= 0) e->frame_release(enc->refs[k]);
    enc->refs[k] = out_frame;
    if (k) e->frame_retain(out_frame);
  }
  enc->has_state = true;
  remember_frame(enc, qi, lf);
  enc->last_ssim = ssim;
  enc->stat_frames++;
  return VP8GPU_OK;
}

// The macroblock loop of encode_raster (encode_intra.cc:409-443): once, or -- key frame of a two-pass Encoder -- twice,
// the second time with trellis quantisation.  Between the passes the reference keeps two things of the first one:
// the token probability updates it derived from it (optimize_probability_tables runs after EACH pass on the same
// frame header: the second pass adds to them) and every block's has_nonzero, of which the second pass reads only
// those it does not recompute: the Y2 blocks of its B_PRED macroblocks.
static int encode_passes(vp8gpu_encoder* enc, bool key, int qi, int* frame) {
  if (!(key && enc->two_pass)) return encode_core(enc, key, qi, 1, frame);
  Engine* e = enc->e;
  const vp8::Geom& g = e->geom();
  const size_t n_mbs = (size_t)g.mb_cols * g.mb_rows, y2_off = align_up(sizeof(vp8::TrellisTables), 256);
  if (!enc->d_trellis) {
    if (cudaMalloc(&enc->d_trellis, y2_off + align_up(n_mbs, 256)) != cudaSuccess) return e->fail(VP8GPU_ERR_NOMEM, "trellis tables");
    vp8::TrellisTables* t = new vp8::TrellisTables();
    vp8::build_trellis_tables(*t);
    const cudaError_t ce = cudaMemcpy(enc->d_trellis, t, sizeof(*t), cudaMemcpyHostToDevice);
    delete t;
    if (ce != cudaSuccess) return e->cuda_fail(ce, "trellis tables upload");
  }
  int rc = encode_core(enc, true, qi, 1, frame);
  if (rc != VP8GPU_OK) return rc;
  e->frame_release(*frame);
  *frame = -1;
  if (enc->writer == 0) {  // optimize_probability_tables of the first pass: only its effect on the header state matters
    std::vector<uint8_t> discard;
    uint8_t probs[1056];
    memcpy(probs, enc->dec_state->coef_probs, 1056);
    rc = encode_bytes(enc, true, qi, 0, 1, true, probs, discard);
    if (rc != VP8GPU_OK) return rc;
  }
  std::vector<uint8_t> y2(n_mbs, 0);
  for (size_t i = 0; i < n_mbs; i++) {
    const vp8gpu_mb& m = enc->h_mbs[i];
    if (m.y_mode == VP8GPU_B_PRED) {  // Y2 untouched (a fresh key_frame_ object: false); Y blocks left as "Y without Y2"
      y2[i] = 2;
      continue;
    }
    for (unsigned t = 0; t < m.tok_cnt; t++) {
      const uint32_t tk = enc->h_tokens[m.tok_off + t];
      if (((tk >> 20) & 31) == 24 && (tk & 0xFFFF)) y2[i] = 1;
    }
  }
  if (cudaMemcpy(enc->d_trellis + y2_off, y2.data(), n_mbs, cudaMemcpyHostToDevice) != cudaSuccess)
    return e->fail(VP8GPU_ERR_CUDA, "two-pass: Y2 flags upload");
  rc = encode_core(enc, true, qi, 1, frame, nullptr, true);
  if (rc != VP8GPU_OK) return rc;
  for (size_t i = 0; i < n_mbs; i++) enc->h_mbs[i].reserved = 0;  // the kernel's has_nonzero masks are not part of a record
  return VP8GPU_OK;
}

// encode at qi, choose the loop filter, serialize: Encoder::encode_raster + write_frame (encoder.cc:140-178)
static int encode_final(vp8gpu_encoder* enc, bool key, int qi, uint8_t* out, size_t cap, size_t* size) {
  int frame = -1, lf = 0;
  double ssim = -1.0;
  int rc;
  {
    Phase ph(&enc->tl[3]);
    rc = encode_passes(enc, key, qi, &frame);
  }
  if (rc != VP8GPU_OK) return rc;
  std::vector<uint8_t> bytes;
  uint8_t probs[1056];
  memcpy(probs, enc->dec_state->coef_probs, 1056);
  if (enc_speculate()) {
    // The writer needs the loop-filter level only where the frame header spells it out, after the token partitions
    // -- most of its work -- are done: it runs on a pool thread (hostpool.h; host code only: records and tokens of the
    // pass are in pinned memory) while this thread drives the loop-filter search on the device, and picks the level up
    // when it gets there.
    LateLevel late;
    int wrc = VP8GPU_OK;
    vp8::HostPool::Group writer;
    writer.run([&] {
      Phase ph(&enc->tl[5]);
      wrc = encode_bytes(enc, key, qi, 0, 1, true, probs, bytes, &late);
    });
    {
      Phase ph(&enc->tl[4]);
      rc = choose_loop_filter(enc, &frame, key, &lf, &ssim);
    }
    late.set(rc == VP8GPU_OK ? lf : 0);
    writer.wait();
    enc->tl[5] -= late.waited_ms;  // the writer's own work
    if (rc == VP8GPU_OK) rc = wrc;
  } else {
    {
      Phase ph(&enc->tl[4]);
      rc = choose_loop_filter(enc, &frame, key, &lf, &ssim);
    }
    Phase ph(&enc->tl[5]);
    if (rc == VP8GPU_OK) rc = encode_bytes(enc, key, qi, lf, 1, true, probs, bytes);
  }
  if (rc != VP8GPU_OK) {
    enc->e->frame_release(frame);
    return rc;
  }
  Phase ph(&enc->tl[6]);
  return finish_frame(enc, key, bytes, frame, qi, lf, ssim, out, cap, size);
}

// Encoder::estimate_frame_size (size_estimation.cc:36-181): code the 1/16 sample at y_ac_qi, serialize it
// with the current probability tables, multiply by 16
// second half of an estimate: the sampled frame whose records and tokens are in h_mbs / h_tokens, serialised
static int estimate_bytes(vp8gpu_encoder* enc, bool key, int qi, size_t* size) {
  std::vector<uint8_t> bytes;
  const int rc = encode_bytes(enc, key, qi, 0, 4, false, enc->dec_state->coef_probs, bytes);
  if (rc == VP8GPU_OK) *size = bytes.size() * 16;
  if (rc == VP8GPU_OK) {
    if (const char* path = getenv("VP8GPU_EST_DUMP")) {  // diagnostic (tools/enc_estimates.py): the sampled frame itself
      if (FILE* f = fopen(path, "wb")) {
        fwrite(bytes.data(), 1, bytes.size(), f);
        fclose(f);
      }
    }
  }
  return rc;
}
static int estimate_size(vp8gpu_encoder* enc, bool key, int qi, size_t* size) {
  int frame = -1;
  int rc = encode_core(enc, key, qi, 4, &frame);
  if (rc != VP8GPU_OK) return rc;
  enc->e->frame_release(frame);
  return estimate_bytes(enc, key, qi, size);
}

// ---- speculative size estimates -----------------------------------------------------------------------------
// Encoder::encode_with_target_size bisects over y_ac_qi, and every probe is a sampled pass (estimate_size) that
// depends on the source, the references and its quantiser only -- not on the probes before it.  A sampled pass is a
// wavefront of (cols + 2 rows) dependent macroblock steps however many SMs there are, so the probes the search can
// still reach are coded in ONE k_enc_rd launch (n jobs: own records, token pool, counters, reconstruction raster);
// the bisection then reads results.  Five or six dependent launch / wait / download rounds per frame become one.
// What the reference carries from probe to probe -- the header state of its subsampled frame objects, the rd
// multipliers of the last probe -- is carried the same way, because serialisation (estimate_batch_size) still
// happens probe by probe in the order of the search.
static int estimate_batch_launch(vp8gpu_encoder* enc, bool key, const int* qis, int n) {
  Engine* e = enc->e;
  const vp8::Geom& g = e->geom();
  enc->est_n = 0;
  int pw, ph, cols, rows;
  pass_dims(enc, 4, &pw, &ph, &cols, &rows);
  if (cols < 1 || rows < 1) return e->fail(VP8GPU_ERR_UNSUPPORTED, "frame too small for the sampled size estimate");
  if (n < 1 || n > kEstMax) return e->fail(VP8GPU_ERR_LOGIC, "estimate_batch_launch: bad candidate count");
  const size_t n_mbs = (size_t)cols * rows;
  if (!enc->d_est) {
    const size_t off = est_layout(enc);
    if (cudaMalloc(&enc->d_est, off) != cudaSuccess ||
        cudaHostAlloc(&enc->h_est, align_up(sizeof(vp8::EncJob) * kEstMax, 256) + sizeof(uint32_t) * 64, cudaHostAllocDefault) != cudaSuccess) {
      if (enc->d_est) cudaFree(enc->d_est);
      enc->d_est = nullptr;
      return e->fail(VP8GPU_ERR_NOMEM, "size estimates: scratch allocation failed");
    }
  }
  if (int rc = e->ensure_lane(enc->lane)) return rc;
  cudaStream_t s = e->stream(enc->lane);
  int ids[2] = {enc->src, enc->refs[0]};
  int rc = e->acquire_frames(enc->lane, ids, key ? 1 : 2, 0u);  // both only read
  if (rc != VP8GPU_OK) return rc;
  vp8::EncJob* ej = reinterpret_cast<vp8::EncJob*>(enc->h_est);
  memset(ej, 0, sizeof(vp8::EncJob) * n);
  int* d_sync = reinterpret_cast<int*>(enc->d_est + enc->est_off_sync);
  for (int i = 0; i < n; i++) {
    vp8::EncJob& j = ej[i];
    uint32_t rate = enc->rd_rate, dist = enc->rd_dist;
    j.src = e->frame_dev(enc->src);
    j.ref = key ? nullptr : e->frame_dev(enc->refs[0]);
    j.out = enc->d_est + enc->est_off_out + (size_t)i * enc->est_out_stride;
    j.mbs = reinterpret_cast<vp8gpu_mb*>(enc->d_est + enc->est_off_mbs) + (size_t)i * n_mbs;
    j.tokens = reinterpret_cast<vp8gpu_token*>(enc->d_est + enc->est_off_tokens) + (size_t)i * enc->est_tok_cap;
    j.tok_counter = reinterpret_cast<uint32_t*>(d_sync + 32 + i);
    j.tok_cap = enc->est_tok_cap;
    j.progress = d_sync + 128 + (size_t)i * rows;
    j.tab = reinterpret_cast<const vp8::EncTables*>(enc->dev + enc->off_tab);
    j.q = make_quant(qis[i]);
    vp8::rd_multipliers(j.q.y_ac, &rate, &dist);  // update_rd_multipliers( quantizer ) of this probe
    j.rate_mult = rate;
    j.dist_mult = dist;
    j.cols = (uint16_t)cols;
    j.rows = (uint16_t)rows;
    j.sub = 4;
    j.key_frame = key;
    j.lf_level = 1;
    j.sad_per_bit = k_sad_per_bit16[clamp_q(qis[i])];
    j.realtime = enc->quality == VP8GPU_QUALITY_REALTIME;
    j.mv_costs_zero = !key && !enc->mv_costs_filled;
    j.mv_sad_zero = !key && !enc->mv_sad_filled;
    enc->est_qi[i] = qis[i];
    enc->est_rate[i] = rate;
    enc->est_dist[i] = dist;
  }
  uint32_t* h_counts = reinterpret_cast<uint32_t*>(enc->h_est + align_up(sizeof(vp8::EncJob) * kEstMax, 256));
  CUE(cudaMemcpyAsync(enc->d_est, ej, sizeof(vp8::EncJob) * n, cudaMemcpyHostToDevice, s));
  CUE(cudaMemsetAsync(d_sync, 0, sizeof(int) * (128 + (size_t)n * rows), s));
  if (int ce = vp8::launch_enc_rd(reinterpret_cast<const vp8::EncJob*>(enc->d_est), n, rows, g, d_sync + 0, s))
    return e->cuda_fail((cudaError_t)ce, "k_enc_rd (size estimates)");
  e->count_launches(1);
  e->mark_frames(enc->lane, ids, key ? 1 : 2, 0u);
  CUE(cudaMemcpyAsync(h_counts, d_sync + 32, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, s));
  CUE(cudaStreamSynchronize(s));
  enc->est_n = n;
  return VP8GPU_OK;
}

// the estimate of candidate idx of the current batch: its records and tokens to the host, then what estimate_size does
static int estimate_batch_size(vp8gpu_encoder* enc, bool key, int idx, size_t* size) {
  Engine* e = enc->e;
  cudaStream_t s = e->stream(enc->lane);
  int pw, ph, cols, rows;
  pass_dims(enc, 4, &pw, &ph, &cols, &rows);
  const size_t n_mbs = (size_t)cols * rows;
  const uint32_t n_tok = reinterpret_cast<const uint32_t*>(enc->h_est + align_up(sizeof(vp8::EncJob) * kEstMax, 256))[idx];
  if (n_tok > enc->est_tok_cap) return e->fail(VP8GPU_ERR_NOMEM, "encoder token pool overflow");
  CUE(cudaMemcpyAsync(enc->h_mbs, reinterpret_cast<const vp8gpu_mb*>(enc->d_est + enc->est_off_mbs) + (size_t)idx * n_mbs,
                      n_mbs * sizeof(vp8gpu_mb), cudaMemcpyDeviceToHost, s));
  if (n_tok)
    CUE(cudaMemcpyAsync(enc->h_tokens, reinterpret_cast<const vp8gpu_token*>(enc->d_est + enc->est_off_tokens) + (size_t)idx * enc->est_tok_cap,
                        (size_t)n_tok * sizeof(vp8gpu_token), cudaMemcpyDeviceToHost, s));
  CUE(cudaStreamSynchronize(s));
  enc->rd_rate = enc->est_rate[idx];  // what update_rd_multipliers of this probe leaves behind
  enc->rd_dist = enc->est_dist[idx];
  return estimate_bytes(enc, key, enc->est_qi[idx], size);
}

// the candidates to code when the search stands at [lo, hi] and needs a probe that is not on the device: the whole
// range if it fits one launch, else the nodes of the next three levels of the bisection tree
static void bisection_nodes(int lo, int hi, int depth, int* out, int* n) {
  if (lo > hi || depth == 0) return;
  const int mid = (lo + hi) / 2;
  out[(*n)++] = mid;
  bisection_nodes(lo, mid - 1, depth - 1, out, n);
  bisection_nodes(mid + 1, hi, depth - 1, out, n);
}
static int estimate_probe(vp8gpu_encoder* enc, bool key, int lo, int hi, int qi, size_t* size) {
  if (!enc_speculate()) {
    Phase ph(&enc->tl[1]);  // candidate by candidate: launch, wait, download and serialise are one thing
    return estimate_size(enc, key, qi, size);
  }
  int idx = -1;
  for (int i = 0; i < enc->est_n; i++)
    if (enc->est_qi[i] == qi) idx = i;
  if (idx < 0) {
    int qis[kEstMax], n = 0;
    if (hi - lo + 1 <= kEstMax) {
      for (int q = lo; q <= hi; q++) qis[n++] = q;
    } else {
      bisection_nodes(lo, hi, 3, qis, &n);
    }
    int rc;
    {
      Phase ph(&enc->tl[1]);
      rc = estimate_batch_launch(enc, key, qis, n);
    }
    if (rc != VP8GPU_OK) return rc;
    for (int i = 0; i < enc->est_n; i++)
      if (enc->est_qi[i] == qi) idx = i;
    if (idx < 0) return enc->e->fail(VP8GPU_ERR_LOGIC, "size estimates: probe missing from its batch");
  }
  Phase ph(&enc->tl[2]);
  return estimate_batch_size(enc, key, idx, size);
}

int vp8gpu_encoder_encode_with_quantizer(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u,
                                         const uint8_t* v, size_t uv_stride, int y_ac_qi, uint8_t* out, size_t cap,
                                         size_t* size) {
  if (!enc || !y || !u || !v || !size || y_ac_qi < 0 || y_ac_qi > 127) return VP8GPU_ERR_LOGIC;
  cudaSetDevice(enc->e->device());
  memset(enc->tl, 0, sizeof(enc->tl));
  Phase whole(&enc->tl[7]);
  int rc;
  {
    Phase ph(&enc->tl[0]);
    rc = upload_source(enc, y, y_stride, u, v, uv_stride);
  }
  if (rc != VP8GPU_OK) return rc;
  return encode_final(enc, !enc->has_state, y_ac_qi, out, cap, size);
}

int vp8gpu_encoder_encode_with_target_size(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u,
                                           const uint8_t* v, size_t uv_stride, size_t target_size, uint8_t* out,
                                           size_t cap, size_t* size, int* chosen_qi) {
  if (!enc || !y || !u || !v || !size) return VP8GPU_ERR_LOGIC;
  cudaSetDevice(enc->e->device());
  memset(enc->tl, 0, sizeof(enc->tl));
  Phase whole(&enc->tl[7]);
  int rc;
  {
    Phase ph(&enc->tl[0]);
    rc = upload_source(enc, y, y_stride, u, v, uv_stride);
  }
  if (rc != VP8GPU_OK) return rc;
  // Encoder::encode_with_target_size (encoder.cc:592-629), statement for statement: bisection over y_ac_qi in
  // [4, 127] or within 16 of the last frame's index; a candidate's size is the sampled estimate
  const bool key = !enc->has_state;
  enc->est_n = 0;  // estimates of an earlier source are not this frame's
  int lo = 4, hi = 127;
  if (enc->last_qi >= 0) {
    if (enc->last_qi - 16 >= lo) lo = enc->last_qi - 16;
    if (enc->last_qi + 16 < hi) hi = enc->last_qi + 16;
  }
  int best = 255;
  while (lo <= hi) {
    const int qi = (lo + hi) / 2;
    size_t est = 0;
    rc = estimate_probe(enc, key, lo, hi, qi, &est);
    if (rc != VP8GPU_OK) return rc;
    if (est <= target_size || (lo == hi && best == 255)) {
      best = qi;
      hi = qi - 1;
    } else {
      lo = qi + 1;
    }
  }
  if (best == 255) return enc->e->fail(VP8GPU_ERR_LOGIC, "target size search failed");
  if (chosen_qi) *chosen_qi = best;
  return encode_final(enc, key, best, out, cap, size);
}

// Encoder::encode_with_minimum_ssim -> encode_with_quantizer_search (encoder.cc:510-557, 577-590): the
// coarsest quantiser whose reconstruction (after the loop-filter choice) still reaches minimum_ssim
int vp8gpu_encoder_encode_with_minimum_ssim(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u,
                                            const uint8_t* v, size_t uv_stride, double minimum_ssim, uint8_t* out,
                                            size_t cap, size_t* size, int* chosen_qi) {
  if (!enc || !y || !u || !v || !size) return VP8GPU_ERR_LOGIC;
  cudaSetDevice(enc->e->device());
  int rc = upload_source(enc, y, y_stride, u, v, uv_stride);
  if (rc != VP8GPU_OK) return rc;
  const bool key = !enc->has_state;
  int lo = 0, hi = 127, best = 0;
  bool found = false;
  while (lo <= hi) {
    const int qi = (lo + hi) / 2;
    int frame = -1, lf = 0;
    double ssim = -1.0;
    rc = encode_core(enc, key, qi, 1, &frame);
    if (rc != VP8GPU_OK) return rc;
    rc = choose_loop_filter(enc, &frame, key, &lf, &ssim);
    enc->e->frame_release(frame);
    if (rc != VP8GPU_OK) return rc;
    if (ssim >= minimum_ssim || (lo == hi && !found)) {
      found = true;
      best = qi;
    }
    if (lo == hi) break;
    if (ssim < minimum_ssim) hi = qi - 1;
    else lo = qi + 1;
  }
  if (chosen_qi) *chosen_qi = best;
  return encode_final(enc, key, best, out, cap, size);
}

int vp8gpu_encoder_estimate_frame_size(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u,
                                       const uint8_t* v, size_t uv_stride, int y_ac_qi, size_t* size) {
  if (!enc || !y || !u || !v || !size || y_ac_qi < 0 || y_ac_qi > 127) return VP8GPU_ERR_LOGIC;
  cudaSetDevice(enc->e->device());
  int rc = upload_source(enc, y, y_stride, u, v, uv_stride);
  if (rc != VP8GPU_OK) return rc;
  return estimate_size(enc, !enc->has_state, y_ac_qi, size);
}

// Encoder( ..., two_pass, ... ) (encoder.hh:347-351): key frames are coded twice, the second time with trellis
// quantisation (encoder.cc:220-408); inter frames are unaffected, as in the reference (encode_inter.cc codes FIRST_PASS)
int vp8gpu_encoder_set_two_pass(vp8gpu_encoder* enc, int on) {
  if (!enc) return VP8GPU_ERR_LOGIC;
  enc->two_pass = on != 0;
  return VP8GPU_OK;
}

// Encoder( ..., quality ): fixed once the first frame is written, like the constructor argument it stands for
int vp8gpu_encoder_set_quality(vp8gpu_encoder* enc, int quality) {
  if (!enc || (quality != VP8GPU_QUALITY_BEST && quality != VP8GPU_QUALITY_REALTIME)) return VP8GPU_ERR_LOGIC;
  if (enc->quality_fixed) return enc->e->fail(VP8GPU_ERR_LOGIC, "set_quality: the encoder has written a frame");
  enc->quality = quality;
  return VP8GPU_OK;
}

// bitstream writer: 0 = byte-identical to the reference Encoder's output (default), 1 = compact / parallel
int vp8gpu_encoder_set_writer(vp8gpu_encoder* enc, int mode) {
  if (!enc || mode < 0 || mode > 1) return VP8GPU_ERR_LOGIC;
  enc->writer = mode;
  return VP8GPU_OK;
}

// EncoderStats (encoder.hh:118-127) of the last frame: luma SSIM after the loop filter, the chosen
// loop-filter level and quantiser index
int vp8gpu_encoder_stats(const vp8gpu_encoder* enc, double* ssim, int* loop_filter_level, int* y_ac_qi) {
  if (!enc) return VP8GPU_ERR_LOGIC;
  if (ssim) *ssim = enc->last_ssim;
  if (loop_filter_level) *loop_filter_level = enc->stat_lf;
  if (y_ac_qi) *y_ac_qi = enc->stat_qi;
  return VP8GPU_OK;
}

int vp8gpu_encoder_timeline(const vp8gpu_encoder* enc, double* ms, int n) {
  if (!enc || !ms || n < 0) return VP8GPU_ERR_LOGIC;
  for (int i = 0; i < n && i < 8; i++) ms[i] = enc->tl[i];
  return VP8GPU_OK;
}

// the reconstruction kept as LAST (one new reference for the caller)
int vp8gpu_encoder_reconstruction(vp8gpu_encoder* enc, vp8gpu_frame_id* out) {
  if (!enc || !out || enc->refs[0] < 0) return VP8GPU_ERR_LOGIC;
  const int rc = enc->e->frame_retain(enc->refs[0]);
  if (rc == VP8GPU_OK) *out = enc->refs[0];
  return rc;
}

// Encoder::export_decoder (encoder.hh:378): a Decoder in the state a receiver is in after the frames emitted
// so far -- DecoderState + the three references (shared, not copied)
int vp8gpu_encoder_export_decoder(vp8gpu_encoder* enc, vp8gpu_decoder** out) {
  if (!enc || !out) return VP8GPU_ERR_LOGIC;
  // an Encoder that has not emitted a frame yet exports the Decoder it was built with: a fresh one
  // (Encoder( width, height, ... ) holds DecoderState( width, height ) and blank References, encoder.cc:68-90)
  if (!enc->has_state) return vp8gpu_decoder_create(enc->ctx, out);
  const std::vector<uint8_t> blob = enc->dec_state->serialize();
  vp8gpu_state* st = nullptr;
  int rc = vp8gpu_state_deserialize(blob.data(), blob.size(), &st);
  if (rc != VP8GPU_OK) return rc;
  rc = vp8gpu_decoder_create_from(enc->ctx, st, enc->refs, out);
  vp8gpu_state_destroy(st);
  return rc;
}

// Encoder::minihash (encoder.hh:382) = export_decoder().minihash()
int vp8gpu_encoder_minihash(vp8gpu_encoder* enc, uint32_t* out) {
  if (!enc || !out) return VP8GPU_ERR_LOGIC;
  vp8gpu_decoder* d = nullptr;
  int rc = vp8gpu_encoder_export_decoder(enc, &d);
  if (rc != VP8GPU_OK) return rc;
  uint64_t h = 0;
  rc = vp8gpu_decoder_hash(d, &h);
  vp8gpu_decoder_destroy(d);
  if (rc == VP8GPU_OK) *out = (uint32_t)(h ^ (h >> 32));  // same fold as Decoder::minihash
  return rc;
}

// ---- re-encoding (SURVEY.md 8 row f3; encoder/reencode.cc) -------------------------------------------------

// Encoder::write_frame's state update (encoder.cc:146-170): decode the emitted frame like any receiver
// (Frame::decode + loopfilter + copy_to on the device, through the library's own Decoder) and adopt the
// DecoderState and References it ends with.
// mbs / tokens: the records and token lists the frame was serialised from (enc->h_mbs / h_tokens), when it was --
// the decode then skips parsing the DCT partitions back (capi.cc vp8gpu_decoder_decode_known_tokens)
static int apply_emitted_frame(vp8gpu_encoder* enc, const uint8_t* data, size_t len, const vp8gpu_mb* mbs, const vp8gpu_token* tokens,
                               uint32_t n_tok) {
  Engine* e = enc->e;
  vp8gpu_decoder* d = nullptr;
  int rc = vp8gpu_encoder_export_decoder(enc, &d);
  if (rc != VP8GPU_OK) return rc;
  int shown = 0;
  vp8gpu_frame_id raster = -1;
  if (mbs && enc_speculate()) rc = vp8gpu_decoder_decode_known_tokens(d, data, len, mbs, tokens, n_tok, &shown, &raster);
  else rc = vp8gpu_decoder_decode(d, data, len, &shown, &raster);
  if (rc == VP8GPU_OK) {
    if (raster >= 0) e->frame_release(raster);
    const std::vector<uint8_t> blob = [&] {
      const vp8gpu_state* st = vp8gpu_decoder_state(d);
      std::vector<uint8_t> b(vp8gpu_state_serialize(st, nullptr, 0));
      vp8gpu_state_serialize(st, b.data(), b.size());
      return b;
    }();
    if (!vp8::State::deserialize(blob.data(), blob.size(), *enc->dec_state)) rc = e->fail(VP8GPU_ERR_LOGIC, "write_frame: bad decoder state");
  }
  if (rc == VP8GPU_OK) {
    vp8gpu_frame_id refs[3];
    vp8gpu_decoder_references(d, refs);
    for (int k = 0; k < 3; k++)
      if (refs[k] >= 0) e->frame_retain(refs[k]);
    for (int k = 0; k < 3; k++) {
      if (enc->refs[k] >= 0) e->frame_release(enc->refs[k]);
      enc->refs[k] = refs[k];
    }
    enc->has_state = true;
    enc->stat_frames++;
  }
  vp8gpu_decoder_destroy(d);
  return rc;
}

static int emit(vp8gpu_encoder* enc, const std::vector<uint8_t>& bytes, uint8_t* out, size_t cap, size_t* size, const vp8gpu_mb* mbs = nullptr,
                const vp8gpu_token* tokens = nullptr, uint32_t n_tok = 0) {
  *size = bytes.size();
  if (!out || cap < bytes.size()) return enc->e->fail(VP8GPU_ERR_NOMEM, "output buffer too small");
  memcpy(out, bytes.data(), bytes.size());
  return apply_emitted_frame(enc, bytes.data(), bytes.size(), mbs, tokens, n_tok);
}

// Encoder::write_frame( KeyFrame ) (encoder.cc:146-176) as Encoder::reencode uses it for a key frame that is kept
// (reencode.cc option 3): Frame::serialize of the parsed frame -- its own bytes -- and the Encoder moves past it.
int vp8gpu_encoder_write_frame(vp8gpu_encoder* enc, const vp8gpu_parsed* frame, uint8_t* out, size_t cap, size_t* size) {
  const vp8::ParsedFrame* pf = vp8gpu_parsed_frame(frame);
  if (!enc || !pf || !size) return VP8GPU_ERR_LOGIC;
  if (!pf->desc.key_frame) return enc->e->fail(VP8GPU_ERR_UNSUPPORTED, "write_frame: only key frames are written back unchanged");
  if (pf->desc.width != enc->e->width() || pf->desc.height != enc->e->height()) return enc->e->fail(VP8GPU_ERR_LOGIC, "write_frame: raster size mismatch");
  cudaSetDevice(enc->e->device());
  const std::vector<uint8_t> bytes = vp8::serialize_parsed(*pf);
  if (bytes.empty()) return enc->e->fail(VP8GPU_ERR_LOGIC, "write_frame: the frame was parsed without vp8gpu_parsed_keep_labels");
  const int rc = emit(enc, bytes, out, cap, size);
  if (rc == VP8GPU_OK) remember_frame(enc, pf->verbatim.y_ac_qi, pf->verbatim.lf_level);
  return rc;
}

// Encoder::update_residues + write_frame (encoder/reencode.cc:131-313): the prediction frame's modes, vectors,
// references and header are kept, its residues are recomputed against THIS encoder's references so that the frame
// decodes close to the target raster; y_ac_qi < 0 keeps the frame's own quantiser index (the deltas always stay).
int vp8gpu_encoder_update_residues(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u, const uint8_t* v,
                                   size_t uv_stride, const vp8gpu_parsed* prediction_frame, int y_ac_qi, int last_frame, uint8_t* out,
                                   size_t cap, size_t* size) {
  const vp8::ParsedFrame* pf = vp8gpu_parsed_frame(prediction_frame);
  if (!enc || !y || !u || !v || !pf || !size || y_ac_qi > 127) return VP8GPU_ERR_LOGIC;
  Engine* e = enc->e;
  const vp8::Geom& g = e->geom();
  const vp8::Verbatim& vb = pf->verbatim;
  const size_t n_mbs = (size_t)g.mb_cols * g.mb_rows;
  if (pf->desc.key_frame) return e->fail(VP8GPU_ERR_LOGIC, "update_residues: the prediction frame is a key frame");
  if (vb.header_tape.empty() || vb.mb_coded.size() != n_mbs)
    return e->fail(VP8GPU_ERR_LOGIC, "update_residues: the prediction frame was parsed without vp8gpu_parsed_keep_labels");
  if (pf->desc.mb_cols != g.mb_cols || pf->desc.mb_rows != g.mb_rows) return e->fail(VP8GPU_ERR_LOGIC, "update_residues: raster size mismatch");
  if (!enc->has_state || enc->refs[0] < 0 || enc->refs[1] < 0 || enc->refs[2] < 0)
    return e->fail(VP8GPU_ERR_LOGIC, "update_residues: the encoder has no references yet");
  // The reference copies update_segmentation into the new header but not the macroblocks' segment ids (a blank
  // frame's macroblocks carry none, reencode.cc:259, macroblock.cc:55-58): when the prediction frame updates the
  // segment map the frame the reference writes cannot be parsed.  Not reproduced.  Segmentation without a map
  // update is reproduced as it is: one Quantizer for the residues (reencode.cc:283) whatever the segments say.
  if (vb.read_segment) return e->fail(VP8GPU_ERR_UNSUPPORTED, "update_residues: the prediction frame updates the segment map");
  cudaSetDevice(e->device());
  int rc = upload_source(enc, y, y_stride, u, v, uv_stride);
  if (rc != VP8GPU_OK) return rc;
  if (int lrc = e->ensure_lane(enc->lane)) return lrc;
  cudaStream_t s = e->stream(enc->lane);

  const int qi = y_ac_qi < 0 ? vb.y_ac_qi : y_ac_qi;
  vp8gpu_quant q;  // Quantizer::Quantizer (quantization.cc:83-93) of the frame's indices with y_ac_qi replaced
  q.y_ac = k_ac_q[clamp_q(qi)];
  q.y_dc = k_dc_q[clamp_q(qi + vb.q_delta[0])];
  q.y2_dc = static_cast<uint16_t>(k_dc_q[clamp_q(qi + vb.q_delta[1])] * 2);
  q.y2_ac = static_cast<uint16_t>(k_ac_q[clamp_q(qi + vb.q_delta[2])] * 155 / 100);
  q.uv_dc = k_dc_q[clamp_q(qi + vb.q_delta[3])];
  q.uv_ac = k_ac_q[clamp_q(qi + vb.q_delta[4])];
  if (q.y2_ac < 8) q.y2_ac = 8;
  if (q.uv_dc > 132) q.uv_dc = 132;

  // records: the frame's, with empty token lists (step 1 predicts, steps 2 and 4 fill the lists in)
  size_t n_intra = 0;
  for (size_t i = 0; i < n_mbs; i++) {
    vp8gpu_mb m = pf->mbs.data()[i];
    m.tok_off = 0;
    m.tok_cnt = 0;
    m.flags = (m.y_mode != VP8GPU_B_PRED && m.y_mode != VP8GPU_SPLITMV) ? VP8GPU_MB_HAS_Y2 : 0;
    if (m.y_mode == VP8GPU_SPLITMV && m.split_idx >= pf->desc.n_split) return e->fail(VP8GPU_ERR_LOGIC, "update_residues: bad split index");
    n_intra += m.ref_frame == VP8GPU_REF_CURRENT;
    enc->h_mbs[i] = m;
  }
  const size_t split_bytes = (size_t)pf->desc.n_split * sizeof(vp8gpu_split_mvs);
  if (split_bytes > enc->split_cap) {
    if (enc->d_split) cudaFree(enc->d_split);
    enc->d_split = nullptr;
    enc->split_cap = 0;
    if (cudaMalloc(&enc->d_split, n_mbs * sizeof(vp8gpu_split_mvs)) != cudaSuccess) return e->fail(VP8GPU_ERR_NOMEM, "update_residues: split buffer");
    enc->split_cap = n_mbs * sizeof(vp8gpu_split_mvs);
  }

  int recon = -1;
  rc = e->frame_alloc(&recon);
  if (rc != VP8GPU_OK) return rc;
  auto fail = [&](int code) {
    e->frame_release(recon);
    return code;
  };
  int ids[5] = {enc->src, recon, enc->refs[0], -1, -1};
  int n_ids = 3;
  for (int k = 1; k < 3; k++) {
    bool dup = false;
    for (int j = 2; j < n_ids; j++) dup |= ids[j] == enc->refs[k];
    if (!dup) ids[n_ids++] = enc->refs[k];
  }
  rc = e->acquire_frames(enc->lane, ids, n_ids, 2u);  // only `recon` is written
  if (rc != VP8GPU_OK) return fail(rc);

  memset(enc->h_hdr, 0, 1024);
  vp8::ReencJob* rj = reinterpret_cast<vp8::ReencJob*>(enc->h_hdr);
  vp8::DevJob* dj = reinterpret_cast<vp8::DevJob*>(enc->h_hdr + 512);
  int* d_sync = reinterpret_cast<int*>(enc->dev + enc->off_sync);
  vp8gpu_mb* d_mbs = reinterpret_cast<vp8gpu_mb*>(enc->dev + enc->off_mbs);
  vp8gpu_token* d_tok = reinterpret_cast<vp8gpu_token*>(enc->dev + enc->off_tokens);
  rj->target = e->frame_dev(enc->src);
  rj->recon = e->frame_dev(recon);
  rj->mbs_in = d_mbs;
  rj->mbs_out = d_mbs;
  rj->tokens = d_tok;
  rj->tok_counter = reinterpret_cast<uint32_t*>(d_sync + 96);
  rj->tok_cap = enc->tok_cap;
  rj->progress = d_sync + 128;
  rj->q = q;
  rj->cols = (uint16_t)g.mb_cols;
  rj->rows = (uint16_t)g.mb_rows;
  dj->mbs = d_mbs;
  dj->tokens = d_tok;
  dj->split = reinterpret_cast<const vp8gpu_split_mvs*>(enc->d_split);
  dj->out = e->frame_dev(recon);
  for (int k = 0; k < 3; k++) {
    dj->ref[k] = e->frame_dev(enc->refs[k]);
    dj->ref_tmap[k] = e->frame_tmaps(enc->refs[k]);
  }
  dj->intra_progress = d_sync + 128;
  dj->lf_progress = d_sync + 128 + g.mb_rows;
  for (int k = 0; k < 4; k++) dj->quant[k] = q;
#define CUF(call)                                                        \
  do {                                                                   \
    cudaError_t e__ = (call);                                            \
    if (e__ != cudaSuccess) return fail(e->cuda_fail(e__, #call));       \
  } while (0)
  CUF(cudaMemcpyAsync(enc->dev + enc->off_encjob, enc->h_hdr, 1024, cudaMemcpyHostToDevice, s));
  CUF(cudaMemcpyAsync(d_mbs, enc->h_mbs, n_mbs * sizeof(vp8gpu_mb), cudaMemcpyHostToDevice, s));
  if (split_bytes) CUF(cudaMemcpyAsync(enc->d_split, pf->split.data(), split_bytes, cudaMemcpyHostToDevice, s));
  CUF(cudaMemsetAsync(d_sync, 0, sizeof(int) * (128 + 2 * (size_t)g.mb_rows), s));
  const vp8::ReencJob* d_rj = reinterpret_cast<const vp8::ReencJob*>(enc->dev + enc->off_encjob);
  const vp8::DevJob* d_dj = reinterpret_cast<const vp8::DevJob*>(enc->dev + enc->off_encjob + 512);
  int launches = 0;
  if (n_intra < n_mbs) {
    if (int ce = vp8::launch_inter(d_dj, 1, g, s)) return fail(e->cuda_fail((cudaError_t)ce, "k_inter (prediction)"));
    if (int ce = vp8::launch_reenc_inter(d_rj, (int)n_mbs, g, s)) return fail(e->cuda_fail((cudaError_t)ce, "k_reenc_inter"));
    if (int ce = vp8::launch_inter(d_dj, 1, g, s)) return fail(e->cuda_fail((cudaError_t)ce, "k_inter (reconstruction)"));
    launches += 3;
  }
  if (n_intra) {
    if (int ce = vp8::launch_reenc_intra(d_rj, g.mb_rows, g, d_sync + 0, s)) return fail(e->cuda_fail((cudaError_t)ce, "k_reenc_intra"));
    launches++;
  }
  e->count_launches(launches);
  e->mark_frames(enc->lane, ids, n_ids, 2u);
  CUF(cudaMemcpyAsync(enc->h_count, rj->tok_counter, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CUF(cudaMemcpyAsync(enc->h_mbs, d_mbs, n_mbs * sizeof(vp8gpu_mb), cudaMemcpyDeviceToHost, s));
  CUF(cudaStreamSynchronize(s));
  const uint32_t n_tok = *enc->h_count;
  if (n_tok > enc->tok_cap) return fail(e->fail(VP8GPU_ERR_NOMEM, "update_residues: token pool overflow"));
  if (n_tok) {
    CUF(cudaMemcpyAsync(enc->h_tokens, d_tok, (size_t)n_tok * sizeof(vp8gpu_token), cudaMemcpyDeviceToHost, s));
    CUF(cudaStreamSynchronize(s));
  }
#undef CUF
  e->frame_release(recon);  // the reference discards its reconstruction too: write_frame decodes the frame it wrote

  // ---- the frame: header sections of the prediction frame + the reference Encoder's probability decisions ----
  vp8::EncodeHeader h;
  h.key_frame = false;
  h.show_frame = true;  // InterFrame( width, height ): a new frame object is shown
  h.width = e->width();
  h.height = e->height();
  h.y_ac_qi = qi;
  vp8::EncodeFeatures ft;
  vp8::EncodeFeatures::RefWriterState fresh;  // update_residues builds a new InterFrame object every time
  fresh.prob_last = vb.prob_last;              // prob_references_* are copied from the prediction frame (reencode.cc:266-267)
  fresh.prob_golden = vb.prob_golden;
  ft.ref_writer = &fresh;
  ft.residue_of = &vb;
  ft.residue_refresh_all = last_frame != 0;
  ft.log2_partitions = 0;
  uint8_t probs[1056];
  memcpy(probs, enc->dec_state->coef_probs, 1056);
  ft.saved_coef_probs = probs;
  ft.ymode_probs = enc->dec_state->ymode_probs;
  ft.uvmode_probs = enc->dec_state->uvmode_probs;
  ft.mv_probs = enc->dec_state->mv_probs;
  const std::vector<uint8_t> bytes = vp8::serialize_frame(h, enc->h_mbs, enc->h_tokens, pf->split.data(), &ft);
  if (bytes.empty()) return e->fail(VP8GPU_ERR_LOGIC, "update_residues: serializer rejected the records");
  rc = emit(enc, bytes, out, cap, size, enc->h_mbs, enc->h_tokens, n_tok);
  if (rc == VP8GPU_OK) remember_frame(enc, qi, vb.lf_level);  // write_frame
  return rc;
}

// Encoder::reencode_as_interframe + write_frame (encoder/reencode.cc:39-129, 343-351): the chunk's initial key
// frame is coded again as an inter frame predicted from this encoder's LAST -- the ordinary inter-frame decision loop
// (k_enc_rd) at the key frame's quantiser indices with y_ac_qi replaced, without update_rd_multipliers and
// fill_mv_sad_costs (the reference does not call them here), the key frame's sharpness, all references refreshed.
int vp8gpu_encoder_reencode_as_interframe(vp8gpu_encoder* enc, const uint8_t* y, size_t y_stride, const uint8_t* u, const uint8_t* v,
                                          size_t uv_stride, const vp8gpu_parsed* key_frame, int y_ac_qi, uint8_t* out, size_t cap,
                                          size_t* size) {
  const vp8::ParsedFrame* pf = vp8gpu_parsed_frame(key_frame);
  if (!enc || !y || !u || !v || !pf || !size || y_ac_qi < 0 || y_ac_qi > 127) return VP8GPU_ERR_LOGIC;
  Engine* e = enc->e;
  const vp8::Verbatim& vb = pf->verbatim;
  if (!pf->desc.key_frame) return e->fail(VP8GPU_ERR_LOGIC, "reencode_as_interframe: not a key frame");
  if (vb.header_tape.empty()) return e->fail(VP8GPU_ERR_LOGIC, "reencode_as_interframe: the frame was parsed without vp8gpu_parsed_keep_labels");
  if (pf->desc.width != e->width() || pf->desc.height != e->height()) return e->fail(VP8GPU_ERR_LOGIC, "reencode_as_interframe: raster size mismatch");
  if (vb.seg_enabled) return e->fail(VP8GPU_ERR_UNSUPPORTED, "segmentation not supported");  // reencode.cc:49-51
  if (!enc->has_state || enc->refs[0] < 0) return e->fail(VP8GPU_ERR_LOGIC, "reencode_as_interframe: the encoder has no references yet");
  cudaSetDevice(e->device());
  int rc = upload_source(enc, y, y_stride, u, v, uv_stride);
  if (rc != VP8GPU_OK) return rc;
  vp8gpu_quant q;
  q.y_ac = k_ac_q[clamp_q(y_ac_qi)];
  q.y_dc = k_dc_q[clamp_q(y_ac_qi + vb.q_delta[0])];
  q.y2_dc = static_cast<uint16_t>(k_dc_q[clamp_q(y_ac_qi + vb.q_delta[1])] * 2);
  q.y2_ac = static_cast<uint16_t>(k_ac_q[clamp_q(y_ac_qi + vb.q_delta[2])] * 155 / 100);
  q.uv_dc = k_dc_q[clamp_q(y_ac_qi + vb.q_delta[3])];
  q.uv_ac = k_ac_q[clamp_q(y_ac_qi + vb.q_delta[4])];
  if (q.y2_ac < 8) q.y2_ac = 8;
  if (q.uv_dc > 132) q.uv_dc = 132;

  int frame = -1, lf = 0;
  double ssim = -1.0;
  rc = encode_core(enc, false, y_ac_qi, 1, &frame, &q);
  if (rc != VP8GPU_OK) return rc;
  enc->lf_sharpness = pf->desc.sharpness;
  rc = choose_loop_filter(enc, &frame, false, &lf, &ssim);  // apply_best_loopfilter_settings (reencode.cc:126)
  enc->lf_sharpness = 0;
  e->frame_release(frame);  // write_frame decodes the frame it wrote (encoder.cc:153-158)
  if (rc != VP8GPU_OK) return rc;

  vp8::EncodeHeader h;
  h.key_frame = false;
  h.show_frame = true;
  h.width = e->width();
  h.height = e->height();
  h.y_ac_qi = y_ac_qi;
  h.loop_filter_level = lf;
  h.sharpness = pf->desc.sharpness;
  vp8::EncodeFeatures ft;
  vp8::EncodeFeatures::RefWriterState fresh;  // a new InterFrame object
  ft.ref_writer = &fresh;
  ft.from_key = &vb;
  ft.log2_partitions = 0;
  ft.refresh_golden = ft.refresh_alternate = ft.refresh_last = true;
  ft.refresh_entropy_probs = true;
  uint8_t probs[1056];
  memcpy(probs, enc->dec_state->coef_probs, 1056);
  ft.saved_coef_probs = probs;
  ft.mv_probs = enc->dec_state->mv_probs;  // the mode probabilities are the defaults the header itself sets
  std::vector<uint8_t> bytes = vp8::serialize_frame(h, enc->h_mbs, enc->h_tokens, nullptr, &ft);
  if (bytes.empty()) return e->fail(VP8GPU_ERR_LOGIC, "reencode_as_interframe: serializer rejected the device records");
  rc = emit(enc, bytes, out, cap, size, enc->h_mbs, enc->h_tokens, *enc->h_count);
  if (rc == VP8GPU_OK) {
    remember_frame(enc, y_ac_qi, lf);
    enc->last_ssim = ssim;
  }
  return rc;
}

}  // extern "C"
