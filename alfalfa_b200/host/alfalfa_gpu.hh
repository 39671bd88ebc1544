// alfalfa_gpu.hh -- C++ host-side mirror of the reference's decoder interface on top of the C ABI
// (include/vp8gpu.h).  Same class and method names, argument meaning and error behaviour as
// /root/reference/src/decoder/decoder.hh:123-300 and raster_handle.hh, so that callers such as
// FramePlayer::decode (player.cc:60), xc-dump, xc-enc or salsify-receiver keep compiling when
// the include is switched (INTEGRATION.md).  Header-only; link with -lvp8gpu.
#pragma once
#include <cstdint>
#include <cmath>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../include/vp8gpu.h"

namespace alfalfa_gpu {

// util/exception.hh:76-98
class Invalid : public std::runtime_error { public: using std::runtime_error::runtime_error; };
class Unsupported : public std::runtime_error { public: using std::runtime_error::runtime_error; };
class LogicError : public std::logic_error { public: using std::logic_error::logic_error; };
class DeviceError : public std::runtime_error { public: using std::runtime_error::runtime_error; };

inline void check(int rc, vp8gpu_ctx* ctx, const char* what) {
  if (rc == VP8GPU_OK) return;
  const std::string msg = std::string(what) + ": " + (ctx ? vp8gpu_last_error(ctx) : "");
  switch (rc) {
    case VP8GPU_ERR_INVALID: throw Invalid(msg);
    case VP8GPU_ERR_UNSUPPORTED: throw Unsupported(msg);
    case VP8GPU_ERR_LOGIC: throw LogicError(msg);
    default: throw DeviceError(msg);
  }
}

// util/chunk.hh:38: a (pointer, length) view of compressed bytes
struct Chunk {
  const uint8_t* buffer;
  uint64_t size;
  Chunk(const uint8_t* b, uint64_t n) : buffer(b), size(n) {}
  explicit Chunk(const std::vector<uint8_t>& v) : buffer(v.data()), size(v.size()) {}
};

// one context per (device, frame size); shared by every Decoder of that size
class Context {
  std::shared_ptr<vp8gpu_ctx> h_;
 public:
  Context(int device, uint16_t width, uint16_t height, int max_frames = 0) {
    vp8gpu_ctx* c = nullptr;
    check(vp8gpu_ctx_create(device, width, height, max_frames, &c), nullptr, "vp8gpu_ctx_create");
    h_.reset(c, vp8gpu_ctx_destroy);
  }
  vp8gpu_ctx* get() const { return h_.get(); }
  void sync() const { check(vp8gpu_ctx_sync(get()), get(), "sync"); }
  // vp8gpu_decode_ivf: DCT partitions on the device (default) or on the host workers
  void set_device_tokens(bool on) const {
    check(vp8gpu_ctx_set_option(get(), VP8GPU_OPT_DEVICE_TOKENS, on), get(), "set_option");
  }
};

// RasterHandle (raster_handle.hh:95-123): shared, immutable, device resident
class RasterHandle {
  struct Rep {
    Context ctx;
    vp8gpu_frame_id id;
    Rep(const Context& c, vp8gpu_frame_id i) : ctx(c), id(i) {}
    ~Rep() { vp8gpu_frame_release(ctx.get(), id); }
  };
  std::shared_ptr<const Rep> rep_;
 public:
  RasterHandle() = default;
  RasterHandle(const Context& c, vp8gpu_frame_id owned_id) : rep_(std::make_shared<Rep>(c, owned_id)) {}
  vp8gpu_frame_id id() const { return rep_->id; }
  bool initialized() const { return static_cast<bool>(rep_); }
  bool operator==(const RasterHandle& o) const { return rep_ == o.rep_; }
  // BaseRaster::quality (util/raster.cc:63-66): luma SSIM
  double quality(const RasterHandle& other) const {
    double q = 0;
    check(vp8gpu_frame_ssim(rep_->ctx.get(), rep_->id, other.rep_->id, &q), rep_->ctx.get(), "quality");
    return q;
  }
  // BaseRaster::dump (util/raster.cc:85-114): display rectangle, planar Y,U,V; blocks until decoded
  std::vector<uint8_t> dump(uint16_t width, uint16_t height) const {
    std::vector<uint8_t> out(size_t(width) * height + 2 * size_t((width + 1) / 2) * ((height + 1) / 2));
    check(vp8gpu_frame_download_display(rep_->ctx.get(), rep_->id, out.data(), out.size()), rep_->ctx.get(), "dump");
    return out;
  }
};

// DecoderState (decoder.hh:190-225) as a value
class DecoderState {
  std::shared_ptr<vp8gpu_state> h_;
 public:
  DecoderState(unsigned width, unsigned height) {
    vp8gpu_state* s = nullptr;
    check(vp8gpu_state_create(width, height, &s), nullptr, "state_create");
    h_.reset(s, vp8gpu_state_destroy);
  }
  explicit DecoderState(const vp8gpu_state* borrowed) {
    vp8gpu_state* s = nullptr;
    check(vp8gpu_state_clone(borrowed, &s), nullptr, "state_clone");
    h_.reset(s, vp8gpu_state_destroy);
  }
  const vp8gpu_state* get() const { return h_.get(); }
  bool operator==(const DecoderState& o) const { return vp8gpu_state_equal(get(), o.get()); }
  bool operator!=(const DecoderState& o) const { return !(*this == o); }
  size_t hash() const { return vp8gpu_state_hash(get()); }
  // DecoderState::serialize / deserialize (decoder.cc:283-330): the reference's DECODER_STATE record
  std::vector<uint8_t> serialize() const {
    std::vector<uint8_t> b(vp8gpu_state_serialize(get(), nullptr, 0));
    vp8gpu_state_serialize(get(), b.data(), b.size());
    return b;
  }
  static DecoderState deserialize(const std::vector<uint8_t>& blob) {
    vp8gpu_state* s = nullptr;
    check(vp8gpu_state_deserialize(blob.data(), blob.size(), &s), nullptr, "state_deserialize");
    DecoderState out(s);  // clones
    vp8gpu_state_destroy(s);
    return out;
  }
};

// References (decoder.hh:123-149)
struct References {
  RasterHandle last, golden, alternative;
};

// KeyFrame / InterFrame (frame.hh:126-127) in flat form
class ParsedFrame {
  std::shared_ptr<vp8gpu_parsed> h_;
 public:
  ParsedFrame() {
    vp8gpu_parsed* p = nullptr;
    check(vp8gpu_parsed_create(&p), nullptr, "parsed_create");
    h_.reset(p, vp8gpu_parsed_destroy);
  }
  vp8gpu_parsed* get() const { return h_.get(); }
  // the reference's Frame objects keep their header as coded and every label; the flat records keep them on request
  // (needed by Encoder::reencode and by byte-exact re-serialisation)
  void keep_labels(bool on = true) { check(vp8gpu_parsed_keep_labels(get(), on), nullptr, "parsed_keep_labels"); }
  int y_ac_qi() const { return vp8gpu_parsed_y_ac_qi(get()); }  // header().quant_indices.y_ac_qi (needs keep_labels)
  bool show_frame() const { return vp8gpu_parsed_desc(get())->show_frame; }
  bool key_frame() const { return vp8gpu_parsed_desc(get())->key_frame; }
};

// Decoder (decoder.hh:244-300).  Copying is O(1) in pixels and shares the reference rasters.
class Decoder {
  Context ctx_;
  uint16_t width_, height_;
  vp8gpu_decoder* h_ = nullptr;
 public:
  Decoder(const Context& ctx, uint16_t width, uint16_t height) : ctx_(ctx), width_(width), height_(height) {
    check(vp8gpu_decoder_create(ctx_.get(), &h_), ctx_.get(), "decoder_create");
  }
  Decoder(const Context& ctx, const DecoderState& state, const References& refs, uint16_t width, uint16_t height)
      : ctx_(ctx), width_(width), height_(height) {
    const vp8gpu_frame_id ids[3] = {refs.last.id(), refs.golden.id(), refs.alternative.id()};
    check(vp8gpu_decoder_create_from(ctx_.get(), state.get(), ids, &h_), ctx_.get(), "decoder_create_from");
  }
  // takes ownership of a decoder handle made by the C ABI (Encoder::export_decoder)
  Decoder(const Context& ctx, vp8gpu_decoder* owned, uint16_t width, uint16_t height)
      : ctx_(ctx), width_(width), height_(height), h_(owned) {}
  Decoder(const Decoder& o) : ctx_(o.ctx_), width_(o.width_), height_(o.height_) {
    check(vp8gpu_decoder_clone(o.h_, &h_), ctx_.get(), "decoder_clone");
  }
  Decoder& operator=(const Decoder& o) {
    if (this != &o) {
      Decoder tmp(o);
      std::swap(h_, tmp.h_);
    }
    return *this;
  }
  ~Decoder() { vp8gpu_decoder_destroy(h_); }

  uint16_t get_width() const { return width_; }
  uint16_t get_height() const { return height_; }
  vp8gpu_decoder* handle() const { return h_; }
  const Context& context() const { return ctx_; }

  // parse_frame<KeyFrame|InterFrame>( decompress_frame( chunk ) ) (decoder.cc:83-98)
  ParsedFrame parse_frame(const Chunk& compressed_frame, bool keep_labels = false) {
    ParsedFrame p;
    if (keep_labels) p.keep_labels();
    check(vp8gpu_parse_frame(vp8gpu_decoder_state(h_), compressed_frame.buffer, compressed_frame.size, p.get()),
          ctx_.get(), "parse_frame");
    return p;
  }
  // decode_frame (decoder.cc:101-118)
  std::pair<bool, RasterHandle> decode_frame(const ParsedFrame& frame) {
    int shown = 0;
    vp8gpu_frame_id id = -1;
    check(vp8gpu_decoder_decode_parsed(h_, frame.get(), &shown, &id), ctx_.get(), "decode_frame");
    return {shown != 0, RasterHandle(ctx_, id)};
  }
  // get_frame_output (decoder.cc:125-135)
  std::pair<bool, RasterHandle> get_frame_output(const Chunk& compressed_frame) {
    int shown = 0;
    vp8gpu_frame_id id = -1;
    check(vp8gpu_decoder_decode(h_, compressed_frame.buffer, compressed_frame.size, &shown, &id), ctx_.get(),
          "get_frame_output");
    return {shown != 0, RasterHandle(ctx_, id)};
  }
  // leave the DCT partitions of get_frame_output to the device (same output, less host time)
  void set_device_tokens(bool on) { check(vp8gpu_decoder_set_device_tokens(h_, on), ctx_.get(), "set_device_tokens"); }
  // parse_and_decode_frame (decoder.cc:137-141): empty handle for hidden frames
  RasterHandle parse_and_decode_frame(const Chunk& compressed_frame) {
    auto out = get_frame_output(compressed_frame);
    return out.first ? out.second : RasterHandle();
  }
  // Decoder::serialize / deserialize (decoder.cc:54-81): the reference's EncoderStateSerializer format
  std::vector<uint8_t> serialize() const {
    size_t n = 0;
    vp8gpu_decoder_serialize(h_, nullptr, 0, &n);
    std::vector<uint8_t> b(n);
    check(vp8gpu_decoder_serialize(h_, b.data(), b.size(), &n), ctx_.get(), "decoder_serialize");
    return b;
  }
  static Decoder deserialize(const Context& ctx, const std::vector<uint8_t>& blob, uint16_t width, uint16_t height) {
    vp8gpu_decoder* d = nullptr;
    check(vp8gpu_decoder_deserialize(ctx.get(), blob.data(), blob.size(), &d), ctx.get(), "decoder_deserialize");
    return Decoder(ctx, d, width, height);
  }
  DecoderState get_state() const { return DecoderState(vp8gpu_decoder_state(h_)); }
  References get_references() const {
    vp8gpu_frame_id ids[3];
    vp8gpu_decoder_references(h_, ids);
    References r;
    RasterHandle* slots[3] = {&r.last, &r.golden, &r.alternative};
    for (int i = 0; i < 3; i++) {
      check(vp8gpu_frame_retain(ctx_.get(), ids[i]), ctx_.get(), "retain");
      *slots[i] = RasterHandle(ctx_, ids[i]);
    }
    return r;
  }
  // get_hash / minihash (decoder.hh:279-292): equal decoders hash equally (values are this library's)
  uint64_t get_hash() const {
    uint64_t h = 0;
    check(vp8gpu_decoder_hash(h_, &h), ctx_.get(), "decoder_hash");
    return h;
  }
  uint32_t minihash() const {
    const uint64_t h = get_hash();
    return static_cast<uint32_t>(h ^ (h >> 32));
  }
  bool operator==(const Decoder& o) const {
    int eq = 0;
    check(vp8gpu_decoder_equal(h_, o.h_, &eq), ctx_.get(), "decoder_equal");
    return eq != 0;
  }
  bool operator!=(const Decoder& o) const { return !(*this == o); }
};

// Encoder (encoder/encoder.hh:345-382).  The source raster is passed as display-size planes in host memory
// (the reference takes a VP8Raster filled by its input readers).  Like the reference's, an Encoder is a
// copyable value: copies share the (immutable) reference rasters and may encode concurrently on different
// threads (salsify/salsify-sender.cc:492-518).
struct SourceFrame {
  const uint8_t *y, *u, *v;
  size_t y_stride, uv_stride;
};

// EncoderQuality (encoder/encoder.hh:56-60), same order
enum EncoderQuality { BEST_QUALITY = VP8GPU_QUALITY_BEST, REALTIME_QUALITY = VP8GPU_QUALITY_REALTIME };

class Encoder {
  Context ctx_;
  uint16_t width_, height_;
  vp8gpu_encoder* h_ = nullptr;
  std::vector<uint8_t> buf_;

  std::vector<uint8_t> take(size_t n) const { return std::vector<uint8_t>(buf_.begin(), buf_.begin() + n); }

 public:
  Encoder(const Context& ctx, uint16_t width, uint16_t height)
      : ctx_(ctx), width_(width), height_(height), buf_(size_t(width) * height * 3 + 65536) {
    check(vp8gpu_encoder_create(ctx_.get(), &h_), ctx_.get(), "encoder_create");
  }
  // Encoder( const Decoder &, two_pass, quality ) (encoder.hh:350-351): continue the decoder's stream
  explicit Encoder(const Decoder& decoder)
      : ctx_(decoder.context()), width_(decoder.get_width()), height_(decoder.get_height()),
        buf_(size_t(width_) * height_ * 3 + 65536) {
    check(vp8gpu_encoder_create_from_decoder(ctx_.get(), decoder.handle(), &h_), ctx_.get(), "encoder_create_from_decoder");
  }
  // Encoder( width, height, two_pass, quality ) (encoder.hh:346-348)
  Encoder(const Context& ctx, uint16_t width, uint16_t height, bool two_pass, EncoderQuality quality)
      : Encoder(ctx, width, height) {
    set_two_pass(two_pass);
    set_quality(quality);
  }
  // Encoder( const Decoder &, two_pass, quality ) (encoder.hh:350-351)
  Encoder(const Decoder& decoder, bool two_pass, EncoderQuality quality) : Encoder(decoder) {
    set_two_pass(two_pass);
    set_quality(quality);
  }
  // Encoder( const Encoder & ) (encoder.cc:92-102)
  Encoder(const Encoder& o) : ctx_(o.ctx_), width_(o.width_), height_(o.height_), buf_(o.buf_.size()) {
    check(vp8gpu_encoder_clone(o.h_, &h_), ctx_.get(), "encoder_clone");
  }
  Encoder(Encoder&& o) noexcept : ctx_(o.ctx_), width_(o.width_), height_(o.height_), h_(o.h_), buf_(std::move(o.buf_)) {
    o.h_ = nullptr;
  }
  Encoder& operator=(Encoder o) {
    std::swap(h_, o.h_);
    std::swap(buf_, o.buf_);
    width_ = o.width_, height_ = o.height_;
    return *this;
  }
  ~Encoder() { vp8gpu_encoder_destroy(h_); }

  // export_decoder (encoder.hh:378): the Decoder a receiver holds after the frames emitted so far
  Decoder export_decoder() const {
    vp8gpu_decoder* d = nullptr;
    check(vp8gpu_encoder_export_decoder(h_, &d), ctx_.get(), "export_decoder");
    return Decoder(ctx_, d, width_, height_);
  }
  // Encoder( ..., two_pass, ... ) (encoder.hh:347-351): key frames get the trellis pass (encoder.cc:220-408)
  void set_two_pass(bool on) { check(vp8gpu_encoder_set_two_pass(h_, on), ctx_.get(), "set_two_pass"); }
  // Encoder( ..., quality ): only before the first frame is written (LogicError after)
  void set_quality(EncoderQuality quality) { check(vp8gpu_encoder_set_quality(h_, quality), ctx_.get(), "set_quality"); }
  // minihash (encoder.hh:382)
  uint32_t minihash() const {
    uint32_t m = 0;
    check(vp8gpu_encoder_minihash(h_, &m), ctx_.get(), "minihash");
    return m;
  }

  // encode_with_quantizer (encoder.cc:559-590)
  std::vector<uint8_t> encode_with_quantizer(const SourceFrame& f, uint8_t y_ac_qi) {
    size_t n = 0;
    check(vp8gpu_encoder_encode_with_quantizer(h_, f.y, f.y_stride, f.u, f.v, f.uv_stride, y_ac_qi, buf_.data(), buf_.size(), &n),
          ctx_.get(), "encode_with_quantizer");
    return take(n);
  }
  // encode_with_target_size (encoder.cc:592-629)
  std::vector<uint8_t> encode_with_target_size(const SourceFrame& f, size_t target_size) {
    size_t n = 0;
    check(vp8gpu_encoder_encode_with_target_size(h_, f.y, f.y_stride, f.u, f.v, f.uv_stride, target_size, buf_.data(),
                                                 buf_.size(), &n, nullptr),
          ctx_.get(), "encode_with_target_size");
    return take(n);
  }
  // estimate_frame_size (encoder.hh:376): exact size at this quantiser index, state untouched
  size_t estimate_frame_size(const SourceFrame& f, uint8_t y_ac_qi) {
    size_t n = 0;
    check(vp8gpu_encoder_estimate_frame_size(h_, f.y, f.y_stride, f.u, f.v, f.uv_stride, y_ac_qi, &n), ctx_.get(),
          "estimate_frame_size");
    return n;
  }
  // encode_with_minimum_ssim (encoder.cc:577-590)
  std::vector<uint8_t> encode_with_minimum_ssim(const SourceFrame& f, double minimum_ssim) {
    size_t n = 0;
    check(vp8gpu_encoder_encode_with_minimum_ssim(h_, f.y, f.y_stride, f.u, f.v, f.uv_stride, minimum_ssim, buf_.data(),
                                                  buf_.size(), &n, nullptr),
          ctx_.get(), "encode_with_minimum_ssim");
    return take(n);
  }
  // ---- re-encoding (encoder/reencode.cc; xc-enc --reencode, frontend/xc-enc.cc:262-327) ----
  // update_residues + write_frame (reencode.cc:131-313): y_ac_qi < 0 keeps the prediction frame's own index
  std::vector<uint8_t> update_residues(const SourceFrame& target, const ParsedFrame& prediction_frame, int y_ac_qi, bool last_frame) {
    size_t n = 0;
    check(vp8gpu_encoder_update_residues(h_, target.y, target.y_stride, target.u, target.v, target.uv_stride, prediction_frame.get(),
                                         y_ac_qi, last_frame, buf_.data(), buf_.size(), &n),
          ctx_.get(), "update_residues");
    return take(n);
  }
  // reencode_as_interframe + write_frame (reencode.cc:39-129)
  std::vector<uint8_t> reencode_as_interframe(const SourceFrame& target, const ParsedFrame& key_frame, uint8_t y_ac_qi) {
    size_t n = 0;
    check(vp8gpu_encoder_reencode_as_interframe(h_, target.y, target.y_stride, target.u, target.v, target.uv_stride, key_frame.get(),
                                                y_ac_qi, buf_.data(), buf_.size(), &n),
          ctx_.get(), "reencode_as_interframe");
    return take(n);
  }
  // write_frame( KeyFrame ) (encoder.cc:146-176): a key frame that is kept
  std::vector<uint8_t> write_frame(const ParsedFrame& key_frame) {
    size_t n = 0;
    check(vp8gpu_encoder_write_frame(h_, key_frame.get(), buf_.data(), buf_.size(), &n), ctx_.get(), "write_frame");
    return take(n);
  }
  // Encoder::reencode (reencode.cc:315-381), statement for statement; the emitted frames are returned instead of
  // appended to an IVFWriter.  prediction_frames were parsed with keep_labels by the prediction stream's decoder.
  std::vector<std::vector<uint8_t>> reencode(const std::vector<SourceFrame>& original_rasters,
                                             const std::vector<ParsedFrame>& prediction_frames, double kf_q_weight,
                                             bool extra_frame_chunk) {
    if (original_rasters.empty()) throw std::runtime_error("no rasters to re-encode");
    if (original_rasters.size() != prediction_frames.size()) throw std::runtime_error("prediction/original_rasters mismatch");
    std::vector<std::vector<uint8_t>> out;
    const size_t start = extra_frame_chunk ? 1 : 0;
    auto qi_of = [](const ParsedFrame& f) {
      const int q = f.y_ac_qi();
      if (q < 0) throw LogicError("reencode: prediction frames must be parsed with keep_labels");
      return q;
    };
    for (size_t i = start; i < original_rasters.size(); i++) {
      const SourceFrame& target = original_rasters[i];
      const ParsedFrame& pred = prediction_frames[i];
      const bool last = i == prediction_frames.size() - 1;
      if (i == start && pred.key_frame()) {  // option 1: an initial key frame becomes an inter frame
        int qi = qi_of(pred);
        if (i + 1 < prediction_frames.size() && !prediction_frames[i + 1].key_frame())
          qi = (int)lrint(kf_q_weight * qi_of(pred) + (1 - kf_q_weight) * qi_of(prediction_frames[i + 1]));
        out.push_back(reencode_as_interframe(target, pred, (uint8_t)qi));
      } else if (i == start && extra_frame_chunk) {  // option 2: first inter frame of an extra-frame chunk
        if (!prediction_frames[0].key_frame()) throw std::runtime_error("extra-frame chunks must start with a keyframe.");
        const int qi = (int)lrint(kf_q_weight * qi_of(prediction_frames[0]) + (1 - kf_q_weight) * qi_of(pred));
        out.push_back(update_residues(target, pred, qi, last));
      } else if (pred.key_frame()) {  // option 3: another key frame is preserved
        out.push_back(write_frame(pred));
      } else {  // option 4
        out.push_back(update_residues(target, pred, -1, last));
      }
    }
    return out;
  }

  // EncoderStats::ssim of the last frame (encoder.hh:118-127)
  double last_ssim() const {
    double q = -1.0;
    vp8gpu_encoder_stats(h_, &q, nullptr, nullptr);
    return q;
  }
  // the LAST reference of export_decoder() (encoder.hh:378)
  RasterHandle reconstruction() const {
    vp8gpu_frame_id id = -1;
    check(vp8gpu_encoder_reconstruction(h_, &id), ctx_.get(), "reconstruction");
    return RasterHandle(ctx_, id);
  }
};

}  // namespace alfalfa_gpu
