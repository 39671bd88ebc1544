"""Host-side mirror of the reference's decoder interface (src/decoder/decoder.hh:244-300,
player.hh:40-97) for Python callers (tests, bench).  Same names and meaning as the reference:

    Decoder(ctx)                      Decoder(width, height)
    Decoder.parse_frame(chunk)        Decoder::parse_frame<FrameType>  -> ParsedFrame
    Decoder.decode_frame(parsed)      Decoder::decode_frame            -> (shown, RasterHandle)
    Decoder.get_frame_output(chunk)   Decoder::get_frame_output        -> (shown, RasterHandle)
    Decoder.parse_and_decode_frame    -> RasterHandle or None (hidden frame)
    Decoder.get_state / get_references / copy() / ==
    FilePlayer(ctx, ivf_bytes).advance() / eof()

Errors are raised as Invalid / Unsupported / LogicError like the reference's exception classes.
Every call goes through the C ABI in libvpx8gpu.so; nothing here computes pixels.
"""
import ctypes as C
import struct

import numpy as np

from . import capi
from .capi import check


class Context:
    """vp8gpu_ctx: one CUDA device + one frame size (per-context raster pool)."""

    def __init__(self, width, height, device=0, max_frames=0):
        self.L = capi.lib()
        self.width, self.height = width, height
        self.mb_cols, self.mb_rows = (width + 15) // 16, (height + 15) // 16
        self.h = C.c_void_p()
        check(self.L.vp8gpu_ctx_create(device, width, height, max_frames, C.byref(self.h)), None,
              "vp8gpu_ctx_create (is a CUDA device present?)")

    def close(self):
        if self.h:
            self.L.vp8gpu_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def display_bytes(self):
        return self.width * self.height + 2 * ((self.width + 1) // 2) * ((self.height + 1) // 2)

    def sync(self):
        check(self.L.vp8gpu_ctx_sync(self.h), self.h, "sync")

    @property
    def frame_bytes(self):
        return int(self.L.vp8gpu_frame_bytes(self.h))

    def set_device_tokens(self, on):
        """VP8GPU_OPT_DEVICE_TOKENS: decode_ivf decodes the DCT partitions on the device (default on)"""
        check(self.L.vp8gpu_ctx_set_option(self.h, capi.OPT_DEVICE_TOKENS, int(bool(on))), self.h, "set_option")

    def launch_count(self):
        return int(self.L.vp8gpu_launch_count(self.h))

    def alloc_frame(self):
        fid = C.c_int32(-1)
        check(self.L.vp8gpu_frame_alloc(self.h, C.byref(fid)), self.h, "frame_alloc")
        return RasterHandle(self, fid.value)


class RasterHandle:
    """RasterHandle (decoder/raster_handle.hh:95-123): a ref-counted device raster."""

    def __init__(self, ctx, fid):
        self.ctx, self.id = ctx, fid

    def release(self):
        if self.id is not None and self.ctx.h:
            self.ctx.L.vp8gpu_frame_release(self.ctx.h, self.id)
        self.id = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    def planes(self):
        """MB-aligned planes (Y, U, V) as numpy arrays (blocks until the frame is decoded)."""
        c = self.ctx
        W, H = 16 * c.mb_cols, 16 * c.mb_rows
        y = np.empty((H, W), np.uint8)
        u = np.empty((H // 2, W // 2), np.uint8)
        v = np.empty((H // 2, W // 2), np.uint8)
        check(c.L.vp8gpu_frame_download(c.h, self.id, y.ctypes.data, W, u.ctypes.data, v.ctypes.data, W // 2), c.h,
              "frame_download")
        return y, u, v

    def ssim(self, other):
        """BaseRaster::quality: luma SSIM against another raster of the same context"""
        q = C.c_double(0)
        check(self.ctx.L.vp8gpu_frame_ssim(self.ctx.h, self.id, other.id, C.byref(q)), self.ctx.h, "frame_ssim")
        return q.value

    def export_to(self, ptr, nbytes):
        """whole raster (ctx.frame_bytes, pitched planes) into a host or same-device buffer"""
        check(self.ctx.L.vp8gpu_frame_export(self.ctx.h, self.id, ptr, nbytes), self.ctx.h, "frame_export")

    def import_from(self, ptr, nbytes):
        check(self.ctx.L.vp8gpu_frame_import(self.ctx.h, self.id, ptr, nbytes), self.ctx.h, "frame_import")

    def upload(self, y, u, v):
        c = self.ctx
        y, u, v = (np.ascontiguousarray(a, dtype=np.uint8) for a in (y, u, v))
        check(c.L.vp8gpu_frame_upload(c.h, self.id, y.ctypes.data, y.shape[1], u.ctypes.data, v.ctypes.data,
                                      u.shape[1]), c.h, "frame_upload")

    def hash(self):
        """RasterHandle::hash(): 64-bit content hash computed on the device"""
        c = self.ctx
        h = C.c_uint64(0)
        check(c.L.vp8gpu_frame_hash(c.h, self.id, C.byref(h)), c.h, "frame_hash")
        return int(h.value)

    def display_bytes(self):
        """BaseRaster::dump (util/raster.cc:85-114)"""
        c = self.ctx
        buf = np.empty(c.display_bytes, np.uint8)
        check(c.L.vp8gpu_frame_download_display(c.h, self.id, buf.ctypes.data, buf.size), c.h, "download_display")
        return buf.tobytes()


class DecoderState:
    """DecoderState (decoder.hh:190-225) handle."""

    def __init__(self, width=None, height=None, _h=None, _owned=True):
        self.L = capi.lib()
        self._owned = _owned
        if _h is not None:
            self.h = _h
        else:
            self.h = C.c_void_p()
            check(self.L.vp8gpu_state_create(width, height, C.byref(self.h)))

    def clone(self):
        h = C.c_void_p()
        check(self.L.vp8gpu_state_clone(self.h, C.byref(h)))
        return DecoderState(_h=h)

    def __eq__(self, other):
        return bool(self.L.vp8gpu_state_equal(self.h, other.h))

    def hash(self):
        return int(self.L.vp8gpu_state_hash(self.h))

    def serialize(self):
        """DecoderState::serialize (decoder.cc:283-314): the reference's DECODER_STATE record"""
        n = self.L.vp8gpu_state_serialize(self.h, None, 0)
        buf = (C.c_uint8 * n)()
        assert self.L.vp8gpu_state_serialize(self.h, buf, n) == n
        return bytes(buf)

    @staticmethod
    def deserialize(blob):
        h = C.c_void_p()
        check(capi.lib().vp8gpu_state_deserialize(blob, len(blob), C.byref(h)), None, "state_deserialize")
        return DecoderState(_h=h)

    def __del__(self):
        try:
            if self._owned and self.h:
                self.L.vp8gpu_state_destroy(self.h)
        except Exception:
            pass


class ParsedFrame:
    """KeyFrame / InterFrame (frame.hh:126-127) in the flat form of include/vp8gpu.h."""

    def __init__(self):
        self.L = capi.lib()
        self.h = C.c_void_p()
        check(self.L.vp8gpu_parsed_create(C.byref(self.h)))

    def __del__(self):
        try:
            self.L.vp8gpu_parsed_destroy(self.h)
        except Exception:
            pass

    @property
    def desc(self):
        return self.L.vp8gpu_parsed_desc(self.h).contents

    def arrays(self):
        """copies of (mbs, tokens, split)"""
        d = self.desc
        n = d.mb_cols * d.mb_rows
        mbs = np.frombuffer(C.string_at(self.L.vp8gpu_parsed_mbs(self.h), n * 32), dtype=capi.MB_DTYPE).copy()
        tok = (np.frombuffer(C.string_at(self.L.vp8gpu_parsed_tokens(self.h), d.n_tokens * 4), dtype="<u4").copy()
               if d.n_tokens else np.zeros(0, "<u4"))
        sp = (np.frombuffer(C.string_at(self.L.vp8gpu_parsed_split(self.h), d.n_split * 64), dtype="<i2").copy()
              .reshape(-1, 16, 2) if d.n_split else np.zeros((0, 16, 2), "<i2"))
        return mbs, tok, sp


class Decoder:
    """Decoder (decoder.hh:244-300): DecoderState + References with explicit state passing."""

    def __init__(self, ctx, _h=None):
        self.ctx, self.L = ctx, ctx.L
        if _h is not None:
            self.h = _h
        else:
            self.h = C.c_void_p()
            check(self.L.vp8gpu_decoder_create(ctx.h, C.byref(self.h)), ctx.h, "decoder_create")

    def __del__(self):
        try:
            if self.h and self.ctx.h:
                self.L.vp8gpu_decoder_destroy(self.h)
        except Exception:
            pass

    @staticmethod
    def from_state(ctx, state, refs):
        """Decoder(DecoderState, References) (decoder.hh:254); refs = (last, golden, alternative) RasterHandles"""
        ids = (C.c_int32 * 3)(*[r.id for r in refs])
        h = C.c_void_p()
        check(ctx.L.vp8gpu_decoder_create_from(ctx.h, state.h, ids, C.byref(h)), ctx.h, "decoder_create_from")
        return Decoder(ctx, h)

    def copy(self):
        """copy construction: O(1) in pixels, shares the reference rasters"""
        h = C.c_void_p()
        check(self.L.vp8gpu_decoder_clone(self.h, C.byref(h)), self.ctx.h, "decoder_clone")
        return Decoder(self.ctx, h)

    def serialize(self):
        """Decoder::serialize (decoder.cc:54-69): the reference's tag-length-value blob (state + LAST raster)"""
        size = C.c_size_t(0)
        self.L.vp8gpu_decoder_serialize(self.h, None, 0, C.byref(size))
        buf = (C.c_uint8 * size.value)()
        check(self.L.vp8gpu_decoder_serialize(self.h, buf, size.value, C.byref(size)), self.ctx.h, "decoder_serialize")
        return bytes(buf)

    @staticmethod
    def deserialize(ctx, blob):
        """Decoder::deserialize (decoder.cc:71-81); golden = alternative = last as in the reference"""
        h = C.c_void_p()
        check(ctx.L.vp8gpu_decoder_deserialize(ctx.h, blob, len(blob), C.byref(h)), ctx.h, "decoder_deserialize")
        return Decoder(ctx, h)

    def get_state(self):
        return DecoderState(_h=C.c_void_p(self.L.vp8gpu_decoder_state(self.h)), _owned=False).clone()

    def get_references(self):
        """(last, golden, alternative) as new RasterHandles"""
        ids = (C.c_int32 * 3)()
        self.L.vp8gpu_decoder_references(self.h, ids)
        out = []
        for i in ids:
            check(self.L.vp8gpu_frame_retain(self.ctx.h, i), self.ctx.h, "retain")
            out.append(RasterHandle(self.ctx, i))
        return tuple(out)

    def parse_frame(self, chunk, keep_labels=False):
        """Decoder::decompress_frame + parse_frame: updates the decoder's state.  keep_labels: keep the header as coded
        and every ambiguous label, like the reference's Frame object does (needed by ParsedFrame re-serialisation
        and by Encoder.reencode)"""
        p = ParsedFrame()
        if keep_labels:
            check(self.L.vp8gpu_parsed_keep_labels(p.h, 1), self.ctx.h, "keep_labels")
        st = C.c_void_p(self.L.vp8gpu_decoder_state(self.h))
        check(self.L.vp8gpu_parse_frame(st, chunk, len(chunk), p.h), self.ctx.h, "parse_frame")
        return p

    def parse_frame_device(self, chunk):
        """parse_frame with the DCT partitions decoded on the device (same records)"""
        p = ParsedFrame()
        st = C.c_void_p(self.L.vp8gpu_decoder_state(self.h))
        check(self.L.vp8gpu_parse_frame_device(self.ctx.h, st, chunk, len(chunk), p.h), self.ctx.h, "parse_frame_device")
        return p

    def set_device_tokens(self, on):
        """get_frame_output leaves the DCT partitions to the device (same output)"""
        check(self.L.vp8gpu_decoder_set_device_tokens(self.h, int(bool(on))), self.ctx.h, "set_device_tokens")

    def decode_frame(self, parsed):
        shown, fid = C.c_int(0), C.c_int32(-1)
        check(self.L.vp8gpu_decoder_decode_parsed(self.h, parsed.h, C.byref(shown), C.byref(fid)), self.ctx.h,
              "decode_frame")
        return bool(shown.value), RasterHandle(self.ctx, fid.value)

    def get_frame_output(self, chunk):
        shown, fid = C.c_int(0), C.c_int32(-1)
        check(self.L.vp8gpu_decoder_decode(self.h, chunk, len(chunk), C.byref(shown), C.byref(fid)), self.ctx.h,
              "get_frame_output")
        return bool(shown.value), RasterHandle(self.ctx, fid.value)

    def parse_and_decode_frame(self, chunk):
        shown, raster = self.get_frame_output(chunk)
        return raster if shown else None

    def get_hash(self):
        """Decoder::get_hash: state + the three reference rasters"""
        out = C.c_uint64(0)
        check(self.L.vp8gpu_decoder_hash(self.h, C.byref(out)), self.ctx.h, "decoder_hash")
        return out.value

    def minihash(self):
        h = self.get_hash()
        return (h ^ (h >> 32)) & 0xFFFFFFFF

    def __eq__(self, other):
        eq = C.c_int(0)
        check(self.L.vp8gpu_decoder_equal(self.h, other.h, C.byref(eq)), self.ctx.h, "decoder_equal")
        return bool(eq.value)


def read_ivf(data):
    """util/ivf.cc:36-82 -> (width, height, [frames])"""
    if data[:4] != b"DKIF":
        raise capi.Invalid(capi.ERR_INVALID, "missing IVF file header")
    w, h = struct.unpack_from("<HH", data, 12)
    n = struct.unpack_from("<I", data, 24)[0]
    frames, pos = [], 32
    for _ in range(n):
        if pos + 12 > len(data):
            raise capi.Invalid(capi.ERR_INVALID, "IVF file truncated")
        flen = struct.unpack_from("<I", data, pos)[0]
        frames.append(bytes(data[pos + 12:pos + 12 + flen]))
        pos += 12 + flen
    return w, h, frames


def ivf_expected_decoder_minihash(data):
    """IVF::expected_decoder_minihash (util/ivf.cc:46): header bytes 28..31"""
    if len(data) < 32 or data[:4] != b"DKIF":
        raise capi.Invalid(capi.ERR_INVALID, "missing IVF file header")
    return struct.unpack_from("<I", data, 28)[0]


class FilePlayer:
    """FilePlayer (player.cc:88-143): starts at the first key frame, advance() skips hidden frames."""

    def __init__(self, ctx, ivf_bytes):
        w, h, self.frames = read_ivf(ivf_bytes)
        if (w, h) != (ctx.width, ctx.height):
            raise capi.Unsupported(capi.ERR_UNSUPPORTED, "IVF size does not match the context")
        self.decoder = Decoder(ctx)
        self.frame_no = 0
        while self.frame_no < len(self.frames) and (self.frames[self.frame_no][0] & 1):
            self.frame_no += 1

    def eof(self):
        return self.frame_no == len(self.frames)

    def advance(self):
        while not self.eof():
            r = self.decoder.parse_and_decode_frame(self.frames[self.frame_no])
            self.frame_no += 1
            if r is not None:
                return r
        raise capi.Unsupported(capi.ERR_UNSUPPORTED, "hidden frames at end of file")


def decode_ivf(ctx, ivf_bytes, threads=1, want_output=True):
    """Whole-stream decode through vp8gpu_decode_ivf (GOP-parallel host workers).
    Returns (display bytes of all shown frames or None, n_decoded, n_shown)."""
    L = ctx.L
    _, _, frames = read_ivf(ivf_bytes)
    start = 0
    while start < len(frames) and (frames[start][0] & 1):
        start += 1
    n_shown_guess = sum(1 for f in frames[start:] if len(f) and (f[0] >> 4) & 1)
    size = n_shown_guess * ctx.display_bytes
    dst = None
    ptr = C.c_void_p()
    if want_output and size:
        check(L.vp8gpu_host_alloc(C.byref(ptr), size), ctx.h, "host_alloc")
    nd, ns = C.c_uint32(0), C.c_uint32(0)
    try:
        check(L.vp8gpu_decode_ivf(ctx.h, ivf_bytes, len(ivf_bytes), threads, ptr, size if ptr else 0, C.byref(nd),
                                  C.byref(ns)), ctx.h, "decode_ivf")
        check(L.vp8gpu_ctx_sync(ctx.h), ctx.h, "sync")
        if ptr:
            dst = C.string_at(ptr, ns.value * ctx.display_bytes)
    finally:
        if ptr:
            L.vp8gpu_host_free(ptr)
    return dst, nd.value, ns.value


class Encoder:
    """Encoder (encoder/encoder.hh:345-382): a copyable value like the reference's.  Source frames are
    display-size (Y, U, V) numpy planes; the result is one compressed VP8 frame.  quality: "realtime" (Salsify's
    setting, the default) or "best" (ExCamera's xc-enc default), see set_quality."""

    def __init__(self, ctx, _h=None, quality="realtime"):
        self.ctx, self.L = ctx, ctx.L
        self.h = C.c_void_p()
        if _h is not None:
            self.h = _h
        else:
            check(self.L.vp8gpu_encoder_create(ctx.h, C.byref(self.h)), ctx.h, "encoder_create")
        self._out = np.empty(ctx.width * ctx.height * 3 + (1 << 16), np.uint8)
        if _h is None and quality != "realtime":
            self.set_quality(quality)

    def copy(self):
        """Encoder( const Encoder & ) (encoder.cc:92-102): O(1) in pixels, shares the reference rasters"""
        h = C.c_void_p()
        check(self.L.vp8gpu_encoder_clone(self.h, C.byref(h)), self.ctx.h, "encoder_clone")
        return Encoder(self.ctx, _h=h)

    @staticmethod
    def from_decoder(ctx, decoder, quality="realtime"):
        """Encoder( const Decoder &, two_pass, quality ) (encoder.hh:350-351)"""
        h = C.c_void_p()
        check(ctx.L.vp8gpu_encoder_create_from_decoder(ctx.h, decoder.h, C.byref(h)), ctx.h, "encoder_create_from_decoder")
        enc = Encoder(ctx, _h=h)
        if quality != "realtime":
            enc.set_quality(quality)
        return enc

    def export_decoder(self):
        """Encoder::export_decoder (encoder.hh:378)"""
        h = C.c_void_p()
        check(self.L.vp8gpu_encoder_export_decoder(self.h, C.byref(h)), self.ctx.h, "encoder_export_decoder")
        return Decoder(self.ctx, _h=h)

    def set_two_pass(self, on):
        """Encoder( ..., two_pass, ... ): key frames get the trellis pass (encoder.cc:220-408)"""
        check(self.L.vp8gpu_encoder_set_two_pass(self.h, int(bool(on))), self.ctx.h, "encoder_set_two_pass")

    def set_quality(self, quality):
        """Encoder( ..., quality ) (encoder.hh:56-60): "best" tries B_PRED and searches a new motion vector at every
        inter-frame macroblock and starts every quantiser and loop-filter search from scratch; "realtime" does
        neither.  LogicError once the encoder has written a frame."""
        codes = {"best": capi.QUALITY_BEST, "realtime": capi.QUALITY_REALTIME}
        if quality not in codes:
            raise capi.LogicError(capi.ERR_LOGIC, "set_quality: %r is neither 'best' nor 'realtime'" % (quality,))
        check(self.L.vp8gpu_encoder_set_quality(self.h, codes[quality]), self.ctx.h, "encoder_set_quality")

    def set_writer(self, mode):
        """0: bitstream byte-identical to the reference encoder's (default); 1: compact writer, 8 partitions"""
        check(self.L.vp8gpu_encoder_set_writer(self.h, int(mode)), self.ctx.h, "encoder_set_writer")

    def minihash(self):
        out = C.c_uint32(0)
        check(self.L.vp8gpu_encoder_minihash(self.h, C.byref(out)), self.ctx.h, "encoder_minihash")
        return out.value

    def __del__(self):
        try:
            if self.h and self.ctx.h:
                self.L.vp8gpu_encoder_destroy(self.h)
        except Exception:
            pass

    def _planes(self, y, u, v):
        return tuple(np.ascontiguousarray(a, dtype=np.uint8) for a in (y, u, v))

    def encode_with_quantizer(self, y, u, v, y_ac_qi):
        y, u, v = self._planes(y, u, v)
        size = C.c_size_t(0)
        check(self.L.vp8gpu_encoder_encode_with_quantizer(self.h, y.ctypes.data, y.shape[1], u.ctypes.data, v.ctypes.data,
                                                          u.shape[1], y_ac_qi, self._out.ctypes.data, self._out.size,
                                                          C.byref(size)), self.ctx.h, "encode_with_quantizer")
        return self._out[:size.value].tobytes()

    def encode_with_target_size(self, y, u, v, target_size):
        y, u, v = self._planes(y, u, v)
        size, qi = C.c_size_t(0), C.c_int(0)
        check(self.L.vp8gpu_encoder_encode_with_target_size(self.h, y.ctypes.data, y.shape[1], u.ctypes.data, v.ctypes.data,
                                                            u.shape[1], target_size, self._out.ctypes.data, self._out.size,
                                                            C.byref(size), C.byref(qi)), self.ctx.h, "encode_with_target_size")
        return self._out[:size.value].tobytes(), qi.value

    def encode_with_minimum_ssim(self, y, u, v, minimum_ssim):
        """Encoder::encode_with_minimum_ssim (encoder.cc:577-590) -> (frame bytes, chosen y_ac_qi)"""
        y, u, v = self._planes(y, u, v)
        size, qi = C.c_size_t(0), C.c_int(0)
        check(self.L.vp8gpu_encoder_encode_with_minimum_ssim(self.h, y.ctypes.data, y.shape[1], u.ctypes.data, v.ctypes.data,
                                                             u.shape[1], float(minimum_ssim), self._out.ctypes.data,
                                                             self._out.size, C.byref(size), C.byref(qi)), self.ctx.h,
              "encode_with_minimum_ssim")
        return self._out[:size.value].tobytes(), qi.value

    def estimate_frame_size(self, y, u, v, y_ac_qi):
        """Encoder::estimate_frame_size: bytes at this quantiser index, without committing the frame"""
        y, u, v = self._planes(y, u, v)
        size = C.c_size_t(0)
        check(self.L.vp8gpu_encoder_estimate_frame_size(self.h, y.ctypes.data, y.shape[1], u.ctypes.data, v.ctypes.data,
                                                        u.shape[1], y_ac_qi, C.byref(size)), self.ctx.h, "estimate_frame_size")
        return size.value

    def update_residues(self, y, u, v, prediction_frame, y_ac_qi=-1, last_frame=False):
        """Encoder::update_residues + write_frame (encoder/reencode.cc:131-313): keep the prediction frame's modes
        and vectors, recompute its residues against this encoder's references towards the target planes"""
        y, u, v = self._planes(y, u, v)
        size = C.c_size_t(0)
        check(self.L.vp8gpu_encoder_update_residues(self.h, y.ctypes.data, y.shape[1], u.ctypes.data, v.ctypes.data, u.shape[1],
                                                    prediction_frame.h, int(y_ac_qi), int(bool(last_frame)), self._out.ctypes.data,
                                                    self._out.size, C.byref(size)), self.ctx.h, "update_residues")
        return self._out[:size.value].tobytes()

    def write_frame(self, frame):
        """Encoder::write_frame( KeyFrame ) (encoder.cc:146-176): emit a parsed key frame unchanged, move past it"""
        size = C.c_size_t(0)
        check(self.L.vp8gpu_encoder_write_frame(self.h, frame.h, self._out.ctypes.data, self._out.size, C.byref(size)), self.ctx.h,
              "write_frame")
        return self._out[:size.value].tobytes()

    def reencode(self, original_rasters, prediction_frames, kf_q_weight=1.0, extra_frame_chunk=False):
        """Encoder::reencode (encoder/reencode.cc:315-381), statement for statement.  original_rasters: (y, u, v)
        planes per frame; prediction_frames: ParsedFrame per frame, parsed with keep_labels by the prediction
        stream's own decoder state.  Returns the list of emitted frames (what the reference appends to its IVFWriter)."""
        if not original_rasters:
            raise RuntimeError("no rasters to re-encode")
        if len(original_rasters) != len(prediction_frames):
            raise RuntimeError("prediction/original_rasters mismatch")
        out = []
        start = 1 if extra_frame_chunk else 0

        def qi_of(f):
            q = self.L.vp8gpu_parsed_y_ac_qi(f.h)
            if q < 0:
                raise capi.LogicError(capi.ERR_LOGIC, "reencode: prediction frames must be parsed with keep_labels")
            return q

        def lrint(x):  # round half to even, like lrint in the default rounding mode
            return int(round(x))

        for i in range(start, len(original_rasters)):
            y, u, v = original_rasters[i]
            pred = prediction_frames[i]
            last = i == len(prediction_frames) - 1
            is_key = bool(pred.desc.key_frame)
            if i == start and is_key:
                # option 1: an initial key frame becomes an inter frame (reencode_as_interframe, reencode.cc:39-129)
                qi = qi_of(pred)
                if i + 1 < len(prediction_frames) and not prediction_frames[i + 1].desc.key_frame:
                    qi = lrint(kf_q_weight * qi_of(pred) + (1 - kf_q_weight) * qi_of(prediction_frames[i + 1]))
                out.append(self.reencode_as_interframe(y, u, v, pred, qi))
            elif i == start and extra_frame_chunk:
                # option 2: first inter frame of an extra-frame chunk: blend in the key frame's quantiser
                if not prediction_frames[0].desc.key_frame:
                    raise RuntimeError("extra-frame chunks must start with a keyframe.")
                qi = lrint(kf_q_weight * qi_of(prediction_frames[0]) + (1 - kf_q_weight) * qi_of(pred))
                out.append(self.update_residues(y, u, v, pred, qi, last))
            elif is_key:
                out.append(self.write_frame(pred))      # option 3: another key frame is preserved
            else:
                out.append(self.update_residues(y, u, v, pred, -1, last))  # option 4
        return out

    def reencode_as_interframe(self, y, u, v, key_frame, y_ac_qi):
        """Encoder::reencode_as_interframe (encoder/reencode.cc:39-129)"""
        y, u, v = self._planes(y, u, v)
        size = C.c_size_t(0)
        check(self.L.vp8gpu_encoder_reencode_as_interframe(self.h, y.ctypes.data, y.shape[1], u.ctypes.data, v.ctypes.data, u.shape[1],
                                                           key_frame.h, int(y_ac_qi), self._out.ctypes.data, self._out.size,
                                                           C.byref(size)), self.ctx.h, "reencode_as_interframe")
        return self._out[:size.value].tobytes()

    TIMELINE = ("upload", "estimates_launch", "estimates_walk", "full_pass", "loop_filter_search", "writer", "state_update", "total")

    def timeline(self):
        """vp8gpu_encoder_timeline: milliseconds per phase of the last encode call (diagnostic)"""
        ms = (C.c_double * 8)()
        check(self.L.vp8gpu_encoder_timeline(self.h, ms, 8), self.ctx.h, "encoder_timeline")
        return dict(zip(self.TIMELINE, (float(x) for x in ms)))

    def stats(self):
        """EncoderStats of the last frame: dict(ssim, loop_filter_level, y_ac_qi)"""
        q, lf, qi = C.c_double(0), C.c_int(0), C.c_int(0)
        check(self.L.vp8gpu_encoder_stats(self.h, C.byref(q), C.byref(lf), C.byref(qi)), self.ctx.h, "encoder_stats")
        return {"ssim": q.value, "loop_filter_level": lf.value, "y_ac_qi": qi.value}

    def reconstruction(self):
        """the encoder's LAST reference (what a decoder holds after decoding the frame just emitted)"""
        fid = C.c_int32(-1)
        check(self.L.vp8gpu_encoder_reconstruction(self.h, C.byref(fid)), self.ctx.h, "encoder_reconstruction")
        return RasterHandle(self.ctx, fid.value)


def write_ivf(width, height, frames, expected_decoder_minihash=0):
    """util/ivf_writer.cc: 32-byte DKIF header + 12-byte frame headers.  Header bytes 28..31 carry ExCamera's
    expected decoder entry minihash (IVFWriter::set_expected_decoder_entry_hash, ivf_writer.cc:92-99): the
    minihash of the Decoder a chunk must be played into; 0 = not set."""
    out = bytearray(b"DKIF" + struct.pack("<HH4sHHIIII", 0, 32, b"VP80", width, height, 30, 1, len(frames),
                                          expected_decoder_minihash & 0xFFFFFFFF))
    for i, f in enumerate(frames):
        out += struct.pack("<IQ", len(f), i) + f
    return bytes(out)
