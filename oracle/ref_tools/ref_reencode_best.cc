/* ref_reencode_best -- TEST INFRASTRUCTURE.  ref_reencode (ref_tools/ref_reencode.cc, same usage) with the reference
 * Encoder built at BEST_QUALITY (encoder/encoder.hh:56-60), the setting "xc-enc --reencode" runs by default, instead of
 * REALTIME_QUALITY: the reference's headers are read first, then the enumerator name ref_reencode.cc passes to the
 * Encoder is redirected to BEST_QUALITY. */
#include "decoder.hh"
#include "enc_state_serializer.hh"
#include "encoder.hh"
#include "ivf.hh"
#include "ivf_writer.hh"
#include "uncompressed_chunk.hh"

#define REALTIME_QUALITY BEST_QUALITY
#include "ref_reencode.cc"
