/* ref_encode_best -- TEST INFRASTRUCTURE.  ref_encode (ref_tools/ref_encode.cc, same usage and environment) with the
 * reference Encoder built at BEST_QUALITY (encoder/encoder.hh:56-60), ExCamera's xc-enc default, instead of
 * REALTIME_QUALITY.  The reference's headers are read first, as ref_encode.cc reads them (private members lifted for its
 * diagnostics); after that the enumerator name ref_encode.cc passes to the Encoder is redirected to BEST_QUALITY. */
#include <array>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <fstream>
#include <iostream>
#include <memory>
#include <sstream>
#include <string>
#include <vector>
#define private public
#define protected public
#include <chrono>
#include <cstdio>
#include <random>

#include "encoder.hh"
#include "ivf_writer.hh"

#define REALTIME_QUALITY BEST_QUALITY
#include "ref_encode.cc"
