// common.cuh — constants and lane-layout types shared by every sm_100a translation unit of the engine.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/bsched.h"

namespace bsk {

constexpr int LANE_CPU = 0, LANE_MEM = 1, LANE_EPH = 2, LANE_PODS = 3;
// Sentinels for lanes without a map key.  With |table values| <= BS_VALUE_LIMIT = 2^56,
// |left| <= 2^57 and every real left-req difference is below 2^58 in magnitude, while any
// difference involving a sentinel is >= 2^61 - 2^57 and < 2^63: it never overflows, never
// fails the >= 0 test, and never wins the min -> score = min over lanes present on BOTH sides.
constexpr int64_t ABSENT_LEFT = (int64_t)1 << 61;      // left lane without a map key: never limits
constexpr int64_t UNCHECKED_REQ = -((int64_t)1 << 61); // request lane without a map key: never checked
// Narrow lanes: a lane whose every |left| and |req| is <= 2^27 (millicores, pod counts, GPUs ...)
// is evaluated in int32: |real diff| < 2^27 < any diff involving a 32-bit sentinel (>= 2^29-2^26),
// and 2^29 - (-2^29) does not overflow.  The narrow set always contains a fixed lane (always a
// real value), so the 32-bit min is always a real difference and widens by sign extension.
constexpr int32_t ABSENT_LEFT32 = 1 << 29;
constexpr int32_t UNCHECKED_REQ32 = -(1 << 29);
// |v| <= 2^26 - 1 on both sides: every real narrow difference is < 2^27, so a fitting pair's score fits 27 bits
// and (score << KEY_BITS) + j stays below 2^31 (the best-node key of the fit kernel)
constexpr int FIT_CAP_LOG2 = 27;
constexpr int64_t NARROW_LIMIT = ((int64_t)1 << (FIT_CAP_LOG2 - 1)) - 1;
// Scaled lanes (round 2): a byte-valued lane whose every `left` and `req` is a multiple of 2^k
// (k = the lane's common trailing zeros, found at upload) and fits |v| >> k <= 2^29 is carried in
// units of 2^k as int32 — EXACT: (left - req) >= 0  <=>  (left>>k) - (req>>k) >= 0, and the
// difference in original units is (left>>k - req>>k) << k.  A fitting pair's score is <= the
// narrow-lane minimum t < 2^27, so a scaled difference only matters below 2^27: the kernel clamps
// it to C = 2^(27-k) (k <= 27; else 1) before shifting back by min(k, 27), i.e. it contributes either its
// exact value or 2^27 ("not the minimum").  Sentinels +-(2^30 - 1): no int32 overflow against 2^29.
constexpr int32_t ABSENT_LEFTS = (1 << 30) - 1;
constexpr int32_t UNCHECKED_REQS = -((1 << 30) - 1);
constexpr int64_t SCALED_LIMIT = (int64_t)1 << 29;
struct LaneMap {
  uint8_t wide[BS_MAX_LANES];    // original lane index of wide slot k   (k < LW)
  uint8_t narrow[BS_MAX_LANES];  // original lane index of narrow slot k (k < LN)
  uint8_t scaled[BS_MAX_LANES];  // original lane index of scaled slot k (k < LS)
  uint8_t sunit[BS_MAX_LANES];   // k: the slot's unit is 2^k
  uint8_t sshift[BS_MAX_LANES];  // min(k, 28): shift back to original units after the clamp
  uint32_t sclamp[BS_MAX_LANES]; // C = 2^(28-k), or 1 when k > 28
  uint32_t LW, LN, LS;
};
constexpr int NODE_TILE = 512;                          // nodes per shared-memory tile
constexpr int FIT_WARPS = 8;                            // consumer warps (each sweeps PODS_PER_WARP pods)
constexpr int FIT_THREADS = (FIT_WARPS + 1) * 32;       // + one producer warp that only drives the TMA ring
constexpr int PODS_PER_WARP = 4;                        // pods evaluated together per node (ILP)
constexpr int PODS_PER_CTA = FIT_WARPS * PODS_PER_WARP; // 32
constexpr int TILE_WORDS = NODE_TILE / 32;              // ballot words per tile and pod
static_assert(TILE_WORDS <= 32 && 32 % TILE_WORDS == 0, "a 32-word bitmap line is a whole number of tiles");
constexpr int TILES_PER_LINE = 32 / TILE_WORDS;         // tiles whose ballot words fill one 128-byte bitmap line
constexpr int KEY_BITS = 4;                             // log2(TILE_WORDS): score (27 bits) + word index fit 31 bits
static_assert(TILE_WORDS == 1 << KEY_BITS, "best-node key: KEY_BITS is log2(TILE_WORDS)");
constexpr int FIT_STAGES = 2;                           // TMA ring depth (full/empty mbarrier pairs)
// class bits of the TILE_WORDS nodes a lane owns in one tile
using ColBits = uint16_t;
static_assert(sizeof(ColBits) * 8 == TILE_WORDS, "ColBits holds one bit per node a lane owns in a tile");

}  // namespace bsk
