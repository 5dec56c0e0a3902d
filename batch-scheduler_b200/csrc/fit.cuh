// fit.cuh — gang_fit_kernel, the dominant kernel of a round (templates only: instantiated slice by
// slice in fit_inst.cu so that the variants compile in parallel; engine.cu reaches them through
// fit_lookup()).
#pragma once
#include "common.cuh"

namespace bsk {

// ---------------------------------------------------------------------------
// K6  gang_fit_kernel — THE hot kernel.  For every (pod, node) pair:
//   fit   = classfit bit  AND  min_d(left_d - req_d) >= 0
//           (compareResourceAndRequire(singleNodeResource(node,pod,1), require(pod)),
//            core.go:634-699, as asserted by core_test.go:108-110)
//   score = fit ? min_d(left_d - req_d) : INT64_MIN      (residual capacity)
// and per pod, in the same launch: feasible count + best node (warp shuffles).  The per-group
// Permit count (core.go:303) follows in gang_admit_kernel.
//
// Mapping: a CTA = FIT_WARPS consumer warps + one producer warp.  It owns PODS_PER_CTA pods (each
// consumer warp PODS_PER_WARP of them, requests in registers) and sweeps the whole node table in
// tiles of NODE_TILE nodes.
//   INPUT: the producer lane streams the tiles of the residual table into a FIT_STAGES-deep
//     shared-memory ring with 1-D TMA bulk copies (cp.async.bulk global->shared, one per lane
//     row), guarded by full/empty mbarrier pairs; consumers never meet at a CTA-wide barrier.
//   OUTPUT: each lane writes the score of every pair it evaluates straight from registers with an
//     8-byte streaming store (st.global.cs, SASS STG.E.EF.64): 256 contiguous bytes of one matrix
//     row per warp store.  Ballot words are assembled in a per-warp shared-memory slab and leave as
//     one aligned 128-byte bitmap line per pod and 1024 nodes.  Staging the scores in shared memory
//     for TMA bulk stores was measured 3 % slower in the kernel (DESIGN §4, profiles/README.md).
// A lane owns nodes lane, lane+32, ... of the tile, keeps their `left` in registers and evaluates
// PODS_PER_WARP pods against them at a time.
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                             uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

__device__ __forceinline__ int64_t min64(int64_t a, int64_t b) { return a < b ? a : b; }
// high word of an int64, opaque to the optimiser (it otherwise re-forms a 2-instruction 64-bit compare)
__device__ __forceinline__ int32_t hi32(int64_t v) {
  int32_t lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v));
  (void)lo;
  return hi;
}
__device__ __forceinline__ uint32_t lo32(int64_t v) {
  int32_t lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v));
  (void)hi;
  return (uint32_t)lo;
}
// Ballot-word store of the hot loop.  volatile (never dropped, kept in order among themselves) but
// WITHOUT a "memory" clobber: the compiler may hoist the next nodes' LDS above it (the slab it writes
// is only read after a __syncwarp, which is a compiler barrier).
__device__ __forceinline__ void sts_u32(uint32_t saddr, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(saddr), "r"(v));
}

struct FitArgs {
  const int64_t* left_w;     // [LW][Npad] wide lanes
  const int32_t* left_n;     // [LN+LS][Npad] narrow lanes, then scaled lanes
  const ColBits* classfit;   // [classes][n_tiles][32] transposed class bits
  const int64_t* req;        // [L][P]
  const uint32_t* req_present;
  const uint32_t* fit_class;
  LaneMap lm;
  // outputs
  uint32_t* feasible_count;
  int32_t* best_node;
  int64_t* best_score;
  uint32_t* fit_bitmap;   // [Ppad][W] or null   (Ppad = P rounded up to PODS_PER_CTA: no pod guard)
  int64_t* score;         // [Ppad][score_pitch] or null
  // Row pitches in BYTES as 64-bit kernel parameters: ptxas 12.9 miscompiles the uniform-datapath
  // form of `int32 base + (uint32 Npad << 2)` (a lone ULEA with the high word zeroed) when the
  // TMA source address of a narrow row is derived from a 32-bit Npad; 64-bit pitches avoid it.
  uint64_t left_w_pitch, left_n_pitch;
  uint64_t score_pitch;   // elements per score row: N rounded up to even (16-byte row starts)
  uint32_t bitmap_pitch;  // words per fit-bitmap row: ceil(N/32) rounded up to 32 (rows are whole 128-byte lines)
  uint32_t P, N, Npad, W;
  // Tail balance: CTA units (PODS_PER_CTA pods x the whole node range) [0, n_full) fill whole waves of the
  // resident CTA slots; each of the remaining units is cut into tail_split node-range pieces (whole bitmap
  // lines), one CTA each, so that the last partial wave spreads over every SM instead of leaving most idle.
  // Pieces combine their per-pod results with atomics (count add, packed (score+1, ~node) max).
  uint32_t n_full, tail_split;
  unsigned long long* best_packed;   // [P] or null (tail_split == 1)
};

// running best score of a lane: int32 on the narrow fast path (scores of fitting pairs are < 2^27,
// "none" = -1), int64 otherwise ("none" = INT64_MIN)
template <bool NARROW> struct BestT { using type = int64_t; };
template <> struct BestT<true> { using type = int32_t; };

// One node tile for the PODS_PER_WARP pods of a warp.
//   narrow lanes: one 32-bit VIADDMNMX (fused subtract+min) each;
//   scaled lanes: x = min(left' - req', C) (one VIADDMNMX: the clamp keeps x << k below 2^31), its sign
//     joins the fit test, x << k (exact original units, or 2^27 = "cannot be the minimum") joins the min;
//   wide lanes: 64-bit subtract, sign through the high word, low word when the high word is 0.
// Ballot words go to a per-warp shared-memory slab (one STS per pair, every lane writes the same word);
// scores (SCORE) go to rows row0 .. row0 + PODS_PER_WARP - 1 of the matrix as int64: fit ? m : INT64_MIN.
// OUT: what leaves the SMs besides the per-pod results — 0 nothing (decisions only: feasible counts come from a
// predicated add, no ballot), 1 the fit bitmap, 2 the score matrix (+ the bitmap when its pointer is set).
enum { FIT_OUT_NONE = 0, FIT_OUT_BITMAP = 1, FIT_OUT_SCORE = 2 };
template <int LW, int LN, int LS, int OUT>
__device__ __forceinline__ void fit_tile(const FitArgs& a, const int64_t* __restrict__ tlw,
                                          const int32_t* __restrict__ tln,
                                          const int64_t (&rqw)[PODS_PER_WARP][LW > 0 ? LW : 1],
                                          const int32_t (&rqn)[PODS_PER_WARP][LN + LS > 0 ? LN + LS : 1],
                                          const ColBits (&colbits)[PODS_PER_WARP],
                                          uint32_t* s_words, uint32_t wbase /*tile's first word in the line*/, uint32_t node_base, uint32_t lane,
                                          typename BestT<(LN > 0)>::type (&best_s)[PODS_PER_WARP],
                                          int32_t (&best_n)[PODS_PER_WARP], int32_t (&kb)[PODS_PER_WARP],
                                          uint32_t (&cnt)[PODS_PER_WARP], uint32_t row0) {
  constexpr bool SCORE = OUT == FIT_OUT_SCORE;
  constexpr bool WORDS = OUT != FIT_OUT_NONE;
  const int64_t* tpw = tlw + lane;
  const int32_t* tpn = tln + lane;
  int32_t node = (int32_t)(node_base + lane);
  uint32_t wp = smem_u32(s_words) + wbase * 4;   // word (wbase + j) of the 32-word line being assembled
  int32_t jrem = TILE_WORDS - 1;   // best-node key: low KEY_BITS bits = TILE_WORDS-1-j (earlier node wins a tie)
#pragma unroll 1
  for (int jb = 0; jb < TILE_WORDS; jb += 4) {
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      int64_t lfw[LW > 0 ? LW : 1];
      int32_t lfn[LN + LS > 0 ? LN + LS : 1];
#pragma unroll
      for (int d = 0; d < LW; ++d) lfw[d] = tpw[d * NODE_TILE + jj * 32];
#pragma unroll
      for (int d = 0; d < LN + LS; ++d) lfn[d] = tpn[d * NODE_TILE + jj * 32];
#pragma unroll
      for (int r = 0; r < PODS_PER_WARP; ++r) {
        if (LN > 0) {
          // Narrow fast path.  t = min over the narrow lanes is a REAL difference (the narrow set
          // holds a fixed lane) with |t| < 2^27, and the pair's score m = min over all lanes <= t.
          // So when the pair fits (every difference >= 0) m is a 32-bit value: the other lanes
          // only matter through (a) their sign and (b) their value when it is below 2^27.
          int32_t t = lfn[0] - rqn[r][0];
#pragma unroll
          for (int d = 1; d < LN; ++d) t = min(t, lfn[d] - rqn[r][d]);
          uint32_t m32 = (uint32_t)t;
          int32_t sgn = t;
#pragma unroll
          for (int d = 0; d < LS; ++d) {
            const int32_t x = min(lfn[LN + d] - rqn[r][LN + d], (int32_t)a.lm.sclamp[d]);
            sgn |= x;
            m32 = min(m32, (uint32_t)x << a.lm.sshift[d]);   // unsigned: valid when all are >= 0
          }
#pragma unroll
          for (int d = 0; d < LW; ++d) {
            const int64_t w = lfw[d] - rqw[r][d];
            const int32_t whi = hi32(w);
            sgn |= whi;                                               // any negative difference -> sign bit
            m32 = min(m32, whi != 0 ? 0xffffffffu : lo32(w));
          }
          const bool fit = (sgn >= 0) && ((colbits[r] >> (jb + jj)) & 1u);
          if (WORDS) sts_u32(wp + (r * 32 + jj) * 4, __ballot_sync(0xffffffffu, fit));
          else if (fit) ++cnt[r];
          // best node of the tile as ONE running max: key = score * 2^KEY_BITS + (TILE_WORDS-1-j) < 2^31
          // (scores of fitting pairs are < 2^27), -1 = none; decoded once per tile
          const int32_t key = (int32_t)(m32 << KEY_BITS) + (jrem - jj);
          if (fit) kb[r] = max(kb[r], key);
          if (SCORE && (uint32_t)(node + jj * 32) < a.N)
            __stcs(reinterpret_cast<unsigned long long*>(a.score) + (size_t)(row0 + r) * a.score_pitch + (node + jj * 32),
                   (unsigned long long)(fit ? m32 : 0u) | ((unsigned long long)(fit ? 0u : 0x80000000u) << 32));
        } else {
          int64_t m = lfw[0] - rqw[r][0];
#pragma unroll
          for (int d = 1; d < LW; ++d) m = min64(m, lfw[d] - rqw[r][d]);
          const bool fit = (hi32(m) >= 0) && ((colbits[r] >> (jb + jj)) & 1u);
          if (WORDS) sts_u32(wp + (r * 32 + jj) * 4, __ballot_sync(0xffffffffu, fit));
          else if (fit) ++cnt[r];
          if (fit && m > best_s[r]) { best_s[r] = m; best_n[r] = node + jj * 32; }
          if (SCORE && (uint32_t)(node + jj * 32) < a.N)
            __stcs(reinterpret_cast<long long*>(a.score) + (size_t)(row0 + r) * a.score_pitch + (node + jj * 32),
                   fit ? (long long)m : (long long)INT64_MIN);
        }
      }
    }
    tpw += 128;
    tpn += 128;
    node += 128;
    jrem -= 4;
    wp += 16;
  }
}

__host__ __device__ constexpr size_t fit_tile_bytes(int LW, int LN, int LS) {
  return (size_t)NODE_TILE * (8 * LW + 4 * (LN + LS));
}
// shared-memory layout: [FIT_STAGES]{[LW][NODE_TILE] i64, [LN+LS][NODE_TILE] i32} | req_w | req_n | mbarriers |
//                       ballot words, 128-byte aligned
__host__ __device__ constexpr size_t gang_fit_smem_bytes(int LW, int LN, int LS) {
  size_t b = FIT_STAGES * fit_tile_bytes(LW, LN, LS) + (size_t)PODS_PER_CTA * (8 * LW + 4 * (LN + LS));
  b = (b + 7) & ~(size_t)7;
  b += 2 * FIT_STAGES * sizeof(uint64_t) + (size_t)PODS_PER_CTA * 32 * sizeof(uint32_t);
  return (b + 127) & ~(size_t)127;
}
// the widest shape (every lane wide) must fit the 227 KB a CTA may have on sm_100a
static_assert(gang_fit_smem_bytes(BS_MAX_LANES, 0, 0) <= 227 * 1024, "gang_fit_kernel: shared memory over 227 KB");

template <int LW, int LN, int LS, int OUT>
__global__ void __launch_bounds__(FIT_THREADS, 2) gang_fit_kernel(FitArgs a) {
  constexpr bool WORDS = OUT != FIT_OUT_NONE;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr size_t STAGE_BYTES = fit_tile_bytes(LW, LN, LS);
  constexpr int LNS = LN + LS;
  unsigned char* s_tile = smem_raw;
  int64_t* s_req_w = reinterpret_cast<int64_t*>(smem_raw + FIT_STAGES * STAGE_BYTES);
  int32_t* s_req_n = reinterpret_cast<int32_t*>(s_req_w + PODS_PER_CTA * LW);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(
      (reinterpret_cast<uintptr_t>(s_req_n + PODS_PER_CTA * LNS) + 7) & ~(uintptr_t)7);
  uint64_t* s_full = s_bar;                 // [FIT_STAGES] TMA bytes landed
  uint64_t* s_empty = s_bar + FIT_STAGES;   // [FIT_STAGES] every warp is done with the stage
  uint32_t* s_words_all = reinterpret_cast<uint32_t*>(s_bar + 2 * FIT_STAGES);

  const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  uint32_t* s_words = s_words_all + wid * PODS_PER_WARP * 32;   // per pod: the 32-word (1024-node) bitmap line being assembled
  uint32_t unit = blockIdx.x, piece = 0, npieces = 1;
  if (blockIdx.x >= a.n_full) {
    const uint32_t tl = blockIdx.x - a.n_full;
    unit = a.n_full + tl / a.tail_split;
    piece = tl % a.tail_split;
    npieces = a.tail_split;
  }
  const uint32_t pod0 = unit * PODS_PER_CTA;
  const uint32_t wpod0 = pod0 + wid * PODS_PER_WARP;  // first pod of this warp
  const uint32_t n_tiles = a.Npad / NODE_TILE;
  // this CTA's tile range: whole bitmap lines (TILES_PER_LINE tiles), split as evenly as lines allow
  const uint32_t n_lines = (n_tiles + TILES_PER_LINE - 1) / TILES_PER_LINE;
  const uint32_t tile_lo = min(n_tiles, (n_lines * piece / npieces) * TILES_PER_LINE);
  const uint32_t tile_hi = min(n_tiles, (n_lines * (piece + 1) / npieces) * TILES_PER_LINE);

  if (tid == 0) {
    for (int st = 0; st < FIT_STAGES; ++st) {
      mbar_init(&s_full[st], 1);
      mbar_init(&s_empty[st], FIT_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // stage the CTA's pod requests (sentinel for lanes without a map key; scaled lanes in their 2^k units)
  for (uint32_t i = tid; i < PODS_PER_CTA * (LW + LNS); i += FIT_THREADS) {
    const uint32_t pl = i / (LW + LNS), k = i % (LW + LNS);
    const uint32_t p = pod0 + pl;
    const bool is_w = k < (uint32_t)LW;
    const uint32_t kn = k - LW;
    const uint32_t d = is_w ? a.lm.wide[k] : (kn < (uint32_t)LN ? a.lm.narrow[kn] : a.lm.scaled[kn - LN]);
    int64_t v = 0;
    bool present = true;
    if (p < a.P) {
      present = d < 4 || ((a.req_present[p] >> d) & 1u);
      v = present ? a.req[(size_t)d * a.P + p] : 0;
    }
    if (is_w) s_req_w[pl * LW + k] = present ? v : UNCHECKED_REQ;
    else if (kn < (uint32_t)LN) s_req_n[pl * LNS + kn] = present ? (int32_t)v : UNCHECKED_REQ32;
    else s_req_n[pl * LNS + kn] = present ? (int32_t)(v >> a.lm.sunit[kn - LN]) : UNCHECKED_REQS;
  }
  __syncthreads();
  auto issue = [&](uint32_t tile, uint32_t stage) {
    mbar_expect_tx(&s_full[stage], (uint32_t)STAGE_BYTES);
    unsigned char* dst = s_tile + stage * STAGE_BYTES;
    const unsigned char* src_w = reinterpret_cast<const unsigned char*>(a.left_w) + (uint64_t)tile * (NODE_TILE * 8);
    const unsigned char* src_n = reinterpret_cast<const unsigned char*>(a.left_n) + (uint64_t)tile * (NODE_TILE * 4);
#pragma unroll
    for (int d = 0; d < LW; ++d)
      tma_bulk_g2s(dst + (size_t)d * NODE_TILE * 8, src_w + (uint64_t)d * a.left_w_pitch, NODE_TILE * 8,
                   &s_full[stage]);
#pragma unroll
    for (int d = 0; d < LNS; ++d)
      tma_bulk_g2s(dst + (size_t)LW * NODE_TILE * 8 + (size_t)d * NODE_TILE * 4,
                   src_n + (uint64_t)d * a.left_n_pitch, NODE_TILE * 4, &s_full[stage]);
  };
  // Warp specialisation: warp FIT_WARPS is the producer.  Its lane 0 walks the tiles, waits until
  // every consumer warp has released the stage (`empty`), and issues the TMA bulk copies that
  // complete on `full`.  Consumers never meet at a CTA-wide barrier during the sweep.
  if (wid == FIT_WARPS) {
    if (lane == 0) {
      for (uint32_t tile = tile_lo; tile < tile_hi; ++tile) {
        const uint32_t st = (tile - tile_lo) % FIT_STAGES, use = (tile - tile_lo) / FIT_STAGES;
        if (use > 0) mbar_wait(&s_empty[st], (use - 1) & 1);
        issue(tile, st);
      }
    }
    return;
  }

  // per-pod state of this warp (requests are warp-uniform, in registers for the whole sweep).
  // The score / bitmap buffers hold PODS_PER_CTA-padded rows, so pods >= P need no guard.
  const bool want_bitmap = a.fit_bitmap != nullptr;
  uint32_t cnt[PODS_PER_WARP];
  typename BestT<(LN > 0)>::type best_s[PODS_PER_WARP];
  int32_t best_n[PODS_PER_WARP];
  int32_t kb[PODS_PER_WARP], kthr[PODS_PER_WARP];   // tile-local best key; smallest key that beats best_s
  int64_t rqw[PODS_PER_WARP][LW > 0 ? LW : 1];
  int32_t rqn[PODS_PER_WARP][LNS > 0 ? LNS : 1];
  uint32_t coff[PODS_PER_WARP];
#pragma unroll
  for (int r = 0; r < PODS_PER_WARP; ++r) {
    cnt[r] = 0; best_n[r] = -1; kb[r] = -1; kthr[r] = 0;
    best_s[r] = LN > 0 ? (typename BestT<(LN > 0)>::type)(-1) : (typename BestT<(LN > 0)>::type)INT64_MIN;
    const uint32_t p = wpod0 + r;
    coff[r] = (p < a.P ? a.fit_class[p] : 0u) * n_tiles * 32 + lane;
#pragma unroll
    for (int d = 0; d < LW; ++d) rqw[r][d] = s_req_w[(wid * PODS_PER_WARP + r) * LW + d];
#pragma unroll
    for (int d = 0; d < LNS; ++d) rqn[r][d] = s_req_n[(wid * PODS_PER_WARP + r) * LNS + d];
  }

  // Consumers: a warp releases a stage by arriving on its `empty` mbarrier and may run up to
  // FIT_STAGES-1 tiles ahead of the slowest warp.
  uint32_t stage = 0, phase = 0;
  ColBits colnext[PODS_PER_WARP];   // class bits are fetched one tile ahead (their L2 latency stays off the tile's critical path)
#pragma unroll
  for (int r = 0; r < PODS_PER_WARP; ++r) colnext[r] = __ldg(a.classfit + coff[r] + min(tile_lo, n_tiles - 1) * 32);
  for (uint32_t tile = tile_lo; tile < tile_hi; ++tile) {
    ColBits colbits[PODS_PER_WARP];
    const uint32_t tnext = tile + 1 < tile_hi ? tile + 1 : tile;
#pragma unroll
    for (int r = 0; r < PODS_PER_WARP; ++r) {
      colbits[r] = colnext[r];
      colnext[r] = __ldg(a.classfit + coff[r] + tnext * 32);
    }
    mbar_wait(&s_full[stage], phase);
    const int64_t* tlw = reinterpret_cast<const int64_t*>(s_tile + stage * STAGE_BYTES);
    const int32_t* tln = reinterpret_cast<const int32_t*>(s_tile + stage * STAGE_BYTES + (size_t)LW * NODE_TILE * 8);
    const uint32_t node_base = tile * NODE_TILE;
    const uint32_t wbase = (tile % TILES_PER_LINE) * TILE_WORDS;
    fit_tile<LW, LN, LS, OUT>(a, tlw, tln, rqw, rqn, colbits, s_words, wbase, node_base, lane, best_s, best_n, kb, cnt, wpod0);
    if (LN > 0) {
      // a tile's best key beats the running best iff key >= (best_s + 1) << KEY_BITS: strictly greater score
      // (an equal score in a later tile loses to the earlier node)
#pragma unroll
      for (int r = 0; r < PODS_PER_WARP; ++r) {
        if (kb[r] >= kthr[r]) {
          best_s[r] = kb[r] >> KEY_BITS;
          best_n[r] = (int32_t)(node_base + lane) + (TILE_WORDS - 1 - (kb[r] & (TILE_WORDS - 1))) * 32;
          kthr[r] = (best_s[r] + 1) << KEY_BITS;
        }
        kb[r] = -1;
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&s_empty[stage]);   // this warp no longer reads the stage
    // Fit bitmap: the ballot words of TILES_PER_LINE tiles make one 128-byte line per pod (the bitmap's row
    // pitch is a multiple of 32 words), written with one fully coalesced store — 4-byte pieces of unaligned rows
    // cost 0.15 ms on the bench workload (partial sectors), a full aligned line costs nothing measurable.
    if (WORDS && ((tile + 1) % TILES_PER_LINE == 0 || tile + 1 == tile_hi)) {
      const uint32_t line = tile / TILES_PER_LINE;
      const uint32_t valid = (tile % TILES_PER_LINE + 1) * TILE_WORDS;   // words assembled in this line
      if (lane < valid) {
#pragma unroll
        for (int r = 0; r < PODS_PER_WARP; ++r) {
          const uint32_t w = s_words[r * 32 + lane];
          cnt[r] += __popc(w);
          if (want_bitmap) a.fit_bitmap[(size_t)(wpod0 + r) * a.bitmap_pitch + line * 32 + lane] = w;
        }
      }
    }
    __syncwarp();                                   // the ballot slab is rewritten by the next tile
    if (++stage == FIT_STAGES) { stage = 0; phase ^= 1; }
  }

  // per-pod reductions across the warp: best = max score, lowest node on ties
#pragma unroll
  for (int k = 0; k < PODS_PER_WARP; ++k) {
    int32_t n = best_n[k];
    int64_t s = n < 0 ? INT64_MIN : (int64_t)best_s[k];
    uint32_t c = cnt[k];
    for (int o = 16; o; o >>= 1) {
      const int64_t os = __shfl_xor_sync(0xffffffffu, s, o);
      const int32_t on = __shfl_xor_sync(0xffffffffu, n, o);
      c += __shfl_xor_sync(0xffffffffu, c, o);
      if (on >= 0 && (n < 0 || os > s || (os == s && on < n))) { s = os; n = on; }
    }
    const uint32_t p = wpod0 + k;
    if (p < a.P && lane == 0) {
      if (npieces == 1) {
        a.feasible_count[p] = c;
        a.best_node[p] = n;
        a.best_score[p] = s;
      } else {
        // a piece of a split unit: max of (score + 1) << 32 | ~node picks the highest score, then the lowest
        // node; 0 = none (fit_unpack_kernel turns it back into best_node / best_score)
        if (c) atomicAdd(&a.feasible_count[p], c);
        if (n >= 0) atomicMax(&a.best_packed[p], ((unsigned long long)(uint32_t)(s + 1) << 32) | (uint32_t)(~(uint32_t)n));
      }
    }
  }
}

// per-pod results of the split tail units: max((score + 1) << 32 | ~node) -> best_node / best_score
static __global__ void fit_unpack_kernel(const unsigned long long* __restrict__ packed, uint32_t p0, uint32_t P,
                                         int32_t* __restrict__ best_node, int64_t* __restrict__ best_score) {
  const uint32_t p = p0 + blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const unsigned long long v = packed[p];
  if (v == 0) { best_node[p] = -1; best_score[p] = INT64_MIN; return; }
  best_node[p] = (int32_t)(~(uint32_t)v);
  best_score[p] = (int64_t)(v >> 32) - 1;
}
constexpr uint32_t FIT_TAIL_SPLIT = 8;   // pieces a tail unit is cut into at most

}  // namespace bsk

// ---- variant table ---------------------------------------------------------------------------
// (LW wide, LN narrow, LS scaled) shapes that are instantiated, each with and without the score matrix:
//   LN == 0 : all lanes wide, LW = 4..16 (fallback when no fixed lane is narrow);
//   LN 1..8 : (LW, LS) in FIT_WS_COMBOS.
// fit_inst.cu compiles slice n (BS_FIT_SLICE): 0 = the all-wide kernels, n = 1..8 the kernels with LN = n.
namespace bsk {
// launches gang_fit_kernel over `units` CTA units (tail units split, see FitArgs); *launches gets the number of
// kernels launched (1, or 2 with the unpack kernel)
// ev_a / ev_b (null = none) are recorded right around the gang_fit_kernel launch itself, inside the tail's memsets
// and unpack kernel: the stage time the roofline uses is that one kernel's duration
using FitFn = cudaError_t (*)(const FitArgs&, uint32_t units, cudaStream_t, uint32_t* launches, cudaEvent_t ev_a, cudaEvent_t ev_b);   // one per (shape, FIT_OUT_*)
constexpr int FIT_MAX_LN = 8;
constexpr int FIT_N_SLICES = FIT_MAX_LN + 1;
struct FitWS { int lw, ls; };
constexpr FitWS FIT_WS_COMBOS[] = {{0, 0}, {1, 0}, {2, 0}, {3, 0}, {4, 0}, {0, 1}, {0, 2}, {0, 3}, {1, 1}, {1, 2}, {2, 1}};
constexpr int FIT_N_WS = sizeof(FIT_WS_COMBOS) / sizeof(FIT_WS_COMBOS[0]);
inline bool fit_variant_exists(uint32_t LW, uint32_t LN, uint32_t LS) {
  if (LN == 0) return LS == 0 && LW >= 4 && LW <= BS_MAX_LANES;
  if (LN > (uint32_t)FIT_MAX_LN || LW + LN + LS < 4 || LW + LN + LS > BS_MAX_LANES) return false;
  for (int i = 0; i < FIT_N_WS; ++i)
    if ((uint32_t)FIT_WS_COMBOS[i].lw == LW && (uint32_t)FIT_WS_COMBOS[i].ls == LS) return true;
  return false;
}
// defined in fit_inst.cu (one definition per slice); nullptr when the slice does not hold the shape
FitFn fit_lookup_slice0(uint32_t LW, uint32_t LN, uint32_t LS, int out);
FitFn fit_lookup_slice1(uint32_t LW, uint32_t LN, uint32_t LS, int out);
FitFn fit_lookup_slice2(uint32_t LW, uint32_t LN, uint32_t LS, int out);
FitFn fit_lookup_slice3(uint32_t LW, uint32_t LN, uint32_t LS, int out);
FitFn fit_lookup_slice4(uint32_t LW, uint32_t LN, uint32_t LS, int out);
FitFn fit_lookup_slice5(uint32_t LW, uint32_t LN, uint32_t LS, int out);
FitFn fit_lookup_slice6(uint32_t LW, uint32_t LN, uint32_t LS, int out);
FitFn fit_lookup_slice7(uint32_t LW, uint32_t LN, uint32_t LS, int out);
FitFn fit_lookup_slice8(uint32_t LW, uint32_t LN, uint32_t LS, int out);
inline FitFn fit_lookup(uint32_t LW, uint32_t LN, uint32_t LS, int out) {
  switch (LN) {
    case 0: return fit_lookup_slice0(LW, LN, LS, out);
    case 1: return fit_lookup_slice1(LW, LN, LS, out);
    case 2: return fit_lookup_slice2(LW, LN, LS, out);
    case 3: return fit_lookup_slice3(LW, LN, LS, out);
    case 4: return fit_lookup_slice4(LW, LN, LS, out);
    case 5: return fit_lookup_slice5(LW, LN, LS, out);
    case 6: return fit_lookup_slice6(LW, LN, LS, out);
    case 7: return fit_lookup_slice7(LW, LN, LS, out);
    case 8: return fit_lookup_slice8(LW, LN, LS, out);
  }
  return nullptr;
}
}  // namespace bsk
