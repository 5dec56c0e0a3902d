// fit_inst.cu — instantiates one slice of the gang_fit_kernel variant table (fit.cuh).
// Compiled FIT_N_SLICES times with -DBS_FIT_SLICE=n, in parallel (build.py): slice 0 holds the
// all-wide kernels (LN = 0, LW = 4..16), slice n >= 1 the kernels with LN = n narrow lanes.
#include <algorithm>

#include "fit.cuh"

#ifndef BS_FIT_SLICE
#error "compile with -DBS_FIT_SLICE=<0..8>"
#endif

namespace bsk {
namespace {

template <int LW, int LN, int LS, int OUT>
cudaError_t launch_fit_t(const FitArgs& a0, uint32_t units, cudaStream_t s, uint32_t* launches, cudaEvent_t ev_a, cudaEvent_t ev_b) {
  const size_t smem = gang_fit_smem_bytes(LW, LN, LS);
  // per launch, not cached: the attribute is per device and one process may drive several GPUs
  cudaError_t er = cudaFuncSetAttribute(gang_fit_kernel<LW, LN, LS, OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)smem);
  if (er != cudaSuccess) return er;
  FitArgs a = a0;
  a.n_full = units;
  a.tail_split = 1;
  // Tail balance (FitArgs): whole waves of resident CTA slots run full-range units; the units of the last,
  // partial wave are cut into node-range pieces so that every SM gets a share of it.  Narrow shapes only
  // (the packed best needs scores below 2^31).
  if (LN > 0 && a.best_packed && units) {
    int per_sm = 0, dev = 0, sms = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gang_fit_kernel<LW, LN, LS, OUT>, FIT_THREADS, smem) == cudaSuccess &&
        cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess &&
        per_sm > 0 && sms > 0) {
      const uint32_t slots = (uint32_t)per_sm * (uint32_t)sms;
      const uint32_t n_tiles = a.Npad / NODE_TILE, n_lines = (n_tiles + TILES_PER_LINE - 1) / TILES_PER_LINE;
      const uint32_t n_full = units / slots * slots, tail = units - n_full;
      const uint32_t split = std::min(FIT_TAIL_SPLIT, n_lines);
      if (tail && split > 1 && tail * 10 < slots * 9) {   // a nearly full last wave is left alone
        a.n_full = n_full;
        a.tail_split = split;
      }
    }
  }
  const uint32_t tail_units = units - a.n_full;
  if (a.tail_split > 1) {
    const uint32_t p0 = a.n_full * PODS_PER_CTA;
    if (p0 < a.P) {
      er = cudaMemsetAsync(a.feasible_count + p0, 0, (size_t)(a.P - p0) * 4, s);
      if (er == cudaSuccess) er = cudaMemsetAsync(a.best_packed + p0, 0, (size_t)(a.P - p0) * 8, s);
      if (er != cudaSuccess) return er;
    }
  }
  if (ev_a) cudaEventRecord(ev_a, s);
  gang_fit_kernel<LW, LN, LS, OUT><<<a.n_full + tail_units * a.tail_split, FIT_THREADS, smem, s>>>(a);
  if (ev_b) cudaEventRecord(ev_b, s);
  if (launches) *launches = 1;
  if (a.tail_split > 1) {
    const uint32_t p0 = a.n_full * PODS_PER_CTA;
    if (p0 < a.P) {
      fit_unpack_kernel<<<(a.P - p0 + 255) / 256, 256, 0, s>>>(a.best_packed, p0, a.P, a.best_node, a.best_score);
      if (launches) *launches = 2;
    }
  }
  return cudaGetLastError();
}

template <int LW, int LN, int LS>
FitFn pick(int out) {
  return out == FIT_OUT_SCORE ? launch_fit_t<LW, LN, LS, FIT_OUT_SCORE>
                              : (out == FIT_OUT_BITMAP ? launch_fit_t<LW, LN, LS, FIT_OUT_BITMAP> : launch_fit_t<LW, LN, LS, FIT_OUT_NONE>);
}

}  // namespace

#define BS_CAT2(a, b) a##b
#define BS_CAT(a, b) BS_CAT2(a, b)

FitFn BS_CAT(fit_lookup_slice, BS_FIT_SLICE)(uint32_t LW, uint32_t LN, uint32_t LS, int score) {
#if BS_FIT_SLICE == 0
  if (LN != 0 || LS != 0) return nullptr;
  switch (LW) {
    case 4: return pick<4, 0, 0>(score);
    case 5: return pick<5, 0, 0>(score);
    case 6: return pick<6, 0, 0>(score);
    case 7: return pick<7, 0, 0>(score);
    case 8: return pick<8, 0, 0>(score);
    case 9: return pick<9, 0, 0>(score);
    case 10: return pick<10, 0, 0>(score);
    case 11: return pick<11, 0, 0>(score);
    case 12: return pick<12, 0, 0>(score);
    case 13: return pick<13, 0, 0>(score);
    case 14: return pick<14, 0, 0>(score);
    case 15: return pick<15, 0, 0>(score);
    case 16: return pick<16, 0, 0>(score);
  }
  return nullptr;
#else
  constexpr int N = BS_FIT_SLICE;
  if (LN != (uint32_t)N || !fit_variant_exists(LW, LN, LS)) return nullptr;
  const uint32_t key = LW * 8 + LS;
  switch (key) {
#define BS_CASE(lw, ls)                                                        \
  case lw * 8 + ls:                                                            \
    if constexpr (lw + N + ls >= 4) return pick<lw, N, ls>(score); else break;
    BS_CASE(0, 0) BS_CASE(1, 0) BS_CASE(2, 0) BS_CASE(3, 0) BS_CASE(4, 0) BS_CASE(0, 1) BS_CASE(0, 2) BS_CASE(0, 3)
    BS_CASE(1, 1) BS_CASE(1, 2) BS_CASE(2, 1)
#undef BS_CASE
  }
  return nullptr;
#endif
}

}  // namespace bsk
