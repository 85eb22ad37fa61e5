// ozaki_layout.h — sizes of the INT8 digit-plane layout (ozaki.cu).  The kernels, the plan builder (plan.cpp, which
// stays CUDA-free) and the C API all size their buffers from here, so the plan arena always matches what the split
// kernel writes.
#pragma once
#include <cstdint>

namespace ecw {

constexpr int OZ_BK = 32;        // k per stage = K of one kind::i8 MMA
constexpr int OZ_TM = 128;       // tile rows  (MMA M)
constexpr int OZ_DEFAULT_NS = 7; // digits (FP64-level accuracy) the plane slots are sized for while the engine is off

// tile columns: NS accumulators of TN int32 columns must fit the 512 TMEM columns; every MMA needs N % 16 == 0
constexpr int ozaki_tile_n(int ns) { return ns >= 3 && ns <= 5 ? 96 : (ns == 6 ? 80 : 64); }
constexpr int64_t ozaki_padded_rows(int64_t R) { return (R + OZ_TM - 1) / OZ_TM * OZ_TM; }
constexpr int64_t ozaki_kblocks(int64_t K1, int64_t K2) { return K1 * ((K2 + OZ_BK - 1) / OZ_BK); }
// + one tile of slack: the last tile of the last slab may start inside the padded rows and run past them
constexpr int64_t ozaki_plane_bytes2(int64_t R, int64_t K1, int64_t K2, int ns) {
  return ozaki_padded_rows(R) * ozaki_kblocks(K1, K2) * OZ_BK * ns + OZ_TM * OZ_BK;
}
constexpr int64_t ozaki_plane_bytes(int64_t R, int64_t K, int ns) { return ozaki_plane_bytes2(R, 1, K, ns); }
// plane bytes in 8-byte elements: buffer slots and workspace offsets count doubles
constexpr int64_t ozaki_plane_elems(int64_t R, int64_t K1, int64_t K2, int ns) {
  return (ozaki_plane_bytes2(R, K1, K2, ns) + 7) / 8;
}
constexpr int64_t ozaki_stat_elems(int64_t R, int64_t K1) { return (K1 > 1 ? 2 + K1 : 2) * ozaki_padded_rows(R); }
// digits of a context's plane slots: its configured count, else OZ_DEFAULT_NS
constexpr int ozaki_digits(int oz_ns) { return oz_ns > 0 ? oz_ns : OZ_DEFAULT_NS; }

}  // namespace ecw
