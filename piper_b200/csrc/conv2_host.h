// Host side of the persistent tensor-core convolution (conv2_body.inl): tiling plan, stacked weight
// packing and launch-argument fill.  Plain C++ (no CUDA calls): shared by conv_mma2.cu and the CPU model in tests/sim.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <vector>

#include "kernels.cuh"

namespace pb200 {
namespace conv2 {

struct Plan {
  bool ok = false, tf32 = false;
  int prec = 0;                       // conv2::PREC_BF16 / PREC_TF32 / PREC_F16
  int n_tile = 0, n_tiles = 0, mt = 128, kc = 0, stage_rows = 0, raw_stride = 0, t_slots = 1, tmem_cols = 0, chains = 1;
  int mh_stride = 0;
  size_t smem = 0, w_bytes = 0;
};

inline int pow2_cols(int n) { return n <= 32 ? 32 : n <= 64 ? 64 : n <= 128 ? 128 : n <= 256 ? 256 : 512; }

// Output-row tile N (<= 128 so that the stacked instruction has N' = 2N <= 256), K-chains (2 for tf32x3, DESIGN.md
// section 3), tile height, TMEM double-buffering and the largest channel chunk that fits 196 KB of shared memory.
// prec: 0 bf16x3, 1 tf32x3, 2 fp16x3.  chains: K-chains per accumulator pair (2 where fp32-grade accuracy is needed).
// opts bit 0: allow 256-row tiles for multi-chain fp16 / bf16 layers (one TMEM set, but every weight unit serves twice the rows)
inline bool plan(int ci, int rows, int k, int dil, int prec, int chains, Plan& p, int opts = 0) {
  const bool tf32 = prec == 1;
  p = Plan{};
  p.tf32 = tf32;
  p.prec = prec;
  const int es = tf32 ? 4 : 2, kstep = tf32 ? 8 : 16;
  if (ci % kstep != 0 || rows % 16 != 0 || rows < 16) return false;
  p.chains = chains;
  // candidates: (n_tile, mt) with the accumulator sets of one tile within 512 columns; prefer two TMEM sets
  // (epilogue overlaps the next tile), then the wider row tile (fewer activation re-reads), then the taller tile
  int best_score = -1;
  for (int nt = 1; nt <= 64; ++nt) {
    if (rows % nt || (rows / nt) % 16 || rows / nt > 128) continue;
    const int n_tile = rows / nt;
    if (chains > 1 && n_tile > 64 && (!(ci * k >= 900 && rows >= 256) || (opts & 4))) continue;   // wide tiles only for long reductions (opts bit 2: never - keeps two TMEM sets)
    for (int mt : {256, 128}) {
      if (tf32 && mt != 128) continue;                     // no 256-row tf32 kernel instantiation
      if (chains > 1 && mt != 128 && !(opts & 1)) continue;
      const int set_cols = mt / 128 * p.chains * 2 * n_tile;
      if (set_cols > 512) continue;
      const int slots = 2 * set_cols <= 512 ? 2 : 1;
      // accumulator halves start at multiples of n_tile columns: keep them 32-column aligned when the layer allows it
      // (every accumulator the shipped kernel has exercised on hardware is)
      int score = (n_tile % 32 == 0 ? 1000000 : 0) + slots * 100000 + n_tile * 5000 + mt / 128;
      if ((opts & 1) && chains > 1 && mt == 256) score += 500000;    // the option asks for the tall tile where it fits
      if ((opts & 2) && mt == 128) score += 2;                       // option: prefer 128-row tiles (larger channel chunks fit)
      if (score > best_score) {
        best_score = score;
        p.n_tile = n_tile; p.n_tiles = nt; p.mt = mt; p.t_slots = slots;
      }
    }
  }
  if (best_score < 0) return false;
  p.mh_stride = p.chains * 2 * p.n_tile;
  p.tmem_cols = pow2_cols(p.t_slots * (p.mt / 128) * p.mh_stride);
  p.stage_rows = (p.mt + (k - 1) * dil + 7) & ~7;
  if (p.stage_rows * 16 >= (1 << 18)) return false;
  p.raw_stride = p.stage_rows + 8;
  for (int c = ci; c >= kstep; c -= kstep) {
    if (ci % c) continue;
    const size_t bytes = size_t(2) * c * p.raw_stride * 4 + size_t(2) * 2 * c * p.stage_rows * es + size_t(4) * c * 2 * p.n_tile * es;
    if (bytes <= (size_t(196) << 10)) {
      p.kc = c;
      p.smem = bytes;
      break;
    }
  }
  if (!p.kc) return false;
  p.w_bytes = size_t(rows / p.n_tile) * k * ci * 2 * p.n_tile * es;
  p.ok = true;
  return true;
}

inline uint16_t f32_to_bf16_rn(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return uint16_t((u >> 16) | 0x40);
  return uint16_t((u + 0x7fffu + ((u >> 16) & 1u)) >> 16);
}
inline float bf16_to_f32(uint16_t h) {
  uint32_t u = uint32_t(h) << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
inline float f32_to_tf32_rna(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7f800000u) == 0x7f800000u) return f;
  u = (u + 0x1000u) & 0xffffe000u;
  memcpy(&f, &u, 4);
  return f;
}

// IEEE binary16 round-to-nearest-even (overflow -> inf, subnormals kept): what cvt.rn.f16.f32 does
inline uint16_t f32_to_f16_rn(float f) {
  uint32_t x;
  memcpy(&x, &f, 4);
  const uint32_t sign = (x >> 16) & 0x8000u;
  x &= 0x7fffffffu;
  if (x >= 0x7f800000u) return uint16_t(sign | 0x7c00u | (x > 0x7f800000u ? 0x200u : 0u));   // inf / nan
  if (x >= 0x477ff000u) return uint16_t(sign | 0x7c00u);                                         // rounds to >= 65520: inf
  if (x < 0x33000001u) return uint16_t(sign);                                                    // below half the smallest subnormal
  int e = int(x >> 23) - 127;
  uint32_t m = (x & 0x7fffffu) | 0x800000u;
  int shift;
  uint32_t base;
  if (e < -14) { shift = 13 + (-14 - e); base = 0; }                                             // subnormal result
  else { shift = 13; base = uint32_t(e + 15) << 10; m &= 0x7fffffu; }
  const uint32_t q = m >> shift, rem = m & ((1u << shift) - 1), halfway = 1u << (shift - 1);
  uint32_t r = base + q;
  if (rem > halfway || (rem == halfway && (q & 1u))) ++r;                                        // carries into the exponent correctly
  return uint16_t(sign | r);
}
inline float f16_to_f32(uint16_t h) {
  const uint32_t sign = uint32_t(h & 0x8000u) << 16, e = (h >> 10) & 0x1fu, m = h & 0x3ffu;
  uint32_t x;
  if (e == 0) {
    if (m == 0) x = sign;
    else {
      int sh = 0;
      uint32_t mm = m;
      while (!(mm & 0x400u)) { mm <<= 1; ++sh; }
      x = sign | (uint32_t(113 - sh) << 23) | ((mm & 0x3ffu) << 13);
    }
  } else if (e == 31) x = sign | 0x7f800000u | (m << 13);
  else x = sign | ((e + 112) << 23) | (m << 13);
  float f;
  memcpy(&f, &x, 4);
  return f;
}

// wsrc: the engine's fp32 layout [ci][k][rows_p] (row fastest).  out: [n tile][tap][ci / E][W_hi rows | W_lo rows][E].
inline void pack(const float* wsrc, int ci, int k, int rows_p, const Plan& p, uint8_t* out) {
  const int es = p.tf32 ? 4 : 2, E = 16 / es, NT = p.n_tile;
  for (int nt = 0; nt < p.n_tiles; ++nt)
    for (int j = 0; j < k; ++j) {
      uint8_t* base = out + (size_t(nt) * k + j) * (ci / E) * 2 * NT * 16;
      for (int cin = 0; cin < ci; ++cin)
        for (int n = 0; n < NT; ++n) {
          const float v = wsrc[(size_t(cin) * k + j) * rows_p + nt * NT + n];
          uint8_t* g = base + size_t(cin / E) * 2 * NT * 16;
          const size_t hi_pos = size_t(n) * E + (cin % E), lo_pos = size_t(NT + n) * E + (cin % E);
          if (p.tf32) {
            const float hi = f32_to_tf32_rna(v), lo = v - hi;
            memcpy(g + hi_pos * 4, &hi, 4);
            memcpy(g + lo_pos * 4, &lo, 4);
          } else if (p.prec == 2) {
            const uint16_t hi = f32_to_f16_rn(v), lo = f32_to_f16_rn(v - f16_to_f32(hi));
            memcpy(g + hi_pos * 2, &hi, 2);
            memcpy(g + lo_pos * 2, &lo, 2);
          } else {
            const uint16_t hi = f32_to_bf16_rn(v), lo = f32_to_bf16_rn(v - bf16_to_f32(hi));
            memcpy(g + hi_pos * 2, &hi, 2);
            memcpy(g + lo_pos * 2, &lo, 2);
          }
        }
    }
}

// plan -> the tiling fields of the launch arguments; returns the grid size (0: nothing to do)
// tm: stage the activation rows with one tensor-map TMA copy per channel chunk (two when the staged window is wider than
// the 256-element box limit) instead of one bulk copy per channel row; `td` then describes the tensor and the box.
constexpr size_t kAstatSmem = size_t(212) << 10;
inline int fill_args(MmaConvArgs& a, const Plan& p, int B, int max_len, bool tm = false, TmapDesc* td = nullptr, bool astat_ok = false,
                     size_t* smem_out = nullptr) {
  a.n_tile = p.n_tile; a.chains = p.chains; a.mh_stride = p.mh_stride;
  a.kc = p.kc; a.stage_rows = p.stage_rows; a.raw_stride = p.raw_stride; a.t_slots = p.t_slots; a.tmem_cols = p.tmem_cols;
  a.chains = std::min(p.chains, (a.ci / p.kc) * a.k);          // never more chains than weight units
  if (p.chains > 2) throw std::runtime_error("conv2: at most two K-chains (the kernel picks the chain by comparison)");
  // flat mode divides a concatenated position by the slot width with a 32-bit reciprocal multiplication (conv2_body.inl)
  if (a.flat_tg > 0 && (a.flat_tg < 2 || ((long long)a.flat_n * a.flat_tg + 1024) * a.flat_tg >= (1LL << 32)))
    throw std::runtime_error("conv2: flat launch outside the range of the reciprocal division");
  a.tiles_per_item = (max_len + p.mt - 1) / p.mt;
  a.total_tiles = a.tiles_per_item * B * p.n_tiles;
  a.batch = B;
  {
    // Launches with one or two tiles per CTA are a latency chain (load -> convert -> MMA -> epilogue): with the whole
    // reduction in one channel chunk nothing overlaps.  Cut it into about four chunks so the stages pipeline within a
    // tile.  (The packed weights do not depend on the chunk size; a smaller chunk only uses less of the planned smem.)
    const int grid = std::min(a.total_tiles, 148);
    const int per_cta = grid > 0 ? (a.total_tiles + grid - 1) / grid : 0;
    const int kstep = p.tf32 ? 8 : 16;
    if (per_cta <= 2 && a.ci / p.kc < 4) {
      int pick = 0;
      for (int c = p.kc; c >= kstep; c -= kstep) {
        if (a.ci % c) continue;
        if (c < 32 && pick) break;
        pick = c;
        if (a.ci / c >= 4) break;
      }
      if (pick) a.kc = pick;
    }
    a.chains = std::min(p.chains, (a.ci / a.kc) * a.k);
  }
  // A-stationary order where it pays and is possible: several output-row tiles per position, and every channel chunk of a
  // position resident in the operand ring at once.  The ring then gets one slot per chunk (a_slots = C_in / kc <= 12) and
  // the chunk size is re-chosen so that raw staging (2 slots) + the whole converted window + the weight ring (4 slots)
  // fit kAstatSmem; the window is converted ONCE per position instead of once per output-row tile (9x for the q|k|v conv,
  // 12x for the first FFN conv: the role waits showed the MMA warp waiting for operands 40 % of those launches).
  a.n_tiles = p.n_tiles;
  a.a_slots = 2;
  a.astat = 0;
  if (smem_out) *smem_out = p.smem;
  if (astat_ok && p.n_tiles > 1) {
    const int es = p.tf32 ? 4 : 2, kstep = p.tf32 ? 8 : 16;
    int pick = 0;
    for (int c = a.ci; c >= kstep; c -= kstep) {
      if (a.ci % c) continue;
      const int n_kc = a.ci / c;
      if (n_kc > 12) break;
      const size_t bytes = size_t(2) * c * p.raw_stride * 4 + size_t(2) * a.ci * p.stage_rows * es + size_t(4) * c * 2 * p.n_tile * es;
      if (bytes > kAstatSmem) continue;
      pick = c;
      if (n_kc >= 4) break;                                // enough chunks for load / convert / MMA to overlap inside a position
    }
    if (pick) {
      a.kc = pick;
      a.a_slots = std::max(2, a.ci / pick);
      a.astat = 1;
      a.chains = std::min(p.chains, (a.ci / a.kc) * a.k);
      if (smem_out)
        *smem_out = size_t(2) * pick * p.raw_stride * 4 + size_t(a.a_slots) * 2 * pick * p.stage_rows * es + size_t(4) * pick * 2 * p.n_tile * es;
    }
  }
  a.tm_boxes = 0;
  if (tm && td) {
    // the innermost start coordinate of a tiled tensor copy must be 16-byte aligned (an unaligned one is an illegal
    // instruction on the B200: tools/probe/tma_probe.cu), so the window starts at t_lo rounded down to 4 floats and is
    // raw_stride = stage_rows + 8 wide, like the per-row path
    a.tm_boxes = p.raw_stride > 256 ? 2 : 1;
    td->base = a.x.p;
    td->dims[0] = a.x.cs; td->dims[1] = a.ci; td->dims[2] = B;
    td->stride1 = (long long)a.x.cs * 4; td->stride2 = a.x.bs * 4;
    td->box[0] = p.raw_stride / a.tm_boxes; td->box[1] = a.kc; td->box[2] = 1;
  }
  return std::min(a.total_tiles, 148);
}

}  // namespace conv2
}  // namespace pb200
