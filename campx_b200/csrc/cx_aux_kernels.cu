// Small kernels around the step path: reset (Engine.its_showtime state, engine.py:487-544), render of
// the current state (engine.py:295-324), layers / layered_board from finished boards
// (rendering.py:181-219), action format conversion (boat_race.py:26,40-49), synthetic Philox actions,
// entity state access and the boat_race safety metric (boat_race.py:117-151).
#include <math.h>
#include <string.h>

#include "cx_internal.cuh"
#include "cx_philox.cuh"
#include "cx_policy.cuh"


namespace {

constexpr int TB = 256;
inline unsigned blocks_for(int64_t n, int per_block = TB) { return (unsigned)((n + per_block - 1) / per_block); }

__device__ __forceinline__ double stat_identity(int i) {
  return (i == CX_STAT_RETURN_MAX || i == CX_STAT_NEG_RETURN_MIN) ? -INFINITY : 0.0;
}

// head block + every stripe (cx_internal.cuh: CX_STAT_STRIPES)
__global__ void k_stats_init(double* stats) {
  const int i = blockIdx.x * TB + threadIdx.x;
  if (i < (1 + CX_STAT_STRIPES) * CX_STATS_DOUBLES) stats[i] = stat_identity(i % CX_STATS_DOUBLES);
}

// Add the stripes into the head block and clear them: one block, thread = (stripe group, statistic); sums are taken
// in a fixed order, so the result does not depend on which warp added to which stripe first.
__global__ void k_stats_fold(double* stats) {
  __shared__ double part[TB];
  const int i = threadIdx.x % CX_STATS_DOUBLES, grp = threadIdx.x / CX_STATS_DOUBLES, ngrp = TB / CX_STATS_DOUBLES;
  const bool is_max = i == CX_STAT_RETURN_MAX || i == CX_STAT_NEG_RETURN_MIN;
  double acc = stat_identity(i);
  for (int s = grp; s < CX_STAT_STRIPES; s += ngrp) {
    double* p = stats + (1 + s) * CX_STATS_DOUBLES + i;
    const double v = *p;
    acc = is_max ? fmax(acc, v) : acc + v;
    *p = stat_identity(i);
  }
  part[threadIdx.x] = acc;
  __syncthreads();
  if (grp == 0) {
    double tot = stats[i];
    for (int g = 0; g < ngrp; ++g) tot = is_max ? fmax(tot, part[g * CX_STATS_DOUBLES + i]) : tot + part[g * CX_STATS_DOUBLES + i];
    stats[i] = tot;
  }
}

__global__ void k_agent_reset(uint8_t* cell, uint16_t* tstep, float* ret, float* perf, uint64_t* pick,
                              uint64_t all_items, int track, int init_cell, const uint8_t* mask, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n || (mask && !mask[i])) return;
  cell[i] = (uint8_t)init_cell;
  if (track) {
    tstep[i] = 0;
    ret[i] = 0.0f;
  }
  if (perf) perf[i] = 0.0f;
  if (pick) pick[i] = all_items;   // every item back on the board
}

struct GenInit {
  uint16_t init[CX_MAX_DYN];
  int n_dyn;
};

__global__ void k_generic_reset(uint16_t* dyn, uint16_t* tstep, float* ret, int track, GenInit gi,
                                const uint8_t* mask, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n || (mask && !mask[i])) return;
  for (int d = 0; d < gi.n_dyn; ++d) dyn[(int64_t)d * n + i] = gi.init[d];
  if (track) {
    tstep[i] = 0;
    ret[i] = 0.0f;
  }
}

__global__ void k_dynbd_reset(uint8_t* dynbd, const uint8_t* backdrop, int cells, const uint8_t* mask, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n * cells) return;
  const int64_t e = i / cells;
  if (mask && !mask[e]) return;
  dynbd[i] = backdrop[i - e * cells];
}

// pick (games with pickups, else null): the items each env holds; basech shows every item and every door closed, a
// taken item or an open door's cell shows its under_ch (CxPickItem, CxPickHeader)
__global__ void k_agent_render(const uint8_t* cell, const uint8_t* basech, const uint8_t* shown, int cells,
                               int agent_char, uint8_t* board, int64_t n, const uint64_t* pick,
                               const uint8_t* item_at, const CxPickItem* items, const CxPickHeader ph) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n * cells) return;
  const int64_t e = i / cells;
  const int c = (int)(i - e * cells);
  uint8_t v = basech[c];
  if (pick) {
    const uint32_t k = item_at[c];
    uint64_t closed;
    cx_doors(ph, pick[e], &closed);
    if (k != CX_NO_ITEM && !(((pick[e] | closed) >> k) & 1)) v = items[k].under_ch;
  }
  if (shown[cell[e]] == c) v = (uint8_t)agent_char;
  board[i] = v;
}

__global__ void k_get_agent(const uint8_t* cell, int32_t* out, int cells, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i < n) out[i] = cell[i] >= cells ? -1 : (int32_t)cell[i];
}
__global__ void k_set_agent(uint8_t* cell, const int32_t* in, int cells, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i < n) cell[i] = (in[i] < 0 || in[i] >= cells) ? (uint8_t)cells : (uint8_t)in[i];
}
// a sprite agent always has a position: out of range puts it on cell 0, as k_set_generic does for sprites
__global__ void k_set_agent_sprite(uint8_t* cell, const int32_t* in, int cells, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i < n) cell[i] = (in[i] < 0 || in[i] >= cells) ? (uint8_t)0 : (uint8_t)in[i];
}
// generic: ROLL state is (row_off << 8 | col_off) internally, exposed as row_off * cols + col_off
__global__ void k_get_generic(const uint16_t* dyn, int32_t* out, int is_roll, int cols, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n) return;
  const uint32_t v = dyn[i];
  out[i] = is_roll ? (int32_t)((v >> 8) * cols + (v & 255)) : (v == CX_EMPTY_CELL16 ? -1 : (int32_t)v);
}
__global__ void k_set_generic(uint16_t* dyn, const int32_t* in, int is_roll, int is_cell, int cols, int cells,
                              int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n) return;
  int32_t v = in[i];
  if (is_roll) {
    v = ((v % cells) + cells) % cells;
    dyn[i] = (uint16_t)(((v / cols) << 8) | (v % cols));
  } else if (v < 0 || v >= cells) {
    dyn[i] = is_cell ? (uint16_t)CX_EMPTY_CELL16 : (uint16_t)0;
  } else {
    dyn[i] = (uint16_t)v;
  }
}

__global__ void k_get_episode(const uint16_t* tstep, const float* ret, int32_t* steps, float* returns, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n) return;
  if (steps) steps[i] = (tstep[i] & CX_OVER_BIT) ? -(int32_t)(tstep[i] & ~CX_OVER_BIT) : (int32_t)tstep[i];
  if (returns) returns[i] = ret[i];
}

// rendering.py:204-215: layers[ch] = (board == ord(ch)); layered_board = stack over chars.
// One thread produces 4 consecutive output bytes of the [n, L, cells] tensor (coalesced 4-byte stores).
struct CharTable {
  uint8_t ch[CX_MAX_CHARS];
};
// layers / layered_board from finished boards (campx/rendering.py:204-215: layers[ch] = board == ord(ch)).
// One CTA stages EB boards in shared memory (coalesced 16-byte loads).  The output is produced four cells at
// a time: an unaligned 4-byte window of the board row (two LDS.32 + funnel shift) is compared against the
// channel's character with one SIMD byte compare (__vcmpeq4), and because a 4-cell output word may run over
// the end of a (board, channel) row, every word is the OR of two such segments.  The (board, channel, cell)
// coordinates are divided out once per thread and iteration (16 cells) and advanced incrementally.
// HBM traffic = cells bytes read + chars * cells * sizeof(OutT) bytes written per board.
__device__ __forceinline__ uint32_t bytes_equal01(uint32_t w, uint32_t ch4) {  // 0x01 where the bytes are equal
  const uint32_t x = w ^ ch4;
  const uint32_t t = (x & 0x7f7f7f7fu) + 0x7f7f7f7fu;   // bit 7 of a byte: one of its low 7 bits is set
  return (~(t | x) >> 7) & 0x01010101u;
}
struct LayerCursor {
  int e, k, c;  // board in the tile, channel, cell
};

// 0/1 bytes of the 4 output cells that start at cursor `cur`; advances the cursor by 4 cells (cells >= 4)
__device__ __forceinline__ uint32_t layer_word(const uint8_t* s_board, const uint32_t* s_ch4, int L, int cells,
                                               LayerCursor& cur) {
  auto window = [&](int byte_off) -> uint32_t {  // 4 board bytes starting at any byte offset of the tile
    const uint32_t* w = reinterpret_cast<const uint32_t*>(s_board) + (byte_off >> 2);
    return __funnelshift_r(w[0], w[1], (byte_off & 3) * 8);
  };
  const int row = cur.e * cells;
  const int l1 = min(4, cells - cur.c);                       // cells left in this (board, channel) row
  uint32_t m = bytes_equal01(window(row + cur.c), s_ch4[cur.k]);
  cur.c += 4;
  if (cur.c >= cells) {                                       // the word runs into the next row
    cur.c -= cells;
    if (++cur.k == L) {
      cur.k = 0;
      ++cur.e;
    }
    if (l1 < 4) {
      const uint32_t keep = (1u << (8 * l1)) - 1u;
      const uint32_t m2 = bytes_equal01(window(cur.e * cells), s_ch4[cur.k]);
      m = (m & keep) | (m2 << (8 * l1));
    }
  }
  return m;
}

// uint8 output, rows of whole 4-byte words (cells % 4 == 0, cells >= 16): the 16 output cells of a thread lie in at
// most two (board, channel) rows and every 4-cell word inside one of them, so a word is ONE aligned LDS.32, a
// select of the row's character and a branch-free zero-byte test; (row, cell) come from two multiplications
// with precomputed inverses instead of divisions.  Stores stay 16-byte chunks of the FLAT output (whole sectors).
struct LayerDivisors {
  uint32_t inv_cells, inv_L;  // ceil(2^32 / d)
  uint32_t inv_per;           // ceil(2^32 / (L * cells)), 0: not exact for this launch (divide instead)
};
__device__ __forceinline__ void layer_words16(const uint32_t* s32, const uint32_t* s_ch4, int L, int cells,
                                              const LayerDivisors dv, uint32_t o, uint32_t (&w)[4]) {
  const uint32_t row = __umulhi(o, dv.inv_cells), c = o - row * (uint32_t)cells;
  const uint32_t e = __umulhi(row, dv.inv_L), k = row - e * (uint32_t)L;
  const uint32_t cw = (uint32_t)cells >> 2;
  const uint32_t left = ((uint32_t)cells - c) >> 2;          // words left in this row (>= 1)
  const bool last = k + 1u == (uint32_t)L;
  const uint32_t i1 = e * cw + (c >> 2), i2 = (last ? e + 1u : e) * cw;
  const uint32_t ch1 = s_ch4[k], ch2 = s_ch4[last ? 0u : k + 1u];
#pragma unroll
  for (uint32_t j = 0; j < 4; ++j) {
    const bool first = j < left;
    w[j] = bytes_equal01(s32[first ? i1 + j : i2 + (j - left)], first ? ch1 : ch2);
  }
}

template <typename OutT, bool WORDS>
__global__ void __launch_bounds__(TB) k_layers(const uint8_t* __restrict__ board, OutT* __restrict__ out, CharTable ct,
                                               int L, int cells, int EB, int64_t n_boards, LayerDivisors dv) {
  extern __shared__ __align__(16) uint8_t s_board[];          // EB * cells bytes + 32 bytes of slack
  __shared__ uint32_t s_ch4[CX_MAX_CHARS];
  const int64_t b0 = (int64_t)blockIdx.x * EB;
  const int nb = (int)min((int64_t)EB, n_boards - b0);
  const int tile_bytes = nb * cells;
  const uint8_t* src = board + b0 * cells;
  if (threadIdx.x < CX_MAX_CHARS) s_ch4[threadIdx.x] = ct.ch[threadIdx.x] * 0x01010101u;
  if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
    const uint4* s16 = reinterpret_cast<const uint4*>(src);
    uint4* d16 = reinterpret_cast<uint4*>(s_board);
    for (int i = threadIdx.x; i < tile_bytes / 16; i += TB) d16[i] = __ldcs(s16 + i);
    for (int i = (tile_bytes & ~15) + threadIdx.x; i < tile_bytes; i += TB) s_board[i] = src[i];
  } else {
    for (int i = threadIdx.x; i < tile_bytes; i += TB) s_board[i] = src[i];
  }
  if (threadIdx.x < 32) s_board[tile_bytes + threadIdx.x] = 0;  // the 4-byte windows may read past the last board
  __syncthreads();
  const int per = L * cells;
  const int total = nb * per;                   // output elements of this CTA (< 2^31)
  OutT* dst = out + b0 * per;
  const bool vec = (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
  for (int o = threadIdx.x * 16; o < total; o += TB * 16) {   // 16 cells per thread and iteration
    uint32_t w[4];
    if (WORDS) {
      layer_words16(reinterpret_cast<const uint32_t*>(s_board), s_ch4, L, cells, dv, (uint32_t)o, w);
    } else {
      LayerCursor cur;
      cur.e = dv.inv_per ? (int)__umulhi((uint32_t)o, dv.inv_per) : o / per;
      const int rem = o - cur.e * per;
      cur.k = dv.inv_per ? (int)__umulhi((uint32_t)rem, dv.inv_cells) : rem / cells;
      cur.c = rem - cur.k * cells;
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = layer_word(s_board, s_ch4, L, cells, cur);
    }
    if (sizeof(OutT) == 1) {
      uint8_t* d8 = reinterpret_cast<uint8_t*>(dst) + o;
      if (vec && o + 16 <= total) {
        __stcs(reinterpret_cast<uint4*>(d8), make_uint4(w[0], w[1], w[2], w[3]));
      } else {
        for (int j = 0; j < 16 && o + j < total; ++j) d8[j] = (uint8_t)(w[j >> 2] >> (8 * (j & 3)));
      }
    } else {
      float* df = reinterpret_cast<float*>(dst) + o;
      if (vec && o + 16 <= total) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          __stcs(reinterpret_cast<float4*>(df) + j,
                 make_float4((float)(w[j] & 1u), (float)((w[j] >> 8) & 1u), (float)((w[j] >> 16) & 1u),
                             (float)(w[j] >> 24)));
      } else {
        for (int j = 0; j < 16 && o + j < total; ++j) df[j] = (float)((w[j >> 2] >> (8 * (j & 3))) & 1u);
      }
    }
  }
}

// float32 output, boards whose rows are whole 4-byte words (cells % 4 == 0; Hello World: 468): one thread owns one
// 16-byte group of the FLAT output (4 cells of one (board, channel) row, which never straddles rows), so a warp
// store is one aligned 512-byte run of whole lines; (board, channel, word) come from two multiplications with
// precomputed inverses, the board word from a cached load (each is read once per channel), the compare is a
// branch-free zero-byte test.
template <typename OutT>
__global__ void __launch_bounds__(TB) k_layers_words(const uint32_t* __restrict__ board, OutT* __restrict__ out,
                                                     CharTable ct, int L, int cw, int EB, int64_t n_boards,
                                                     uint32_t inv_cw, uint32_t inv_L) {
  static_assert(sizeof(OutT) == 4, "float32 layered boards");
  __shared__ uint32_t s_ch4[CX_MAX_CHARS];
  if (threadIdx.x < CX_MAX_CHARS) s_ch4[threadIdx.x] = ct.ch[threadIdx.x] * 0x01010101u;
  __syncthreads();
  const int64_t b0 = (int64_t)blockIdx.x * EB;
  const int nb = (int)min((int64_t)EB, n_boards - b0);
  const uint32_t* src = board + b0 * cw;
  float4* dst4 = reinterpret_cast<float4*>(out + b0 * L * cw * 4);
  const uint32_t total = (uint32_t)nb * (uint32_t)L * (uint32_t)cw;   // 16-byte output groups of this CTA
#pragma unroll 4
  for (uint32_t i = threadIdx.x; i < total; i += TB) {
    // exact: i * cw < 2^32 and row * L < 2^32 (EB * cells <= 32 KB, L <= CX_MAX_CHARS)
    const uint32_t row = __umulhi(i, inv_cw), q = i - row * (uint32_t)cw;
    const uint32_t e = L == 1 ? row : __umulhi(row, inv_L), k = row - e * (uint32_t)L;
    const uint32_t m = bytes_equal01(src[e * (uint32_t)cw + q], s_ch4[k]);   // re-read once per channel: L1 hits
    __stcs(dst4 + i, make_float4((float)(m & 1u), (float)((m >> 8) & 1u), (float)((m >> 16) & 1u), (float)(m >> 24)));
  }
}

// float32 output, any board size: one thread owns one 16-byte group of the FLAT output = 4 consecutive cells of the
// [board, channel, cell] order (they may run over the end of a row), so warp stores are aligned 512-byte runs here
// too.  The cursor (board, channel, cell) comes from two inverse multiplications and advances cell by cell; board
// bytes are staged in shared memory.
__global__ void __launch_bounds__(TB) k_layers_cells_f32(const uint8_t* __restrict__ board, float* __restrict__ out,
                                                         CharTable ct, int L, int cells, int EB, int64_t n_boards,
                                                         uint32_t inv_cells, uint32_t inv_L) {
  extern __shared__ __align__(16) uint8_t s_board[];          // EB * cells bytes
  __shared__ uint8_t s_ch[CX_MAX_CHARS];
  const int64_t b0 = (int64_t)blockIdx.x * EB;
  const int nb = (int)min((int64_t)EB, n_boards - b0);
  const int tile_bytes = nb * cells;
  const uint8_t* src = board + b0 * cells;
  if (threadIdx.x < CX_MAX_CHARS) s_ch[threadIdx.x] = ct.ch[threadIdx.x];
  if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
    const uint4* s16 = reinterpret_cast<const uint4*>(src);
    uint4* d16 = reinterpret_cast<uint4*>(s_board);
    for (int i = threadIdx.x; i < tile_bytes / 16; i += TB) d16[i] = __ldcs(s16 + i);
    for (int i = (tile_bytes & ~15) + threadIdx.x; i < tile_bytes; i += TB) s_board[i] = src[i];
  } else {
    for (int i = threadIdx.x; i < tile_bytes; i += TB) s_board[i] = src[i];
  }
  __syncthreads();
  const uint32_t total = (uint32_t)nb * (uint32_t)L * (uint32_t)cells;   // output elements of this CTA
  float* dst = out + b0 * L * cells;
#pragma unroll 2
  for (uint32_t f = threadIdx.x * 4u; f < total; f += TB * 4u) {
    // exact: f * cells < 2^32 and row * L < 2^32 (checked by the launcher)
    const uint32_t row = __umulhi(f, inv_cells);
    uint32_t c = f - row * (uint32_t)cells;
    const uint32_t e = L == 1 ? row : __umulhi(row, inv_L);
    uint32_t k = row - e * (uint32_t)L, base = e * (uint32_t)cells;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[j] = (f + j < total && s_board[base + c] == s_ch[k]) ? 1.0f : 0.0f;
      if (++c == (uint32_t)cells) {
        c = 0;
        if (++k == (uint32_t)L) {
          k = 0;
          base += cells;
        }
      }
    }
    if (f + 4u <= total) {
      __stcs(reinterpret_cast<float4*>(dst + f), make_float4(v[0], v[1], v[2], v[3]));
    } else {
      for (uint32_t j = 0; f + j < total; ++j) dst[f + j] = v[j];
    }
  }
}

// boards narrower than 4 cells: one element per thread (never on a hot path)
template <typename OutT>
__global__ void k_layers_tiny(const uint8_t* __restrict__ board, OutT* __restrict__ out, CharTable ct, int L, int cells,
                              int64_t n_boards) {
  const int64_t total = n_boards * L * cells;
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= total) return;
  const int per = L * cells;
  const int64_t e = i / per;
  const int rem = (int)(i - e * per);
  const int k = rem / cells, c = rem - k * cells;
  out[i] = (OutT)(board[e * cells + c] == ct.ch[k] ? 1 : 0);
}

// boards per CTA: a multiple of 16 (so that every CTA's input and output tiles start 16-byte aligned) with at
// most 64 KB of boards in shared memory (cells <= 4096)
inline int layers_boards_per_cta(int cells) {
  int eb = (32 * 1024 / cells) / 16 * 16;   // <= 32 KB of boards per CTA (64 KB for the largest boards) ...
  if (eb > 256) eb = 256;                   // ... in fat CTAs: the per-CTA set-up is amortised over >= 40 KB of output
  return eb < 16 ? 16 : eb;
}

template <typename OutT>
int launch_layers(const cx_game* g, const uint8_t* d_board, int64_t n_boards, OutT* d_out, cudaStream_t s) {
  static CxPerDevice configured;
  if (configured.need()) {
    CX_CUDA_OK(cudaFuncSetAttribute(k_layers<OutT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65 * 1024));
    CX_CUDA_OK(cudaFuncSetAttribute(k_layers<OutT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65 * 1024));
    configured.mark();
  }
  CharTable ct;
  memcpy(ct.ch, g->desc.chars, CX_MAX_CHARS);
  const int cells = g->info.cells, EB = layers_boards_per_cta(cells);
  const int64_t grid = (n_boards + EB - 1) / EB;
  if (grid > 0x7fffffff) {
    cx_set_error("cx_layers_from_board: too many boards for one launch");
    return CX_ERR_INVALID_ARG;
  }
  if (cells < 4) {
    const int64_t total = n_boards * g->info.n_chars * cells;
    k_layers_tiny<OutT><<<blocks_for(total), TB, 0, s>>>(d_board, d_out, ct, g->info.n_chars, cells, n_boards);
    CX_CUDA_OK(cudaGetLastError());
    return CX_OK;
  }
  // float32: one board word per thread, 16-byte stores (every (board, channel) row starts 16-byte aligned)
  if (sizeof(OutT) == 4 && cells % 4 == 0 && (reinterpret_cast<uintptr_t>(d_board) & 3) == 0 &&
      (reinterpret_cast<uintptr_t>(d_out) & 15) == 0) {
    const int cw = cells / 4;
    const uint32_t inv_cw = cw == 1 ? 0u : 0xFFFFFFFFu / (uint32_t)cw + 1u;
    if (cw > 1) {
      const int Lc = g->info.n_chars;
      const uint32_t inv_Lc = Lc == 1 ? 0u : 0xFFFFFFFFu / (uint32_t)Lc + 1u;
      k_layers_words<float><<<(unsigned)grid, TB, 0, s>>>(reinterpret_cast<const uint32_t*>(d_board),
                                                           reinterpret_cast<float*>(d_out), ct, Lc, cw, EB, n_boards,
                                                           inv_cw, inv_Lc);
      CX_CUDA_OK(cudaGetLastError());
      return CX_OK;
    }
  }
  const size_t smem = ((size_t)EB * cells + 15) / 16 * 16 + 32;
  const int L = g->info.n_chars;
  if (sizeof(OutT) == 4 && cells > 1 && (reinterpret_cast<uintptr_t>(d_out) & 15) == 0 &&
      (uint64_t)EB * L * cells * (uint64_t)cells < (1ull << 32)) {
    static CxPerDevice configured_cells;
    if (configured_cells.need()) {
      CX_CUDA_OK(cudaFuncSetAttribute(k_layers_cells_f32, cudaFuncAttributeMaxDynamicSharedMemorySize, 65 * 1024));
      configured_cells.mark();
    }
    k_layers_cells_f32<<<(unsigned)grid, TB, smem, s>>>(d_board, reinterpret_cast<float*>(d_out), ct, L, cells, EB, n_boards,
                                                        (uint32_t)(0xFFFFFFFFu / (uint32_t)cells + 1u),
                                                        L == 1 ? 0u : (uint32_t)(0xFFFFFFFFu / (uint32_t)L + 1u));
    CX_CUDA_OK(cudaGetLastError());
    return CX_OK;
  }
  // word path: rows of whole words, and the inverses exact for every output offset of a CTA (x * d < 2^32)
  const bool words = cells % 4 == 0 && cells >= 16 && L > 1 && (uint64_t)EB * L * cells * (uint64_t)cells < (1ull << 32);
  LayerDivisors dv;
  dv.inv_cells = (uint32_t)(0xFFFFFFFFu / (uint32_t)cells + 1u);
  dv.inv_L = L == 1 ? 0u : (uint32_t)(0xFFFFFFFFu / (uint32_t)L + 1u);
  const uint64_t per = (uint64_t)L * cells;   // x / d == umulhi(x, ceil(2^32 / d)) while x * d < 2^32
  dv.inv_per = (cells > 1 && per > 1 && (uint64_t)EB * per * per < (1ull << 32)) ? (uint32_t)(0xFFFFFFFFu / (uint32_t)per + 1u) : 0u;
  if (words)
    k_layers<OutT, true><<<(unsigned)grid, TB, smem, s>>>(d_board, d_out, ct, L, cells, EB, n_boards, dv);
  else
    k_layers<OutT, false><<<(unsigned)grid, TB, smem, s>>>(d_board, d_out, ct, L, cells, EB, n_boards, dv);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

__global__ void k_onehot_to_index(const float* __restrict__ onehot, int A, uint8_t* __restrict__ idx,
                                  int32_t* bad, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n) return;
  int best = 0, ones = 0, others = 0;
  float bestv = -INFINITY;
  for (int a = 0; a < A; ++a) {
    const float v = onehot[i * A + a];
    if (v > bestv) {
      bestv = v;
      best = a;
    }
    if (v == 1.0f)
      ++ones;
    else if (v != 0.0f)
      ++others;
  }
  // a row that is not exactly one-hot is not an action (boat_race.py:48 `assert sum(act) == 1`): index 255 makes
  // the step kernels leave that env untouched and raise CX_FLAG_BAD_ACTION for it
  const bool invalid = ones != 1 || others != 0;
  idx[i] = invalid ? (uint8_t)255 : (uint8_t)best;
  if (invalid && bad) atomicAdd(bad, 1);
}

__global__ void k_fill_actions(uint64_t seed, uint64_t env_offset, uint64_t t0, int32_t T, int64_t n, int32_t A,
                               uint8_t* out) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= (int64_t)T * n) return;
  const int64_t t = i / n, e = i - t * n;
  out[i] = (uint8_t)cx_synth_action(seed, env_offset + (uint64_t)e, t0 + (uint64_t)t, (uint32_t)A);
}

// the same stream, one Philox call per QUAD of envs (its four words serve envs 4q .. 4q+3) and one 4-byte store:
// env_offset and n multiples of 4, output 4-byte aligned
__global__ void k_fill_actions_quads(uint64_t seed, uint64_t env_offset, uint64_t t0, int32_t T, int64_t n, int32_t A,
                                     uint8_t* out) {
  const int64_t nq = n >> 2, i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= (int64_t)T * nq) return;
  const int64_t t = i / nq, q = i - t * nq;
  reinterpret_cast<uint32_t*>(out)[i] =
      cx_synth_actions_quad(seed, (env_offset >> 2) + (uint64_t)q, t0 + (uint64_t)t, (uint32_t)A);
}

// examples/actor_critic.py:90-98: `m = Categorical(probs); action = m.sample()`.  Inverse-CDF sampling, one thread
// per env: u from the counter-based Philox stream (reproducible per (seed, env, step), independent of the launch
// geometry), the first action whose cumulative weight exceeds u * total.  With logits the weights are
// exp(l - max l) -- the softmax the policy head would otherwise run as its own kernel.
__global__ void k_sample_actions(const float* __restrict__ scores, int64_t n, int A, int is_logits, uint64_t seed,
                                 uint64_t env_offset, const uint64_t* __restrict__ d_step, uint64_t step_offset,
                                 uint8_t* __restrict__ actions, float* __restrict__ logp) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n) return;
  float w[CX_MAX_ACTIONS];
#pragma unroll
  for (int a = 0; a < CX_MAX_ACTIONS; ++a) w[a] = a < A ? scores[i * A + a] : 0.0f;
  float lp;
  const int pick = sample_categorical(w, A, is_logits, seed, env_offset + (uint64_t)i,
                                      (d_step ? *d_step : 0ull) + step_offset, &lp);
  actions[i] = (uint8_t)pick;
  if (logp) logp[i] = lp;
}

// The reference's policy head evaluated and sampled in ONE launch (examples/actor_critic.py:64-98: affine1 -> relu ->
// action_head -> softmax -> Categorical.sample()).  At the 4,096 envs of BASELINE config 5 an env-batch step is
// launch-bound; this kernel replaces four launches (two GEMMs, ReLU, sampling) of the rollout loop.
// A CTA of eight warps owns 32 envs, lane = env.  Both operands are staged once with 16-byte loads that are all in
// flight together: the CTA's input rows (one contiguous [32, n_in] block) transposed into xs[d][env] (row pitch 33:
// conflict-free both ways) and W1^T [n_in, 32] as it lies in memory.  Warp w then accumulates hidden units 4w..4w+3
// for its 32 envs: per input one LDS.32 of x and one broadcast LDS.128 of weights feed 4 FFMA (a first version with
// lane = hidden unit re-read the whole 22 KB weight tile per env and staged it transposed inside the kernel: 11.3 us
// per launch at 4,096 envs), multiplies relu(h) into its share of every action logit and leaves the shares in shared
// memory; warp 0 adds them up in warp order and samples, one lane per env, from the same Philox stream and with the
// same arithmetic as cx_sample_actions.  The small operands (b1, W2, b2, the step counter) are requested before the
// tiles so that no load waits behind another.
__global__ void __launch_bounds__(POLICY_THREADS)
    k_policy_sample(const float* __restrict__ x, int64_t n, int n_in, const float* __restrict__ w1t,
                    const float* __restrict__ b1, int n_hidden, const float* __restrict__ w2, const float* __restrict__ b2,
                    int A, uint64_t seed, uint64_t env_offset, const uint64_t* __restrict__ d_step, uint64_t step_offset,
                    uint8_t* __restrict__ actions, float* __restrict__ logp, float* __restrict__ logits_out) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  float* s_w = reinterpret_cast<float*>(smem_raw);             // [n_in][32]  W1^T, hidden units padded to 32 with zeros
  float* s_x = s_w + (size_t)n_in * 32;                        // [n_in][33]  inputs of the CTA's envs, transposed
  float* s_h = s_x + (size_t)n_in * POLICY_PITCH;              // [8 warps][CX_MAX_ACTIONS][33]  the warps' shares of the logits
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t e0 = (int64_t)blockIdx.x * 32;
  const int n_here = (int)min((int64_t)32, n - e0);
  // the small operands first, so that their latency hides behind the tiles'
  const PolicyRegs R = policy_load_small(b1, w2, b2, n_hidden, A, warp, lane);
  const uint64_t step = (d_step ? *d_step : 0ull) + step_offset;
  // ---- staging: every thread requests up to 8 + 8 float4 (weights, inputs) before it stores any of them, so one
  // round of memory latency covers both operands for n_in <= 256 (a loop of load -> store pays it per iteration) ----
  const float* blk = x + e0 * n_in;                            // [n_here][n_in], contiguous
  const int total = n_here * n_in;
  const uint32_t inv = 0xFFFFFFFFu / (uint32_t)n_in + 1u;      // k / n_in by multiplication (k * n_in < 2^32); wraps
                                                               // to 0 for n_in == 1, where k / n_in is k
  const bool w_vec = n_hidden == 32 && (reinterpret_cast<uintptr_t>(w1t) & 15) == 0;
  const bool x_vec = (reinterpret_cast<uintptr_t>(blk) & 15) == 0;
  const int w_q = w_vec ? n_in * 8 : 0, x_q = x_vec ? total / 4 : 0;   // float4 counts on the vector paths
  constexpr int DEPTH = 8;
  for (int base = tid; base < max(w_q, x_q); base += DEPTH * POLICY_THREADS) {
    float4 vw[DEPTH], vx[DEPTH];
#pragma unroll
    for (int u = 0; u < DEPTH; ++u) {
      const int q = base + u * POLICY_THREADS;
      if (q < w_q) vw[u] = __ldg(reinterpret_cast<const float4*>(w1t) + q);
      if (q < x_q) vx[u] = __ldcs(reinterpret_cast<const float4*>(blk) + q);
    }
#pragma unroll
    for (int u = 0; u < DEPTH; ++u) {
      const int q = base + u * POLICY_THREADS;
      if (q < w_q) reinterpret_cast<float4*>(s_w)[q] = vw[u];
      if (q < x_q) {
        const float vv[4] = {vx[u].x, vx[u].y, vx[u].z, vx[u].w};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint32_t k = 4u * q + c, e = n_in == 1 ? k : __umulhi(k, inv), d = k - e * (uint32_t)n_in;
          s_x[d * POLICY_PITCH + e] = vv[c];
        }
      }
    }
  }
  if (!w_vec)
    for (int k = tid; k < n_in * 32; k += POLICY_THREADS) {
      const int d = k >> 5, j = k & 31;
      s_w[k] = j < n_hidden ? __ldg(w1t + (size_t)d * n_hidden + j) : 0.0f;
    }
  for (int k = (x_vec ? (total & ~3) : 0) + tid; k < total; k += POLICY_THREADS) {
    const uint32_t e = n_in == 1 ? (uint32_t)k : __umulhi((uint32_t)k, inv), d = (uint32_t)k - e * (uint32_t)n_in;
    s_x[d * POLICY_PITCH + e] = __ldcs(blk + k);
  }
  if (n_here < 32)                                             // lanes without an env compute on zeros
    for (int k = tid; k < n_in * (32 - n_here); k += POLICY_THREADS) {
      const int d = k / (32 - n_here), e = n_here + k - d * (32 - n_here);
      s_x[d * POLICY_PITCH + e] = 0.0f;
    }
  __syncthreads();
  policy_hidden_shares(s_w, s_x, s_h, n_in, A, R, warp, lane);
  __syncthreads();
  // ---- sum the eight shares in warp order, add b2, sample: warp 0, lane = env ----
  if (warp == 0) {
    float w[CX_MAX_ACTIONS];
    policy_logits(s_h, R, A, lane, w);
    if (lane < n_here) {
      const int64_t i = e0 + lane;
      if (logits_out) {
#pragma unroll
        for (int a = 0; a < CX_MAX_ACTIONS; ++a)
          if (a < A) logits_out[i * A + a] = w[a];
      }
      float lp;
      const int pick = sample_categorical(w, A, 1, seed, env_offset + (uint64_t)i, step, &lp);
      actions[i] = (uint8_t)pick;
      if (logp) logp[i] = lp;
    }
  }
}

// examples/actor_critic.py:119-122: `R = r + gamma * R` backwards; one thread per env, coalesced over envs
__global__ void k_discounted_returns(const float* __restrict__ reward, const float* __restrict__ discount,
                                     const uint8_t* __restrict__ flags, const float* __restrict__ bootstrap, int T,
                                     int64_t n, float gamma, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n) return;
  float g = bootstrap ? bootstrap[i] : 0.0f;
  for (int t = T - 1; t >= 0; --t) {
    const int64_t k = (int64_t)t * n + i;
    const bool ended = flags[k] & (CX_FLAG_TERMINATED | CX_FLAG_TRUNCATED);
    const float c = ended ? 0.0f : (discount ? discount[k] : 1.0f);
    g = __fmaf_rn(__fmul_rn(gamma, c), g, reward[k]);
    out[k] = g;
  }
}

__global__ void k_step_perf(const uint8_t* __restrict__ region, int cells, int n_regions,
                            const int32_t* __restrict__ prev, const int32_t* __restrict__ next, float* perf,
                            int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n) return;
  const int p = prev[i], q = next[i];
  if (p < 0 || q < 0 || p >= cells || q >= cells) return;
  perf[i] += (float)cx_perf_step(region[p], region[q], n_regions);
}

}  // namespace

int cx_launch_stats_fold(void* d_state, cudaStream_t s) {
  k_stats_fold<<<1, TB, 0, s>>>(static_cast<double*>(d_state));   // off_stats == 0
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

int cx_launch_reset(const cx_game* g, void* d_state, int64_t n, const uint8_t* d_mask, cudaStream_t s) {
  const CxStateLayout L = cx_layout(g, n);
  uint8_t* base = static_cast<uint8_t*>(d_state);
  uint16_t* tstep = reinterpret_cast<uint16_t*>(base + L.off_tstep);
  float* ret = reinterpret_cast<float*>(base + L.off_ret);
  if (!d_mask)
    k_stats_init<<<blocks_for((1 + CX_STAT_STRIPES) * CX_STATS_DOUBLES), TB, 0, s>>>(reinterpret_cast<double*>(base + L.off_stats));
  if (g->path == CX_PATH_AGENT) {
    float* perf = g->info.tracks_performance ? reinterpret_cast<float*>(base + L.off_perf) : nullptr;
    uint64_t* pick = g->info.n_pickups ? reinterpret_cast<uint64_t*>(base + L.off_pick) : nullptr;
    k_agent_reset<<<blocks_for(n), TB, 0, s>>>(base + L.off_dyn, tstep, ret, perf, pick, g->ph.all, g->info.tracks,
                                               g->ah.init_cell, d_mask, n);
  } else {
    GenInit gi;
    memset(&gi, 0, sizeof(gi));
    gi.n_dyn = g->gh.n_dyn;
    memcpy(gi.init, g->gh.slot_init, sizeof(gi.init));
    k_generic_reset<<<blocks_for(n), TB, 0, s>>>(reinterpret_cast<uint16_t*>(base + L.off_dyn), tstep, ret,
                                                 g->info.tracks, gi, d_mask, n);
    if (g->gh.has_dynbd)
      k_dynbd_reset<<<blocks_for(n * g->gh.cells), TB, 0, s>>>(base + L.off_dynbd, g->d_blob + g->gh.off_backdrop,
                                                               g->gh.cells, d_mask, n);
  }
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

int cx_launch_render(const cx_game* g, const void* d_state, int64_t n, uint8_t* d_board, cudaStream_t s) {
  if (g->path != CX_PATH_AGENT) return cx_launch_generic_render(g, d_state, n, d_board, s);
  const CxStateLayout L = cx_layout(g, n);
  const uint8_t* base = static_cast<const uint8_t*>(d_state);
  const uint8_t* pk = g->d_blob + g->ph.off;
  k_agent_render<<<blocks_for(n * g->ah.cells), TB, 0, s>>>(
      base + L.off_dyn, g->d_blob + g->ah.off_basech, g->d_blob + g->ah.off_shown, g->ah.cells, g->ah.agent_char, d_board,
      n, g->info.n_pickups ? reinterpret_cast<const uint64_t*>(base + L.off_pick) : nullptr, pk + g->ph.item_at,
      reinterpret_cast<const CxPickItem*>(pk + g->ph.items), g->ph);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

static int dyn_slot_of(const cx_game* g, int z) { return g->gh.ent[z].dyn_slot; }

int cx_launch_get_entity(const cx_game* g, const void* d_state, int64_t n, int32_t z, int32_t* d_out,
                         cudaStream_t s) {
  const CxStateLayout L = cx_layout(g, n);
  const uint8_t* base = static_cast<const uint8_t*>(d_state);
  const int kind = g->desc.entities[z].kind;
  if (kind == CX_KIND_STATIC || kind == CX_KIND_PICKUP || kind == CX_KIND_DOOR) {
    cx_set_error("cx_get_entity_state: entity %d is static, a pickup or a door drape", z);
    return CX_ERR_INVALID_ARG;
  }
  if (g->path == CX_PATH_AGENT) {
    k_get_agent<<<blocks_for(n), TB, 0, s>>>(base + L.off_dyn, d_out, g->ah.cells, n);
  } else {
    const uint16_t* dyn = reinterpret_cast<const uint16_t*>(base + L.off_dyn) + (int64_t)dyn_slot_of(g, z) * n;
    k_get_generic<<<blocks_for(n), TB, 0, s>>>(dyn, d_out, kind == CX_KIND_ROLL, g->gh.cols, n);
  }
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

int cx_launch_set_entity(const cx_game* g, void* d_state, int64_t n, int32_t z, const int32_t* d_in,
                         cudaStream_t s) {
  const CxStateLayout L = cx_layout(g, n);
  uint8_t* base = static_cast<uint8_t*>(d_state);
  const int kind = g->desc.entities[z].kind;
  if (g->path == CX_PATH_AGENT && kind == CX_KIND_SPRITE) {
    k_set_agent_sprite<<<blocks_for(n), TB, 0, s>>>(base + L.off_dyn, d_in, g->ah.cells, n);
  } else if (g->path == CX_PATH_AGENT) {
    k_set_agent<<<blocks_for(n), TB, 0, s>>>(base + L.off_dyn, d_in, g->ah.cells, n);
  } else {
    uint16_t* dyn = reinterpret_cast<uint16_t*>(base + L.off_dyn) + (int64_t)dyn_slot_of(g, z) * n;
    k_set_generic<<<blocks_for(n), TB, 0, s>>>(dyn, d_in, kind == CX_KIND_ROLL, kind == CX_KIND_CELL, g->gh.cols,
                                               g->gh.cells, n);
  }
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

namespace {
__global__ void k_get_render_state(const uint16_t* dyn, int64_t n, int n_ent, int slot_vis, int slot_zperm,
                                   int slot_bd, uint32_t static_vis, int cols, uint32_t* zorder, uint32_t* visible,
                                   int32_t* bd_off) {
  const int64_t i = (int64_t)blockIdx.x * TB + threadIdx.x;
  if (i >= n) return;
  if (zorder) {
    uint32_t perm = 0;
    if (slot_zperm >= 0) {
      perm = (uint32_t)dyn[(int64_t)slot_zperm * n + i] | ((uint32_t)dyn[(int64_t)(slot_zperm + 1) * n + i] << 16);
      if (n_ent < 8) perm &= (1u << (4 * n_ent)) - 1u;
    } else {
      for (int p = 0; p < n_ent && p < 8; ++p) perm |= (uint32_t)p << (4 * p);
    }
    zorder[i] = perm;
  }
  if (visible) visible[i] = slot_vis >= 0 ? dyn[(int64_t)slot_vis * n + i] : static_vis;
  if (bd_off) {
    const uint32_t s = slot_bd >= 0 ? dyn[(int64_t)slot_bd * n + i] : 0u;
    bd_off[i] = (int32_t)((s >> 8) * cols + (s & 255u));
  }
}
}  // namespace

int cx_launch_get_render_state(const cx_game* g, const void* d_state, int64_t n, uint32_t* d_zorder,
                               uint32_t* d_visible, int32_t* d_backdrop_off, cudaStream_t s) {
  const CxStateLayout L = cx_layout(g, n);
  const uint8_t* base = static_cast<const uint8_t*>(d_state);
  uint32_t static_vis = 0;
  for (int z = 0; z < g->desc.n_entities; ++z)
    if (g->desc.entities[z].kind == CX_KIND_SPRITE && g->desc.entities[z].visible) static_vis |= 1u << z;
  const bool gen = g->path == CX_PATH_GENERIC;
  k_get_render_state<<<blocks_for(n), TB, 0, s>>>(
      reinterpret_cast<const uint16_t*>(base + L.off_dyn), n, g->desc.n_entities, gen ? g->gh.slot_vis : -1,
      gen ? g->gh.slot_zperm : -1, gen ? g->gh.slot_bd : -1, static_vis, g->desc.cols, d_zorder, d_visible,
      d_backdrop_off);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

int cx_launch_get_episode(const cx_game* g, const void* d_state, int64_t n, int32_t* d_steps, float* d_ret,
                          cudaStream_t s) {
  const CxStateLayout L = cx_layout(g, n);
  const uint8_t* base = static_cast<const uint8_t*>(d_state);
  k_get_episode<<<blocks_for(n), TB, 0, s>>>(reinterpret_cast<const uint16_t*>(base + L.off_tstep),
                                             reinterpret_cast<const float*>(base + L.off_ret), d_steps, d_ret, n);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

extern "C" int cx_layers_from_board(const cx_game* g, const uint8_t* d_board, int64_t n_boards, uint8_t* d_layered,
                                    void* stream) {
  if (!g || !d_board || !d_layered || n_boards < 1) {
    cx_set_error("cx_layers_from_board: bad argument");
    return CX_ERR_INVALID_ARG;
  }
  if (g->desc.unoccluded_layers) {
    cx_set_error("cx_layers_from_board: unoccluded layers (occlusion_in_layers=False) are not a function of the board; they come from "
                 "cx_step_observations / cx_rollout_observations / cx_render_observations");
    return CX_ERR_UNSUPPORTED;
  }
  return launch_layers<uint8_t>(g, d_board, n_boards, d_layered, (cudaStream_t)stream);
}

extern "C" int cx_layers_from_board_f32(const cx_game* g, const uint8_t* d_board, int64_t n_boards, float* d_layered,
                                        void* stream) {
  if (!g || !d_board || !d_layered || n_boards < 1) {
    cx_set_error("cx_layers_from_board_f32: bad argument");
    return CX_ERR_INVALID_ARG;
  }
  if (g->desc.unoccluded_layers) {
    cx_set_error("cx_layers_from_board_f32: unoccluded layers (occlusion_in_layers=False) are not a function of the board; they come from "
                 "cx_step_observations / cx_rollout_observations / cx_render_observations");
    return CX_ERR_UNSUPPORTED;
  }
  return launch_layers<float>(g, d_board, n_boards, d_layered, (cudaStream_t)stream);
}

extern "C" int cx_onehot_to_index(const float* d_onehot, int64_t n, int32_t A, uint8_t* d_index, int32_t* d_bad,
                                  void* stream) {
  if (!d_onehot || !d_index || n < 1 || A < 1 || A > 255) {
    cx_set_error("cx_onehot_to_index: bad argument");
    return CX_ERR_INVALID_ARG;
  }
  k_onehot_to_index<<<blocks_for(n), TB, 0, (cudaStream_t)stream>>>(d_onehot, A, d_index, d_bad, n);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

extern "C" int cx_sample_actions(const float* d_scores, int64_t n, int32_t A, int32_t is_logits, uint64_t seed,
                                 uint64_t env_offset, const uint64_t* d_step, uint64_t step_offset, uint8_t* d_actions,
                                 float* d_logp, void* stream) {
  if (!d_scores || !d_actions || n < 1 || A < 1 || A > CX_MAX_ACTIONS) {
    cx_set_error("cx_sample_actions: bad argument (n_actions must be in 1..%d)", CX_MAX_ACTIONS);
    return CX_ERR_INVALID_ARG;
  }
  k_sample_actions<<<blocks_for(n), TB, 0, (cudaStream_t)stream>>>(d_scores, n, A, is_logits, seed, env_offset, d_step,
                                                                   step_offset, d_actions, d_logp);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

extern "C" int cx_policy_sample(const float* d_x, int64_t n, int32_t n_in, const float* d_w1t, const float* d_b1,
                                int32_t n_hidden, const float* d_w2, const float* d_b2, int32_t A, uint64_t seed,
                                uint64_t env_offset, const uint64_t* d_step, uint64_t step_offset, uint8_t* d_actions,
                                float* d_logp, float* d_logits, void* stream) {
  if (!d_x || !d_w1t || !d_b1 || !d_w2 || !d_b2 || !d_actions || n < 1 || n_in < 1 || A < 1 || A > CX_MAX_ACTIONS ||
      n_hidden < 1 || n_hidden > 32) {
    cx_set_error("cx_policy_sample: bad argument (n_hidden must be in 1..32, n_actions in 1..%d)", CX_MAX_ACTIONS);
    return CX_ERR_INVALID_ARG;
  }
  const size_t smem = ((size_t)n_in * (32 + POLICY_PITCH) + (POLICY_THREADS / 32) * CX_MAX_ACTIONS * POLICY_PITCH) * sizeof(float);
  if (smem > 200 * 1024 || (int64_t)n_in * 32 >= (1ll << 31) / n_in) {
    cx_set_error("cx_policy_sample: n_inputs %d too large for the shared-memory tiles", n_in);
    return CX_ERR_UNSUPPORTED;
  }
  static CxPerDevice configured;
  if (configured.need()) {
    CX_CUDA_OK(cudaFuncSetAttribute(k_policy_sample, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    configured.mark();
  }
  const int64_t grid = (n + 31) / 32;
  if (grid > 0x7fffffff) {
    cx_set_error("cx_policy_sample: too many environments for one launch");
    return CX_ERR_INVALID_ARG;
  }
  k_policy_sample<<<(unsigned)grid, POLICY_THREADS, smem, (cudaStream_t)stream>>>(d_x, n, n_in, d_w1t, d_b1, n_hidden, d_w2,
                                                                                  d_b2, A, seed, env_offset, d_step,
                                                                                  step_offset, d_actions, d_logp, d_logits);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

extern "C" int cx_fill_actions(uint64_t seed, uint64_t env_offset, uint64_t t0, int32_t T, int64_t n, int32_t A,
                               uint8_t* d_out, void* stream) {
  if (!d_out || n < 1 || T < 1 || A < 1 || A > 255) {
    cx_set_error("cx_fill_actions: bad argument");
    return CX_ERR_INVALID_ARG;
  }
  if ((env_offset & 3) == 0 && (n & 3) == 0 && (reinterpret_cast<uintptr_t>(d_out) & 3) == 0)
    k_fill_actions_quads<<<blocks_for((int64_t)T * (n >> 2)), TB, 0, (cudaStream_t)stream>>>(seed, env_offset, t0, T, n,
                                                                                          A, d_out);
  else
    k_fill_actions<<<blocks_for((int64_t)T * n), TB, 0, (cudaStream_t)stream>>>(seed, env_offset, t0, T, n, A, d_out);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

extern "C" int cx_discounted_returns(const float* d_reward, const float* d_discount, const uint8_t* d_flags,
                                     const float* d_bootstrap, int32_t T, int64_t n, float gamma, float* d_returns,
                                     void* stream) {
  if (!d_reward || !d_flags || !d_returns || T < 1 || n < 1) {
    cx_set_error("cx_discounted_returns: bad argument");
    return CX_ERR_INVALID_ARG;
  }
  k_discounted_returns<<<blocks_for(n), TB, 0, (cudaStream_t)stream>>>(d_reward, d_discount, d_flags, d_bootstrap, T,
                                                                       n, gamma, d_returns);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

extern "C" int cx_step_perf(const uint8_t* d_region, int32_t cells, int32_t n_regions, const int32_t* d_prev,
                            const int32_t* d_next, int64_t n, float* d_perf, void* stream) {
  if (!d_region || !d_prev || !d_next || !d_perf || n < 1 || cells < 1 || n_regions < 2) {
    cx_set_error("cx_step_perf: bad argument");
    return CX_ERR_INVALID_ARG;
  }
  k_step_perf<<<blocks_for(n), TB, 0, (cudaStream_t)stream>>>(d_region, cells, n_regions, d_prev, d_next, d_perf, n);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}
