// dibr_b200.cu — hand-written sm_100a kernels + C ABI (include/dibr_b200.h) for
// Kaolin's DIB-R hot path.  See DESIGN.md for the data layout and the roofline
// of each kernel.  Reference behaviour being reproduced:
//   kaolin/csrc/render/mesh/rasterization_cuda.cu   (forward :43-192, backward :238-402)
//   kaolin/csrc/render/mesh/dibr_soft_mask_cuda.cu  (forward :27-184, backward :230-353)
//   kaolin/render/mesh/rasterization.py:273-371, kaolin/render/mesh/dibr.py:29-73
//
// Pipeline (forward):
//   bin_faces<count> -> scan_bins -> bin_faces<fill> -> dibr_tile_fwd_kernel
//   -> soft_enum_kernel -> soft_eval_kernel (-> soft_tiles_fwd_kernel for leftovers)
//   * every face is turned into the exact integer pixel rectangle of the
//     reference's float bbox test and inserted (<= 4 entries) into the finest
//     level of a 16/64/256/... px bin pyramid where it spans <= 2x2 bins;
//   * one CTA per 16x16 screen tile streams the (<= 6) bins above it into
//     shared memory with TMA bulk copies (cp.async.bulk + mbarrier, double
//     buffered), culls them against the tile, stages the surviving face records,
//     transposes their rectangle masks into per-column/row candidate bit words and
//     lets each thread (one pixel) walk exactly its own rectangle hits;
//   * tiles with uncovered pixels under an enlarged (boxlen) rectangle are filed in
//     a work list; for them the first knum faces by index of every uncovered pixel
//     are enumerated (integer work), evaluated densely — one thread per
//     (pixel, face) pair — and folded per pixel in face order.  The pairs stay in a
//     per-tile cache block for the backward pass.
// Backward: a pixel-parallel scatter with warp-level segmented reduction keyed
// on the face id (rasterize branch) and a dense stream over the cached pairs
// (soft-mask branch; tiles outside the cache are recomputed).
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <type_traits>
#include <vector>
#include <string>
#include <string.h>
#include <stdlib.h>
#include <stdint.h>

#include "../../include/dibr_b200.h"
#include "dibr_math.cuh"

namespace {

using namespace dibr;

// Any tensor pointer not DIBR_B200_ALIGNMENT-byte aligned (NULL is aligned): the kernels read and
// write caller tensors with 16-byte vector and cp.async accesses.
template <typename... P>
bool misaligned(P... p) { return ((((uintptr_t)p) | ... | (uintptr_t)0) & (DIBR_B200_ALIGNMENT - 1)) != 0; }

constexpr int kTile = 16;
constexpr int kThreads = 256;
constexpr int kChunk = 256;
constexpr int kMaxLevels = 6;   // 16 * 4^5 = 16384 px
constexpr int kSoftCap = 1024;  // soft-mask candidates sorted per pass
constexpr int kRound = 12;      // hits a pixel contributes to one pair round
constexpr int kPairCap = kThreads * kRound;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kBandRec = 24;    // ints per record of the soft-mask work list

// ---------------------------------------------------------------------------
// Scene description shared by all kernels (passed by value).
struct Scene {
  int B, H, W;
  int F;                  // faces per view (uniform) — 0 in packed mode
  const int64_t* first;   // packed mode: device (B+1) prefix of faces per view
  int64_t NF;             // faces in all views
  const float* xy;        // (NF,3,2)
  const float* z;         // (NF,3) or null
  int premultiplied;      // xy already scaled by multiplier
  const float* fnz;       // (NF) validity: value >= 0     (nullable)
  const uint8_t* valid;   // (NF) validity: non-zero       (nullable)
  const float* bbox_tight;  // (NF,4) given tight bboxes    (nullable -> min/max)
  const float* bbox_large;  // (NF,4) given enlarged bboxes (nullable -> min/max -/+ margin)
  float multiplier, margin;
  PixelGrid grid;
  int L;
  int ntx[kMaxLevels], nty[kMaxLevels], bin_base[kMaxLevels];
  int NB;                 // bins per view (all levels)
  int* cnt;               // [2][B][NB] (+ pool_ctr right behind it: one memset clears both)
  int* off;               // [2][B][NB]
  int4* entries;          // [2][4*NF]  {face, x_lo|x_hi<<16, y_lo|y_hi<<16, 0}
  // soft-mask hit cache: what the reference keeps as 13*knum bytes for EVERY pixel
  // (close_face_{prob,idx,dist_type}) is kept only for tiles that have hits
  int pool_tiles;         // capacity in tiles (0 = disabled)
  int pool_K;             // knum the blocks are sized for (block = 3 * 256*K words)
  int* pool_ctr;          // [1] blocks handed out
  int4* pool_hdr;         // [pool_tiles] {b, tx, ty, hits}
  uint32_t* pool_data;    // [pool_tiles][3][256*K]: face | prob bits | lx|ly<<4|(dist_type)<<8
  int* pool_na;           // [pool_tiles] uncovered pixels of the tile           } only when
  uint32_t* pool_aux;     // [pool_tiles][256] per such pixel: lx|ly<<4 | hits<<8 } knum <= 32:
  uint16_t* pool_slots;   // [pool_tiles][256][32] its hit slots, face order      } 3-kernel forward
  int* fb_ctr;            // [1] tiles whose hits did not fit the cache (recomputed in backward)
  int* fb_list;           // [B*nty*ntx] their linear tile ids
  int* tile_cnt;          // [B*nty*ceil(ntx/32)] bit per 16x16 tile: an enlarged face rectangle overlaps it (count pass)
  int* view_flag;         // [B] the view has an enlarged rectangle too big to count per tile
  int* band_ctr;          // [1] tiles with uncovered pixels under some enlarged face rectangle
  int* band_list;         // [B*nty*ntx][kBandRec] work list of the soft-mask kernels: per tile
                          //   {linear tile id, 8 x uncovered-pixel ballot, 6 x (large-bin offset, size), pad}
};

__host__ __device__ inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---------------------------------------------------------------------------
// Per-kernel timing for bench.py's roofline table (dibr_b200_trace_begin/_end):
// THREAD-LOCAL state, so the library stays re-entrant; when a trace is open on the
// calling thread every kernel launch is bracketed by a pair of CUDA events on the
// launch stream.  Off (the default) it costs one thread-local load per launch.
struct TraceState {
  bool on = false;
  int used = 0;
  std::vector<cudaEvent_t> pool;
  std::vector<const char*> names;
};
thread_local TraceState g_trace;

struct Span {
  cudaStream_t st;
  bool on;
  Span(const char* name, cudaStream_t st_) : st(st_), on(g_trace.on) {
    if (!on) return;
    TraceState& t = g_trace;
    while ((int)t.pool.size() < t.used + 2) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) { on = false; return; }
      t.pool.push_back(e);
    }
    t.names.push_back(name);
    cudaEventRecord(t.pool[t.used], st);
  }
  ~Span() {
    if (!on) return;
    cudaEventRecord(g_trace.pool[g_trace.used + 1], st);
    g_trace.used += 2;
  }
};

// ---------------------------------------------------------------------------
// PTX helpers: mbarrier + 1-D bulk TMA (global -> shared).
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes,
                                            unsigned long long* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---------------------------------------------------------------------------
// Face -> view lookup and face loading.
__device__ __forceinline__ void face_view(const Scene& s, int64_t i, int& b, int64_t& fbase) {
  if (s.first) {
    int lo = 0, hi = s.B;  // first[lo] <= i < first[hi]
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(s.first + mid) <= i) lo = mid; else hi = mid;
    }
    b = lo;
    fbase = __ldg(s.first + lo);
  } else {
    b = (int)(i / s.F);
    fbase = (int64_t)b * s.F;
  }
}
__device__ __forceinline__ int64_t view_fbase(const Scene& s, int b) {
  return s.first ? __ldg(s.first + b) : (int64_t)b * s.F;
}

// xy of global face g, multiplied exactly as `face_vertices_image * multiplier`
// (rasterization.py:320, dibr.py:32): one fp32 multiply per coordinate.
__device__ __forceinline__ void load_xy(const Scene& s, int64_t g, float v[6]) {
  const float2* p = reinterpret_cast<const float2*>(s.xy + g * 6);
  const float2 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y;
  if (!s.premultiplied) {
#pragma unroll
    for (int i = 0; i < 6; i++) v[i] = fmul(v[i], s.multiplier);
  }
}

// ---------------------------------------------------------------------------
// Binning: one thread per face; pass 1 counts, pass 2 fills (unordered inside a
// bin; consumers that need index order sort their culled candidates).
// Faces that are neighbours in the index buffer are neighbours on screen, so at any
// moment the whole GPU increments the same few bin counters, and same-address L2
// atomics serialise at the full read-modify-write latency (measured: ~10 us per
// returning atomic with 1.3 M faces).  The counters are therefore aggregated twice
// before they reach L2: lanes of a warp that hit the same bin are found with
// match.any, and the warp leaders merge into a per-CTA shared-memory hash table;
// one global atomic per (CTA, distinct bin) is issued by a separate thread each, so
// their round trips overlap.  The entries of a patch land contiguously.
constexpr int kBinThreadsAgg = 512;    // aggregating CTAs: big, so that a CTA merges more (measured: 256 is 35 % slower)
constexpr int kBinThreadsPlain = 256;  // plain-atomics CTAs: small (measured: 5-12 % faster than 512)
constexpr int kBinHT = 4096;           // >= kBinThreadsAgg * 8 targets: the table always fits
constexpr uint32_t kBinEmpty = 0xffffffffu;

struct BinSmem {
  uint32_t keys[kBinHT];   // counter index (set, view, bin)
  int vals[kBinHT];        // faces of this CTA in the bin; after the flush: where they go
};

struct BinSpan { int l, bx0, bx1, by0, by1; bool has; };

__device__ __forceinline__ BinSpan bin_span(const Scene& s, const PixRect& r, bool has) {
  BinSpan sp;
  sp.has = has && r.x_hi > r.x_lo && r.y_hi > r.y_lo;
  sp.l = 0; sp.bx0 = 0; sp.bx1 = -1; sp.by0 = 0; sp.by1 = -1;
  if (sp.has) {
    for (;; ++sp.l) {
      const int sh = 4 + 2 * sp.l;
      sp.bx0 = r.x_lo >> sh; sp.bx1 = (r.x_hi - 1) >> sh;
      sp.by0 = r.y_lo >> sh; sp.by1 = (r.y_hi - 1) >> sh;
      if ((sp.bx1 - sp.bx0 <= 1 && sp.by1 - sp.by0 <= 1) || sp.l == s.L - 1) break;
    }
  }
  return sp;
}

// Registers the <= 2x2 bins of one face in the CTA table; where[k] = (table slot << 16) | rank
// inside the CTA, or -1.  Called by all lanes of the warp.
__device__ __forceinline__ void bin_insert(const Scene& s, BinSmem& sm, int set, int b, const BinSpan& sp,
                                           int (&where)[4]) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int bx = sp.bx0 + (k & 1), by = sp.by0 + (k >> 1);
    const bool on = sp.has && bx <= sp.bx1 && by <= sp.by1;
    const unsigned act = __ballot_sync(kFull, on);
    where[k] = -1;
    if (!on) continue;
    const uint32_t ci = (uint32_t)((set * s.B + b) * s.NB + s.bin_base[sp.l] + by * s.ntx[sp.l] + bx);
    const unsigned peers = __match_any_sync(act, ci);
    const int leader = __ffs(peers) - 1;
    int w = 0;
    if (lane == leader) {
      uint32_t h = (ci * 2654435761u) >> 20;
      while (true) {
        const uint32_t prev = atomicCAS(&sm.keys[h], kBinEmpty, ci);
        if (prev == kBinEmpty || prev == ci) break;
        h = (h + 1) & (kBinHT - 1);
      }
      w = (int)(h << 16) | atomicAdd(&sm.vals[h], __popc(peers));
    }
    w = __shfl_sync(peers, w, leader);
    where[k] = w + __popc(peers & ((1u << lane) - 1u));
  }
}

// AGG = false (sparse meshes, a few faces per tile): plain atomics, no table.
template <bool FILL, bool AGG>
__global__ void __launch_bounds__(AGG ? kBinThreadsAgg : kBinThreadsPlain, AGG ? 2 : 4)
bin_faces_kernel(Scene s, int sets, int warp_agg) {
  constexpr int kBinThreads = AGG ? kBinThreadsAgg : kBinThreadsPlain;
  __shared__ typename std::conditional<AGG, BinSmem, int>::type sm;
  const int tid = threadIdx.x;
  if constexpr (AGG) {
    for (int t = tid; t < kBinHT; t += kBinThreads) { sm.keys[t] = kBinEmpty; sm.vals[t] = 0; }
    __syncthreads();
  }
  int64_t i = (int64_t)blockIdx.x * kBinThreads + tid;
  const bool live = i < s.NF;
  if (!live) i = s.NF - 1;
  int b; int64_t fbase;
  face_view(s, i, b, fbase);
  const int f = (int)(i - fbase);
  float v[6];
  load_xy(s, i, v);
  bool valid = live;
  if (s.fnz) valid = valid && __ldg(s.fnz + i) >= 0.f;
  if (s.valid) valid = valid && (__ldg(s.valid + i) != 0);
  PixRect r[2];
  BinSpan sp[2];
  int where[2][4];
#pragma unroll
  for (int set = 0; set < 2; ++set) {
    sp[set].has = false;
    if (!((sets >> set) & 1)) continue;
    float xmin, ymin, xmax, ymax;
    const float* given = set ? s.bbox_large : s.bbox_tight;
    if (given) {
      const float4 bb = __ldg(reinterpret_cast<const float4*>(given) + i);
      xmin = bb.x; ymin = bb.y; xmax = bb.z; ymax = bb.w;
    } else {
      // tight: torch.min / torch.max over the 3 vertices (rasterization.py:325-327);
      // large: [min - boxlen*m, max + boxlen*m] in fp32 (dibr.py:33-39)
      xmin = fminf(fminf(v[0], v[2]), v[4]); ymin = fminf(fminf(v[1], v[3]), v[5]);
      xmax = fmaxf(fmaxf(v[0], v[2]), v[4]); ymax = fmaxf(fmaxf(v[1], v[3]), v[5]);
      if (set) { xmin = fsub(xmin, s.margin); ymin = fsub(ymin, s.margin); xmax = fadd(xmax, s.margin); ymax = fadd(ymax, s.margin); }
    }
    r[set] = bbox_to_rect(s.grid, xmin, ymin, xmax, ymax);
    sp[set] = bin_span(s, r[set], set ? live : valid);
    const bool small = sp[set].bx1 - sp[set].bx0 <= 1 && sp[set].by1 - sp[set].by0 <= 1;
    bool aggregated = false;
    if constexpr (AGG) {
      aggregated = __all_sync(kFull, small);
      if (aggregated) bin_insert(s, sm, set, b, sp[set], where[set]);
    }
    if (!aggregated && !AGG && warp_agg && __all_sync(kFull, small)) {
      // sparse meshes: neighbours in the index buffer are neighbours on screen, so the lanes of a
      // warp hit a handful of distinct counters; lanes that share one are found with match.any
      // and their leader issues ONE global atomic for all of them
      aggregated = true;
      const int lane = tid & 31;
      const int4 e = make_int4(f, r[set].x_lo | (r[set].x_hi << 16), r[set].y_lo | (r[set].y_hi << 16), 0);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        where[set][k] = -1;
        const int bx = sp[set].bx0 + (k & 1), by = sp[set].by0 + (k >> 1);
        const bool on = sp[set].has && bx <= sp[set].bx1 && by <= sp[set].by1;
        const unsigned act = __ballot_sync(kFull, on);
        if (!on) continue;
        const size_t ci = ((size_t)set * s.B + b) * s.NB + s.bin_base[sp[set].l] + by * s.ntx[sp[set].l] + bx;
        const unsigned peers = __match_any_sync(act, (unsigned long long)ci);
        const int leader = __ffs(peers) - 1;
        int base = 0;
        if (lane == leader) base = atomicAdd(s.cnt + ci, __popc(peers));
        base = __shfl_sync(peers, base, leader);
        if (FILL) s.entries[(size_t)set * 4 * s.NF + 4 * fbase + s.off[ci] + base + __popc(peers & ((1u << lane) - 1u))] = e;
      }
    }
    if (!aggregated) {
      // (also: a warp with a face of the coarsest level spanning more than 2x2 bins)
#pragma unroll
      for (int k = 0; k < 4; ++k) where[set][k] = -1;
      if (sp[set].has) {
        const int4 e = make_int4(f, r[set].x_lo | (r[set].x_hi << 16), r[set].y_lo | (r[set].y_hi << 16), 0);
        for (int by = sp[set].by0; by <= sp[set].by1; ++by)
          for (int bx = sp[set].bx0; bx <= sp[set].bx1; ++bx) {
            const size_t ci = ((size_t)set * s.B + b) * s.NB + s.bin_base[sp[set].l] + by * s.ntx[sp[set].l] + bx;
            const int pos = atomicAdd(s.cnt + ci, 1);
            if (FILL) s.entries[(size_t)set * 4 * s.NF + 4 * fbase + s.off[ci] + pos] = e;
          }
      }
    }
  }
  if (!FILL && (sets & 2) && live && r[1].x_hi > r[1].x_lo && r[1].y_hi > r[1].y_lo) {
    // which 16x16 tiles can see this face in the soft mask (filters the soft-mask work
    // list): one bit per tile, a row of tiles per 32-bit word, so a face ORs one word per
    // tile row
    const int tx0 = r[1].x_lo >> 4, tx1 = (r[1].x_hi - 1) >> 4, ty0 = r[1].y_lo >> 4, ty1 = (r[1].y_hi - 1) >> 4;
    const int w0 = tx0 >> 5, w1 = tx1 >> 5, nw = (s.ntx[0] + 31) >> 5;
    if ((ty1 - ty0 + 1) * (w1 - w0 + 1) <= 64) {
      for (int w = w0; w <= w1; ++w) {
        const int lo = max(tx0 - (w << 5), 0), hi = min(tx1 - (w << 5), 31);
        const uint32_t m = (0xffffffffu >> (31 - hi)) & (0xffffffffu << lo);
        // a (possibly stale) L1 copy that already shows the bits saves the reduction: the
        // faces of a patch all set the same words, and same-address reductions serialise
        for (int t0 = ty0; t0 <= ty1; t0 += 4) {
          int* p = s.tile_cnt + ((size_t)b * s.nty[0] + t0) * nw + w;
          uint32_t have[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) have[j] = t0 + j <= ty1 ? (uint32_t)__ldca(p + (size_t)j * nw) : m;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if ((have[j] & m) != m) atomicOr(p + (size_t)j * nw, (int)m);
        }
      }
    } else {
      atomicOr(s.view_flag + b, 1);
    }
  }
  if constexpr (AGG) {
    __syncthreads();
    // one global atomic per distinct bin of this CTA, each from its own thread
    for (int t = tid; t < kBinHT; t += kBinThreads) {
      const uint32_t ci = sm.keys[t];
      if (ci != kBinEmpty) {
        const int pos = atomicAdd(s.cnt + ci, sm.vals[t]);
        if (FILL) sm.vals[t] = pos + s.off[ci];
      }
    }
    if (!FILL) return;
    __syncthreads();
#pragma unroll
    for (int set = 0; set < 2; ++set) {
      const int4 e = make_int4(f, r[set].x_lo | (r[set].x_hi << 16), r[set].y_lo | (r[set].y_hi << 16), 0);
      int4* dst = s.entries + (size_t)set * 4 * s.NF + 4 * fbase;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int w = where[set][k];
        if (sp[set].has && w >= 0) dst[sm.vals[w >> 16] + (w & 0xffff)] = e;
      }
    }
  }
}

// Exclusive scan of the NB bin counters of one (set, view); resets the counters
// so that the fill pass can reuse them as cursors.
__global__ void __launch_bounds__(1024) scan_bins_kernel(Scene s) {
  __shared__ int warp_sums[32];
  __shared__ int carry;
  int* cnt = s.cnt + (size_t)blockIdx.x * s.NB;
  int* off = s.off + (size_t)blockIdx.x * s.NB;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < s.NB; base += 1024) {
    const int i = base + tid;
    const int v = i < s.NB ? cnt[i] : 0;
    int x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(kFull, x, d);
      if (lane >= d) x += y;
    }
    if (lane == 31) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int w = warp_sums[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(kFull, w, d);
        if (lane >= d) w += y;
      }
      warp_sums[lane] = w;
    }
    __syncthreads();
    const int excl = carry + (warp ? warp_sums[warp - 1] : 0) + x - v;
    if (i < s.NB) { off[i] = excl; cnt[i] = 0; }
    __syncthreads();
    if (tid == 1023) carry = excl + v;
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------
// Tile helpers.
__device__ __forceinline__ uint32_t tile_mask(const int4& e, int tile_x0, int tile_y0) {
  const int x_lo = e.y & 0xffff, x_hi = (int)((unsigned)e.y >> 16);
  const int y_lo = e.z & 0xffff, y_hi = (int)((unsigned)e.z >> 16);
  const int cx0 = max(x_lo - tile_x0, 0), cx1 = min(x_hi - tile_x0, kTile);
  const int cy0 = max(y_lo - tile_y0, 0), cy1 = min(y_hi - tile_y0, kTile);
  if (cx1 <= cx0 || cy1 <= cy0) return 0u;
  const uint32_t cm = ((1u << cx1) - 1u) & ~((1u << cx0) - 1u);
  const uint32_t rm = ((1u << cy1) - 1u) & ~((1u << cy0) - 1u);
  return cm | (rm << 16);
}

struct TileCtx {
  int b, tx, ty, tile_x0, tile_y0;
  int lx, ly, px, py;
  bool in_img;
  float x0, y0;
  uint32_t sel;
  int64_t fbase, pix;
};

__device__ __forceinline__ TileCtx make_tile_ctx(const Scene& s) {
  TileCtx c;
  c.tx = blockIdx.x; c.ty = blockIdx.y; c.b = blockIdx.z;   // grid = (tiles_x, tiles_y, views)
  c.tile_x0 = c.tx * kTile;
  c.tile_y0 = c.ty * kTile;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  c.lx = ((warp & 1) << 3) | (lane & 7);      // each warp owns an 8x4 pixel block
  c.ly = ((warp >> 1) << 2) | (lane >> 3);
  c.px = c.tile_x0 + c.lx;
  c.py = c.tile_y0 + c.ly;
  c.in_img = c.px < s.W && c.py < s.H;
  c.x0 = pix_x(s.grid, c.px);
  c.y0 = pix_y(s.grid, c.py);
  c.sel = (1u << c.lx) | (1u << (16 + c.ly));
  c.fbase = view_fbase(s, c.b);
  c.pix = ((int64_t)c.b * s.H + c.py) * s.W + c.px;
  return c;
}

// bins above tile (tx,ty) in bin set `set`
struct BinRef { const int4* ptr; int n; };
__device__ __forceinline__ BinRef tile_bin(const Scene& s, int b, int tx, int ty, int64_t fbase,
                                           int set, int l) {
  const int sh = 2 * l;
  const int bin = s.bin_base[l] + (ty >> sh) * s.ntx[l] + (tx >> sh);
  const size_t ci = ((size_t)set * s.B + b) * s.NB + bin;
  BinRef r;
  r.n = s.cnt[ci];
  r.ptr = s.entries + (size_t)set * 4 * s.NF + 4 * fbase + s.off[ci];
  return r;
}

// Shared memory of the tile kernels.
struct TileSmem {
  int4 stage[2][kChunk];                 // TMA landing buffers (bin entries)
  float4 cxy0[kChunk];                   // ax ay bx by
  float4 cz[kChunk];                     // az bz cz (pad)
  float2 cxy1[kChunk];                   // cx cy
  uint32_t cmask[kChunk];                // col mask | row mask << 16 (tile local)
  int cface[kChunk];
  unsigned long long list[kSoftCap];     // (face << 32) | mask, unsorted
  unsigned long long sorted[kSoftCap];
  float acc[kChunk][6];                  // soft-mask backward per-candidate sums
  unsigned long long bar[2];
  BinRef bin[2][kMaxLevels];             // the tile's bins (set, level): filled once by warp 0
  uint8_t apix[kThreads];                // compacted uncovered pixels of the tile: lx | ly << 4
  int wcount[kThreads / 32];
  int ncand;
  int nsoft;
  int nent;                              // hits appended to the cache block
  int pool_slot;                         // cache block of this tile (-1: none)
  int npairs;                            // (pixel, face) pairs of the current round
};

// Shared memory of the rasterizing tile kernel (a subset: 4-5 CTAs more per SM).
struct RasterSmem {
  int4 stage[2][kChunk];
  float4 cxy0[kChunk];
  float4 cz[kChunk];
  float2 cxy1[kChunk];
  int cface[kChunk];
  uint32_t colbits[kChunk / 32][16];     // [group of 32 candidates][tile column] -> candidate bits
  uint32_t rowbits[kChunk / 32][16];     // [group][tile row]
  unsigned long long bar[2];
  BinRef bin[2][kMaxLevels];
  int any_uncovered, warps_done;
  unsigned uncmask[kThreads / 32];
};

// Transposes the tile-local rectangle masks of the 32 candidates held by a warp
// (one per lane) into per-column / per-row candidate bit words: a pixel (lx, ly)
// is inside candidate j's rectangle  <=>  bit j of colbits[g][lx] & rowbits[g][ly].
// Every pixel then walks exactly its own rectangle hits (ffs), lane-privately.
__device__ __forceinline__ void store_bit_matrix(uint32_t m, uint32_t (*colbits)[16], uint32_t (*rowbits)[16],
                                                 int g) {
  const int lane = threadIdx.x & 31;
  uint32_t mine = 0;
  if (__any_sync(kFull, m != 0)) {
#pragma unroll
    for (int b = 0; b < 32; ++b) {
      const uint32_t r = __ballot_sync(kFull, (m >> b) & 1u);
      if (lane == b) mine = r;
    }
  }
  if (lane < 16) colbits[g][lane] = mine; else rowbits[g][lane - 16] = mine;
}

// Lanes 0..L-1 / 8..8+L-1 of warp 0 look up the tight / large bins of the tile.
template <typename SM>
__device__ __forceinline__ void load_bin_table(const Scene& s, const TileCtx& c, SM& sm) {
  const int tid = threadIdx.x;
  if (tid < 16) {
    const int set = tid >> 3, l = tid & 7;
    if (l < kMaxLevels) {
      BinRef r; r.ptr = nullptr; r.n = 0;
      if (l < s.L) r = tile_bin(s, c.b, c.tx, c.ty, c.fbase, set, l);
      sm.bin[set][l] = r;
    }
  }
}

// ---------------------------------------------------------------------------
// Rasterization of one tile: walks the "tight" bins of every level.
struct RasterOut { float z, w0, w1, w2; int f; };

template <typename SM>
__device__ __forceinline__ void raster_tile(const Scene& s, const TileCtx& c, const RasterConst& rc,
                                            SM& sm, RasterOut& o) {
  const int tid = threadIdx.x;
  o.z = -INFINITY; o.f = -1; o.w0 = o.w1 = o.w2 = 0.f;

  // The (<= 6) tight bins above the tile form one virtual list, streamed in
  // rounds of kChunk entries: one mbarrier per round, one bulk copy per level piece.
  int nl[kMaxLevels];
  int total = 0;
#pragma unroll
  for (int l = 0; l < kMaxLevels; ++l) { nl[l] = sm.bin[0][l].n; total += nl[l]; }
  if (total == 0) return;  // uniform for the CTA
  const int nrounds = (total + kChunk - 1) / kChunk;

  auto issue = [&](int k) {  // thread 0 only
    const int lo = k * kChunk, hi = min(total, lo + kChunk);
    unsigned long long* bar = &sm.bar[k & 1];
    mbar_expect_tx(bar, (uint32_t)(hi - lo) * 16u);
    int start = 0;
#pragma unroll
    for (int l = 0; l < kMaxLevels; ++l) {
      const int a = max(lo, start), b = min(hi, start + nl[l]);
      if (b > a) tma_load_1d(&sm.stage[k & 1][a - lo], sm.bin[0][l].ptr + (a - start), (uint32_t)(b - a) * 16u, bar);
      start += nl[l];
    }
  };

  if (tid == 0) issue(0);
  for (int k = 0; k < nrounds; ++k) {
    if (tid == 0 && k + 1 < nrounds) issue(k + 1);  // buffer (k+1)&1 was released by the sync ending round k-1
    const int cnt = min(kChunk, total - k * kChunk);
    if ((tid & ~31) < cnt) mbar_wait(&sm.bar[k & 1], (uint32_t)((k >> 1) & 1));   // only the warps that read the buffer poll

    // cull against the tile, gather the face record (candidate id = position in the round)
    uint32_t m = 0;
    if (tid < cnt) {
      const int4 e = sm.stage[k & 1][tid];
      m = tile_mask(e, c.tile_x0, c.tile_y0);
      if (m) {
        const int64_t g = c.fbase + e.x;
        float v[6];
        load_xy(s, g, v);
        const float* zp = s.z + g * 3;
        sm.cxy0[tid] = make_float4(v[0], v[1], v[2], v[3]);
        sm.cxy1[tid] = make_float2(v[4], v[5]);
        sm.cz[tid] = make_float4(__ldg(zp), __ldg(zp + 1), __ldg(zp + 2), 0.f);
        sm.cface[tid] = e.x;
      }
    }
    if ((tid & ~31) < cnt) store_bit_matrix(m, sm.colbits, sm.rowbits, tid >> 5);
    __syncthreads();
    const int ngroups = (cnt + 31) >> 5;
    for (int g = 0; g < ngroups; ++g) {
      uint32_t bits = sm.colbits[g][c.lx] & sm.rowbits[g][c.ly];
      while (bits) {  // lane-private walk over this pixel's rectangle hits
        const int j = (g << 5) + __ffs(bits) - 1;
        bits &= bits - 1;
        const float4 q0 = sm.cxy0[j];
        const float2 q1 = sm.cxy1[j];
        float w0, w1, w2;
        if (!raster_weights(rc, c.x0, c.y0, q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, w0, w1, w2)) continue;
        const float4 zz = sm.cz[j];
        const float zv = raster_depth(zz.x, zz.y, zz.z, w0, w1, w2);
        const int f = sm.cface[j];
        // reference: strict '>' in ascending face order == (z, lowest index) maximum
        if (!(zv <= o.z) || (zv == o.z && f < o.f)) { o.z = zv; o.f = f; o.w0 = w0; o.w1 = w1; o.w2 = w2; }
      }
    }
    if (k + 1 < nrounds) __syncthreads();
  }
}

// ---------------------------------------------------------------------------
// Soft mask of one tile (forward) / its gradient (backward).  Candidates are the
// faces of the "large" bins whose enlarged rectangle meets the tile, visited in
// ascending face index; a pixel stops after knum hits.
template <bool FILTER_ONLY_COUNT, typename SM>
__device__ __forceinline__ int soft_collect(const Scene& s, const TileCtx& c, SM& sm, int lo, int hi) {
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid == 0) sm.nsoft = 0;
  __syncthreads();
  for (int l = 0; l < s.L; ++l) {
    const BinRef bin = sm.bin[1][l];
    for (int base = 0; base < bin.n; base += kThreads) {
      const int i = base + tid;
      uint32_t m = 0; int f = 0;
      if (i < bin.n) {
        const int4 e = __ldg(bin.ptr + i);
        f = e.x;
        if (f > lo && f <= hi) m = tile_mask(e, c.tile_x0, c.tile_y0);
      }
      const unsigned vote = __ballot_sync(kFull, m != 0);
      if (vote) {
        int wbase = 0;
        if (lane == 0) wbase = atomicAdd(&sm.nsoft, __popc(vote));
        wbase = __shfl_sync(kFull, wbase, 0);
        if (!FILTER_ONLY_COUNT && m) {
          const int slot = wbase + __popc(vote & ((1u << lane) - 1u));
          if (slot < kSoftCap) sm.list[slot] = ((unsigned long long)(uint32_t)f << 32) | m;
        }
      }
    }
  }
  __syncthreads();
  const int n = sm.nsoft;
  __syncthreads();  // everyone has read the count before a following call resets it
  return n;
}

// Collects the tile's soft-mask candidates with face index in (lo, hi] into sm.list.
// Normally hi = INT_MAX takes everything; when more than kSoftCap faces remain
// (sub-pixel triangles) a prefix window in index order is taken instead: its upper end
// is guessed from the average index density and halved until it fits (1-3 counting
// passes), the caller continues with lo = hi until every pixel has its knum faces.
template <typename SM>
__device__ __forceinline__ int soft_window(const Scene& s, const TileCtx& c, SM& sm, int lo, int maxf, int& hi) {
  hi = 0x7fffffff;
  int n = soft_collect<false>(s, c, sm, lo, hi);
  if (n > kSoftCap) {
    const int span = maxf - 1 - lo;  // indices lo+1 .. maxf-1
    int width = (int)(((long long)span * kSoftCap * 3) / ((long long)n * 4));
    if (width < 1) width = 1;
    while (true) {
      hi = lo + width;
      if (soft_collect<true>(s, c, sm, lo, hi) <= kSoftCap || width == 1) break;
      width = width > 1 ? width / 2 : 1;
    }
    n = soft_collect<false>(s, c, sm, lo, hi);
  }
  return n;
}

// Sorts sm.list[0..n) by face index into sm.sorted (keys are unique: a face lives in one
// level and a tile reads one bin per level).  Small lists (the usual case) use a rank
// sort, n^2/256 compares per thread and one barrier; big lists (sub-pixel triangles,
// up to kSoftCap) a shared-memory bitonic network, log^2(n) barriers.  Ends with a barrier.
template <typename SM>
__device__ __forceinline__ void soft_sort(SM& sm, int n) {
  const int tid = threadIdx.x;
  if (n <= 320) {
    for (int j = tid; j < n; j += kThreads) {
      const unsigned long long key = sm.list[j];
      int rank = 0;
      for (int i = 0; i < n; ++i) rank += (sm.list[i] < key) ? 1 : 0;
      sm.sorted[rank] = key;
    }
    __syncthreads();
    return;
  }
  int np = 512;
  while (np < n) np <<= 1;
  for (int j = tid; j < np; j += kThreads) sm.sorted[j] = j < n ? sm.list[j] : ~0ull;
  __syncthreads();
  for (int k = 2; k <= np; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = tid; t < (np >> 1); t += kThreads) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));  // lower element of the pair
        const int l = i | j;
        const unsigned long long a = sm.sorted[i], b = sm.sorted[l];
        const bool up = (i & k) == 0;
        if ((a > b) == up) { sm.sorted[i] = b; sm.sorted[l] = a; }
      }
      __syncthreads();
    }
  }
}

struct SoftFwdOut {
  float* prob; int64_t* idx; uint8_t* type;  // K-lists (nullable)
};

__device__ __forceinline__ int tile_linear(const Scene& s, const TileCtx& c) {
  return (c.b * s.nty[0] + c.ty) * s.ntx[0] + c.tx;
}

struct SoftIO {
  float* out_soft;                                   // forward
  SoftFwdOut kl;                                     // forward, operator contract (nullable)
  const float* grad_soft; const float* soft;         // backward
  float* grad_xy;                                    // backward
};

// Soft mask of one tile.  `uncovered` is the calling thread's own pixel; the
// uncovered pixels of the tile are first compacted so that the expensive
// per-(pixel, face) distance work runs on densely packed warps (thread t owns the
// t-th uncovered pixel).  Covered pixels (soft = 1) are written by their own thread.
// CACHE (forward only): every hit (pixel, face, prob, dist_type) is appended to the
// tile's block of the hit cache so that the backward pass is a dense stream over
// hits instead of a second walk (the reference stores 13*knum bytes per pixel).
template <bool BWD, bool KLISTS>
__device__ __forceinline__ void soft_tile(const Scene& s, const TileCtx& c, TileSmem& sm, bool uncovered,
                                          float sigmainv, int K, bool cache, const SoftIO& io) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (!BWD && c.in_img && !uncovered) {
    io.out_soft[c.pix] = 1.0f;
    if (KLISTS) {  // padding the reference gets from at::zeros / at::full(-1)
      for (int k = 0; k < K; ++k) {
        const int64_t o = c.pix * K + k;
        io.kl.prob[o] = 0.f; io.kl.idx[o] = -1; io.kl.type[o] = 0;
      }
    }
  }
  const unsigned av = __ballot_sync(kFull, uncovered);
  if (lane == 0) sm.wcount[warp] = __popc(av);
  __syncthreads();
  int before = 0, na = 0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) {
    const int cw = sm.wcount[w];
    if (w < warp) before += cw;
    na += cw;
  }
  if (na == 0) return;  // uniform
  if (uncovered) sm.apix[before + __popc(av & ((1u << lane) - 1u))] = (uint8_t)(c.lx | (c.ly << 4));
  if (BWD) {
    for (int i = tid; i < kChunk * 6; i += kThreads) (&sm.acc[0][0])[i] = 0.f;
  }
  __syncthreads();
  // thread t now owns the t-th uncovered pixel
  const bool active = tid < na;
  int lx = 0, ly = 0;
  if (active) { const int p = sm.apix[tid]; lx = p & 15; ly = p >> 4; }
  const int px = c.tile_x0 + lx, py = c.tile_y0 + ly;
  const float x0 = pix_x(s.grid, px), y0 = pix_y(s.grid, py);
  const uint32_t sel = (1u << lx) | (1u << (16 + ly));
  const int64_t pix = ((int64_t)c.b * s.H + py) * s.W + px;
  float dLdp = 0.f, soft_saved = 0.f;
  if (BWD && active) { dLdp = io.grad_soft[pix]; soft_saved = io.soft[pix]; }

  float allprob = 1.0f;
  int kid = 0;
  const int maxf = s.first ? (int)(__ldg(s.first + c.b + 1) - c.fbase) : s.F;
  const size_t E = (size_t)256 * s.pool_K;
  uint32_t* blk = nullptr;
  bool first_window = true;
  int lo = -1;
  while (true) {
    int hi;
    int n = soft_window(s, c, sm, lo, maxf, hi);
    if (!BWD && cache && first_window) {
      first_window = false;
      if (tid == 0) {
        int slot = -1;
        if (n > 0) {
          slot = atomicAdd(s.pool_ctr, 1);
          if (slot >= s.pool_tiles) {   // cache full: this tile is recomputed in backward
            slot = -1;
            s.fb_list[atomicAdd(s.fb_ctr, 1)] = tile_linear(s, c);
          }
        }
        sm.pool_slot = slot;
        sm.nent = 0;
      }
      __syncthreads();
      if (sm.pool_slot >= 0) blk = s.pool_data + (size_t)sm.pool_slot * 3 * E;
    }
    soft_sort(sm, n);  // by face index
    bool all_done = false;
    for (int c0 = 0; c0 < n && !all_done; c0 += kChunk) {
      const int cn = min(kChunk, n - c0);
      if (tid < cn) {
        const unsigned long long key = sm.sorted[c0 + tid];
        const int f = (int)(key >> 32);
        float v[6];
        load_xy(s, c.fbase + f, v);
        sm.cxy0[tid] = make_float4(v[0], v[1], v[2], v[3]);
        sm.cxy1[tid] = make_float2(v[4], v[5]);
        sm.cmask[tid] = (uint32_t)key;
        sm.cface[tid] = f;
      }
      __syncthreads();
      if (warp * 32 < na) {  // warps that own no uncovered pixel have nothing to do
        for (int j = 0; j < cn; ++j) {
          const bool hit = active && kid < K && ((sm.cmask[j] & sel) == sel);
          float g[6];
          float prob = 0.f;
          int edgeid = 0;
          if (hit) {
            const float4 q0 = sm.cxy0[j];
            const float2 q1 = sm.cxy1[j];
            const float v[6] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y};
            const float d2 = soft_min_dist(x0, y0, v, s.multiplier, edgeid);
            prob = soft_prob(d2, sigmainv, s.multiplier);
            if (!BWD) {
              allprob = soft_accumulate(allprob, prob);
              if (KLISTS) {
                const int64_t o = pix * K + kid;
                io.kl.prob[o] = prob; io.kl.idx[o] = sm.cface[j]; io.kl.type[o] = (uint8_t)(edgeid + 1);
              }
            } else {
              soft_backward_terms(x0, y0, v, edgeid, prob, soft_saved, dLdp, sigmainv, s.multiplier, g);
            }
            ++kid;
          }
          if (!BWD && blk != nullptr) {
            const unsigned vote = __ballot_sync(kFull, hit);
            if (vote) {
              int wb = 0;
              if (lane == 0) wb = atomicAdd(&sm.nent, __popc(vote));
              wb = __shfl_sync(kFull, wb, 0);
              if (hit) {
                const size_t e = (size_t)wb + __popc(vote & ((1u << lane) - 1u));
                blk[e] = (uint32_t)sm.cface[j];
                blk[E + e] = __float_as_uint(prob);
                blk[2 * E + e] = (uint32_t)lx | ((uint32_t)ly << 4) | ((uint32_t)(edgeid + 1) << 8);
              }
            }
          }
          if (BWD) {
            if (__any_sync(kFull, hit)) {
#pragma unroll
              for (int q = 0; q < 6; ++q) {
                float x = hit ? g[q] : 0.f;
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(kFull, x, d);
                if (lane == 0 && x != 0.f) atomicAdd(&sm.acc[j][q], x);
              }
            }
          }
        }
      }
      all_done = __syncthreads_and(!active || kid >= K);
      if (BWD) {
        if (tid < cn) {
          float* gp = io.grad_xy + (c.fbase + sm.cface[tid]) * 6;
#pragma unroll
          for (int q = 0; q < 6; ++q) {
            const float x = sm.acc[tid][q];
            if (x != 0.f) { atomicAdd(gp + q, x); sm.acc[tid][q] = 0.f; }
          }
        }
        __syncthreads();
      }
    }
    if (hi == 0x7fffffff || all_done) break;
    lo = hi;
  }
  if (!BWD) {
    if (active) {
      io.out_soft[pix] = soft_finish(allprob);
      if (KLISTS) {
        for (int k = kid; k < K; ++k) {
          const int64_t o = pix * K + k;
          io.kl.prob[o] = 0.f; io.kl.idx[o] = -1; io.kl.type[o] = 0;
        }
      }
    }
    if (blk != nullptr && tid == 0) s.pool_hdr[sm.pool_slot] = make_int4(c.b, c.tx, c.ty, sm.nent);
  }
}

// ---------------------------------------------------------------------------
// Soft mask forward of one tile, pair-parallel.  The uncovered pixels are
// compacted; in rounds, every pixel claims its next (<= kRound) faces in ascending
// index (respecting knum) straight from its hit bit words, the claimed (pixel, face)
// pairs are laid out face-major in shared memory, ALL 256 threads evaluate the
// expensive distance/probability of one pair each, and finally every pixel folds
// its own results in order — the same sequence of fp32/fp64 operations per pixel as
// the reference's sequential loop, with the work spread over every lane.
struct SoftSmem {
  unsigned long long list[kSoftCap];     // (face << 32) | mask, unsorted
  unsigned long long sorted[kSoftCap];
  float4 cxy0[kChunk];
  float2 cxy1[kChunk];
  int cface[kChunk];
  uint32_t colbits[kChunk / 32][16];
  uint32_t rowbits[kChunk / 32][16];
  int cnt_c[kChunk];                     // claims per face in this round
  int off_c[kChunk];                     // face-major pair offsets
  float res_prob[kPairCap];
  uint16_t claim[kThreads][kRound];      // per pixel: (face | pos << 8), then the pair slot
  uint8_t pair_cand[kPairCap];
  uint8_t pair_pix[kPairCap];
  uint8_t res_type[kPairCap];
  uint8_t apix[kThreads];
  BinRef bin[2][kMaxLevels];
  int wcount[kThreads / 32];
  int nsoft, nent, pool_slot, npairs;
};

template <bool KLISTS>
__device__ __forceinline__ void soft_tile_fwd(const Scene& s, const TileCtx& c, SoftSmem& sm, bool uncovered,
                                              float sigmainv, int K, bool cache, const SoftIO& io) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned av = __ballot_sync(kFull, uncovered);
  if (lane == 0) sm.wcount[warp] = __popc(av);
  __syncthreads();
  int before = 0, na = 0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) {
    const int cw = sm.wcount[w];
    if (w < warp) before += cw;
    na += cw;
  }
  if (na == 0) return;  // uniform
  if (uncovered) sm.apix[before + __popc(av & ((1u << lane) - 1u))] = (uint8_t)(c.lx | (c.ly << 4));
  __syncthreads();
  const bool active = tid < na;  // thread t owns the t-th uncovered pixel
  int lx = 0, ly = 0;
  if (active) { const int p = sm.apix[tid]; lx = p & 15; ly = p >> 4; }
  const int64_t pix = ((int64_t)c.b * s.H + (c.tile_y0 + ly)) * s.W + (c.tile_x0 + lx);

  float allprob = 1.0f;
  int kid = 0;
  const int maxf = s.first ? (int)(__ldg(s.first + c.b + 1) - c.fbase) : s.F;
  const size_t E = (size_t)256 * s.pool_K;
  uint32_t* blk = nullptr;
  bool first_window = true;
  int lo = -1;
  while (true) {
    int hi;
    int n = soft_window(s, c, sm, lo, maxf, hi);
    if (first_window) {
      first_window = false;
      if (tid == 0) {
        int slot = -1;
        if (cache && n > 0) {
          slot = atomicAdd(s.pool_ctr, 1);
          if (slot >= s.pool_tiles) {   // cache full: this tile is recomputed in backward
            slot = -1;
            s.fb_list[atomicAdd(s.fb_ctr, 1)] = tile_linear(s, c);
          }
        }
        sm.pool_slot = slot;
        sm.nent = 0;
      }
      __syncthreads();
      if (sm.pool_slot >= 0) blk = s.pool_data + (size_t)sm.pool_slot * 3 * E;
    }
    soft_sort(sm, n);  // by face index
    bool all_done = false;
    for (int c0 = 0; c0 < n && !all_done; c0 += kChunk) {
      const int cn = min(kChunk, n - c0);
      const int ngroups = (cn + 31) >> 5;
      uint32_t m = 0;
      if (tid < cn) {
        const unsigned long long key = sm.sorted[c0 + tid];
        const int f = (int)(key >> 32);
        m = (uint32_t)key;
        float v[6];
        load_xy(s, c.fbase + f, v);
        sm.cxy0[tid] = make_float4(v[0], v[1], v[2], v[3]);
        sm.cxy1[tid] = make_float2(v[4], v[5]);
        sm.cface[tid] = f;
      }
      if (warp < ngroups) store_bit_matrix(m, sm.colbits, sm.rowbits, warp);
      sm.cnt_c[tid] = 0;
      __syncthreads();
      int g = 0;              // hit word being consumed by this pixel
      uint32_t bits = active ? (sm.colbits[0][lx] & sm.rowbits[0][ly]) : 0u;
      while (true) {
        // claim the next <= kRound faces of this pixel, in index order
        int took = 0;
        if (active) {
          while (took < kRound && kid + took < K) {
            while (bits == 0 && g + 1 < ngroups) { ++g; bits = sm.colbits[g][lx] & sm.rowbits[g][ly]; }
            if (bits == 0) break;
            const int j = (g << 5) + __ffs(bits) - 1;
            bits &= bits - 1;
            const int pos = atomicAdd(&sm.cnt_c[j], 1);
            sm.claim[tid][took] = (uint16_t)(j | (pos << 8));
            ++took;
          }
        }
        if (!__syncthreads_or(took > 0)) break;
        // face-major offsets
        if (warp == 0) {
          int v[8], sum = 0;
#pragma unroll
          for (int i = 0; i < 8; ++i) { const int j = lane * 8 + i; v[i] = j < cn ? sm.cnt_c[j] : 0; sum += v[i]; }
          int x = sum;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(kFull, x, d); if (lane >= d) x += y; }
          int run = x - sum;
#pragma unroll
          for (int i = 0; i < 8; ++i) { const int j = lane * 8 + i; if (j < cn) sm.off_c[j] = run; run += v[i]; }
          if (lane == 31) sm.npairs = x;
        }
        __syncthreads();
        const int T = sm.npairs;
        const int ebase = sm.nent;
        for (int i = 0; i < took; ++i) {
          const int cl = sm.claim[tid][i];
          const int j = cl & 0xff;
          const int slot = sm.off_c[j] + (cl >> 8);
          sm.pair_cand[slot] = (uint8_t)j;
          sm.pair_pix[slot] = (uint8_t)tid;
          sm.claim[tid][i] = (uint16_t)slot;
        }
        __syncthreads();
        sm.cnt_c[tid] = 0;  // for the next round (ordered by the barrier below)
        // dense evaluation: one (pixel, face) pair per thread
        for (int u = tid; u < T; u += kThreads) {
          const int j = sm.pair_cand[u];
          const int p = sm.apix[sm.pair_pix[u]];
          const int plx = p & 15, ply = p >> 4;
          const float4 q0 = sm.cxy0[j];
          const float2 q1 = sm.cxy1[j];
          const float v[6] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y};
          int edgeid;
          const float d2 = soft_min_dist(pix_x(s.grid, c.tile_x0 + plx), pix_y(s.grid, c.tile_y0 + ply), v,
                                         s.multiplier, edgeid);
          const float prob = soft_prob(d2, sigmainv, s.multiplier);
          sm.res_prob[u] = prob;
          sm.res_type[u] = (uint8_t)(edgeid + 1);
          if (blk != nullptr) {
            const size_t e = (size_t)ebase + u;
            blk[e] = (uint32_t)sm.cface[j];
            blk[E + e] = __float_as_uint(prob);
            blk[2 * E + e] = (uint32_t)plx | ((uint32_t)ply << 4) | ((uint32_t)(edgeid + 1) << 8);
          }
        }
        __syncthreads();
        if (tid == 0) sm.nent = ebase + T;
        // every pixel folds its own results in face order
        for (int i = 0; i < took; ++i) {
          const int slot = sm.claim[tid][i];
          const float prob = sm.res_prob[slot];
          allprob = soft_accumulate(allprob, prob);
          if (KLISTS) {
            const int64_t o = pix * K + kid;
            io.kl.prob[o] = prob; io.kl.idx[o] = sm.cface[sm.pair_cand[slot]]; io.kl.type[o] = sm.res_type[slot];
          }
          ++kid;
        }
      }
      all_done = __syncthreads_and(!active || kid >= K);
    }
    if (hi == 0x7fffffff || all_done) break;
    lo = hi;
  }
  if (active) io.out_soft[pix] = soft_finish(allprob);
  if (blk != nullptr && tid == 0) s.pool_hdr[sm.pool_slot] = make_int4(c.b, c.tx, c.ty, sm.nent);
}

// Large-set bin table of a tile from its work-list record (threads 0..5 write it).
template <typename SM>
__device__ __forceinline__ void bins_from_record(const Scene& s, const int* rec, int64_t fbase, SM& sm) {
  const int tid = threadIdx.x;
  if (tid < kMaxLevels) {
    BinRef r;
    r.n = __ldg(rec + 10 + 2 * tid);
    r.ptr = s.entries + (size_t)4 * s.NF + 4 * fbase + __ldg(rec + 9 + 2 * tid);
    sm.bin[1][tid] = r;
  }
}

__device__ __forceinline__ TileCtx tile_ctx_from_linear(const Scene& s, int t) {
  TileCtx c;
  const int tiles_xy = s.ntx[0] * s.nty[0];
  c.b = t / tiles_xy;
  const int r = t - c.b * tiles_xy;
  c.ty = r / s.ntx[0];
  c.tx = r - c.ty * s.ntx[0];
  c.tile_x0 = c.tx * kTile; c.tile_y0 = c.ty * kTile;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  c.lx = ((warp & 1) << 3) | (lane & 7);
  c.ly = ((warp >> 1) << 2) | (lane >> 3);
  c.px = c.tile_x0 + c.lx; c.py = c.tile_y0 + c.ly;
  c.in_img = c.px < s.W && c.py < s.H;
  c.x0 = 0.f; c.y0 = 0.f; c.sel = 0;
  c.fbase = view_fbase(s, c.b);
  c.pix = ((int64_t)c.b * s.H + c.py) * s.W + c.px;
  return c;
}

// ---------------------------------------------------------------------------
// Feature storage type FT: float, or __nv_bfloat16 (BASELINE configs[3] "bf16 features":
// face_features, interpolated_features and their upstream gradient are bf16 in HBM; all
// arithmetic stays fp32 on the upcast values, the result is rounded once on store, and
// grad_face_features is accumulated in fp32).  Geometry is always fp32.
template <typename FT> struct Feat;
template <> struct Feat<float> {
  static __device__ __forceinline__ float ld(const float* p) { return __ldg(p); }
  static __device__ __forceinline__ float ld_stream(const float* p) { return __ldcs(p); }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
};
template <> struct Feat<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
  static __device__ __forceinline__ float ld_stream(const __nv_bfloat16* p) { return __bfloat162float(__ldcs(p)); }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

// ---------------------------------------------------------------------------
// Forward tile kernel.
struct FwdArgs {
  Scene s;
  RasterConst rc;
  int D;
  const void* feat;         // (NF,3,D) FT
  float sigmainv; int K;
  int cache;                // fill the soft-mask hit cache
  int from_fb;              // soft_tiles_fwd_kernel: walk fb_list instead of band_list
  void* out_feat;           // (B,H,W,D) FT
  int64_t* idx; float* out_w; float* out_soft;  // idx: output if RASTER else input
  SoftFwdOut kl;
};

template <bool RASTER, bool SOFT, bool KLISTS, typename FT>
__global__ void __launch_bounds__(kThreads, 6) dibr_tile_fwd_kernel(const __grid_constant__ FwdArgs a) {
  __shared__ __align__(128) RasterSmem sm;
  const Scene& s = a.s;
  const int tid = threadIdx.x;
  const TileCtx c = make_tile_ctx(s);
  if (RASTER && tid == 32) { mbar_init(&sm.bar[0], 1); mbar_init(&sm.bar[1], 1); mbar_fence_init(); }
  if (tid == 64) { sm.any_uncovered = 0; sm.warps_done = 0; }
  load_bin_table(s, c, sm);
  __syncthreads();
  int best_f;
  if (RASTER) {
    RasterOut o;
    raster_tile(s, c, a.rc, sm, o);
    best_f = o.f;
    if (c.in_img) {
      a.idx[c.pix] = (int64_t)o.f;
      float* wp = a.out_w + c.pix * 3;
      wp[0] = o.w0; wp[1] = o.w1; wp[2] = o.w2;
      FT* fp = static_cast<FT*>(a.out_feat) + c.pix * a.D;
      const FT* feat = static_cast<const FT*>(a.feat);
      if (a.D == 3) {  // the DIB-R tutorial shape (uv + mask), fully unrolled
        float r[3] = {0.f, 0.f, 0.f};
        if (o.f >= 0) {
          const FT* ff = feat + (c.fbase + o.f) * 9;
#pragma unroll
          for (int d = 0; d < 3; ++d)
            r[d] = raster_interp(Feat<FT>::ld(ff + d), Feat<FT>::ld(ff + 3 + d), Feat<FT>::ld(ff + 6 + d),
                                 o.w0, o.w1, o.w2);
        }
        Feat<FT>::st(fp, r[0]); Feat<FT>::st(fp + 1, r[1]); Feat<FT>::st(fp + 2, r[2]);
      } else if (o.f >= 0) {
        const FT* ff = feat + (c.fbase + o.f) * 3 * a.D;
        for (int d = 0; d < a.D; ++d)
          Feat<FT>::st(fp + d, raster_interp(Feat<FT>::ld(ff + d), Feat<FT>::ld(ff + a.D + d),
                                             Feat<FT>::ld(ff + 2 * a.D + d), o.w0, o.w1, o.w2));
      } else {
        for (int d = 0; d < a.D; ++d) Feat<FT>::st(fp + d, 0.f);
      }
    }
  } else {
    best_f = c.in_img ? (int)a.idx[c.pix] : 0;
  }
  if (SOFT) {
    // defaults (covered: 1; uncovered with no neighbour: 1 - 1 = 0) and K-list padding; tiles
    // where an uncovered pixel may lie under an enlarged face go to the soft-mask work list
    const bool uncovered = c.in_img && best_f < 0;
    if (c.in_img) {
      a.out_soft[c.pix] = uncovered ? 0.0f : 1.0f;
      if (KLISTS) {  // padding the reference gets from at::zeros / at::full(-1)
        for (int k = 0; k < a.K; ++k) {
          const int64_t o = c.pix * a.K + k;
          a.kl.prob[o] = 0.f; a.kl.idx[o] = -1; a.kl.type[o] = 0;
        }
      }
    }
    // no CTA barrier: warps retire independently; the last one to finish files the tile
    const unsigned wv = __ballot_sync(kFull, uncovered);
    if ((tid & 31) == 0) {
      sm.uncmask[tid >> 5] = wv;
      if (wv) atomicOr(&sm.any_uncovered, 1);
      __threadfence_block();
      if (atomicAdd(&sm.warps_done, 1) == kThreads / 32 - 1 && atomicOr(&sm.any_uncovered, 0)) {
        const int nlarge = ((__ldg(s.tile_cnt + ((size_t)c.b * s.nty[0] + c.ty) * ((s.ntx[0] + 31) >> 5) + (c.tx >> 5)) >> (c.tx & 31)) & 1) +
                           __ldg(s.view_flag + c.b);
        if (nlarge > 0) {
          // work-list record: everything the soft-mask kernels need to start without
          // re-reading face_idx or the bin tables
          int* rec = s.band_list + (size_t)atomicAdd(s.band_ctr, 1) * kBandRec;
          const int4* ebase = s.entries + (size_t)4 * s.NF + 4 * c.fbase;
          rec[0] = tile_linear(s, c);
          for (int q = 0; q < kThreads / 32; ++q) rec[1 + q] = (int)atomicOr(&sm.uncmask[q], 0u);
          for (int l = 0; l < kMaxLevels; ++l) {
            rec[9 + 2 * l] = sm.bin[1][l].n > 0 ? (int)(sm.bin[1][l].ptr - ebase) : 0;
            rec[10 + 2 * l] = sm.bin[1][l].n;
          }
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------
// Forward tile kernel, second generation.  Same results as dibr_tile_fwd_kernel; what changed
// is where the instructions go (ncu, round 1: 750 warp instructions per 8x4 pixel block, of
// which ~300 were per-tile fixed work shared by only 8 warps, and 6.9 hit-walk iterations for
// the slowest lane of a block):
//   * a CTA owns S x S screen tiles (S = 2: 32x32 px) and stages their candidates ONCE
//     (bin table, TMA rounds, tile cull, face gather, bit matrices); the S*S sub-tiles are
//     then rasterized one after the other with the round-1 thread -> pixel mapping, so the
//     soft-mask work list, the hit cache and every consumer keep their 16x16 tiles;
//   * a face is inserted in up to 2x2 level-0 bins; with several of them under one CTA it is
//     taken from the first of its bins inside the CTA only (integer test on its rectangle);
//   * conservative triangle-vs-block culling: while staging, each candidate gets its three
//     edge functions as AFFINE functions of the CTA-local pixel index (computed in double,
//     oriented so that inside is >= 0), with a margin that dominates the fp32 rounding of the
//     reference's own evaluation.  A warp (8x4 block) lets lane j test candidate j at the
//     block's extreme corners; candidates that are provably outside one edge at every pixel
//     of the block are dropped (8.5 -> 4.9 candidates per block on the benchmark mesh);
//   * the surviving candidates are visited in a WARP-UNIFORM loop (broadcast shared-memory
//     reads, no per-lane bit walk); the per-pixel decision is still the exact reference
//     arithmetic of raster_weights, so face_idx stays bit-exact.
template <int S>
struct FwdSmem {
  static constexpr int kSide = kTile * S;
  static constexpr int kSubs = S * S;
  int4 stage[2][kChunk];
  float4 cxy0[kChunk];
  float4 cz[kChunk];
  float2 cxy1[kChunk];
  int cface[kChunk];
  float4 cedge[kChunk][3];                 // per edge: {A + margin, B, C, -}: s*u_i ~ A + B*lx + C*ly
  uint32_t colbits[kChunk / 32][kSide];
  uint32_t rowbits[kChunk / 32][kSide];
  unsigned long long bar[2];
  BinRef bin0[2][kSubs];                   // level-0 bins of the sub-tiles (set, sub)
  BinRef bin[2][kMaxLevels];               // levels >= 1 (entry 0 unused)
  int any_uncovered[kSubs], warps_done[kSubs];
  unsigned uncmask[kSubs][kThreads / 32];
};

// Affine, sign-normalised edge functions of one face over a CTA tile whose pixel (0,0) has the
// centre (X0, Y0) and whose pixel pitch is (dx, -dy).  See the kernel comment for the contract:
// s*u_i(pixel) computed by the reference in fp32 is < 0 wherever A' + B*lx + C*ly < 0.
__device__ __noinline__ void make_edge_tests(const float v[6], double X0, double Y0, double dx, double dy,
                                                int side, float4 out[3]) {
  const double ax = v[0], ay = v[1], bx = v[2], by = v[3], cx = v[4], cy = v[5];
  const double n = (bx - ax) * (cy - ay) - (by - ay) * (cx - ax);   // u0 + u1 + u2, exact up to 2^-53
  const double sgn = n < 0.0 ? -1.0 : 1.0;
  const double ext_x = side * dx, ext_y = side * dy;
  const double Rx = fmax(fmax(fabs(ax - X0), fabs(bx - X0)), fabs(cx - X0)) + ext_x;
  const double Ry = fmax(fmax(fabs(ay - Y0), fabs(by - Y0)), fabs(cy - Y0)) + ext_y;
  const double coord = fabs(X0) + fabs(Y0) + ext_x + ext_y;
  const double px[3] = {bx, cx, ax}, py[3] = {by, cy, ay};          // u0: P=b,Q=c  u1: P=c,Q=a  u2: P=a,Q=b
  const double qx[3] = {cx, ax, bx}, qy[3] = {cy, ay, by};
  double A[3], B[3], C[3], marg = 0.0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double ux = py[i] - qy[i], uy = qx[i] - px[i];            // du/dx, du/dy
    A[i] = sgn * ((px[i] - X0) * (qy[i] - Y0) - (py[i] - Y0) * (qx[i] - X0));
    B[i] = sgn * ux * dx;
    C[i] = -sgn * uy * dy;
    const double m = 1.9073486328125e-06 * Rx * Ry                                  // 2^-19: fp32 products / fma
                     + 4.76837158203125e-07 * coord * (fabs(ux) + fabs(uy))          // 2^-21: pixel-centre rounding
                     + 9.5367431640625e-07 * (fabs(A[i]) + side * (fabs(B[i]) + fabs(C[i])));  // 2^-20: the block test itself
    marg = fmax(marg, m);
  }
  marg = 4.0 * marg + 1e-6;
  // the orientation must be certain and every quantity in range for the sign argument
  const bool ok = fabs(n) > 16.0 * marg && Rx < 268435456.0 && Ry < 268435456.0 && coord < 268435456.0;
#pragma unroll
  for (int i = 0; i < 3; ++i)
    out[i] = ok ? make_float4((float)(A[i] + marg), (float)B[i], (float)C[i], 0.f)
                : make_float4(INFINITY, 0.f, 0.f, 0.f);           // never culled (also NaN / Inf input)
}

#ifndef DIBR_FWD2_MINB
#define DIBR_FWD2_MINB 6
#endif
template <bool RASTER, bool SOFT, bool KLISTS, typename FT, int S>
__global__ void __launch_bounds__(kThreads, DIBR_FWD2_MINB) dibr_fwd2_kernel(const __grid_constant__ FwdArgs a) {
  using SM = FwdSmem<S>;
  constexpr int kSubs = S * S;
  constexpr int kSide = kTile * S;
  constexpr int kPieces = kSubs + kMaxLevels - 1;
  __shared__ __align__(128) SM sm;
  const Scene& s = a.s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.z;
  const int ctx0 = blockIdx.x * S, cty0 = blockIdx.y * S;   // first 16x16 tile of the CTA
  const int cta_x0 = ctx0 * kTile, cta_y0 = cty0 * kTile;
  const int64_t fbase = view_fbase(s, b);

  if (RASTER && tid == 32) { mbar_init(&sm.bar[0], 1); mbar_init(&sm.bar[1], 1); mbar_fence_init(); }
  if (tid >= 64 && tid < 64 + kSubs) { sm.any_uncovered[tid - 64] = 0; sm.warps_done[tid - 64] = 0; }
  if (tid < 2 * kSubs) {
    const int set = tid / kSubs, sub = tid % kSubs;
    const int tx = ctx0 + sub % S, ty = cty0 + sub / S;
    BinRef r; r.ptr = nullptr; r.n = 0;
    if (tx < s.ntx[0] && ty < s.nty[0]) r = tile_bin(s, b, tx, ty, fbase, set, 0);
    sm.bin0[set][sub] = r;
  } else if (tid >= 96 && tid < 96 + 16) {
    const int set = (tid - 96) >> 3, l = (tid - 96) & 7;
    if (l < kMaxLevels) {
      BinRef r; r.ptr = nullptr; r.n = 0;
      if (l >= 1 && l < s.L) r = tile_bin(s, b, ctx0, cty0, fbase, set, l);
      sm.bin[set][l] = r;
    }
  }
  __syncthreads();

  // the tight bins above the CTA tile as one virtual list: S*S level-0 pieces, then levels 1..
  auto pn = [&](int p) { return p < kSubs ? sm.bin0[0][p].n : sm.bin[0][p - kSubs + 1].n; };
  int total = 0;
  if (RASTER) {
#pragma unroll
    for (int p = 0; p < kPieces; ++p) total += pn(p);
  }
  const int nrounds = (total + kChunk - 1) / kChunk;
  int issued = 0, waited = 0;       // staging iterations (thread 0 / everyone): buffer = n & 1, parity = (n >> 1) & 1
  auto issue = [&](int k) {          // thread 0 only
    const int lo = k * kChunk, hi = min(total, lo + kChunk);
    unsigned long long* bar = &sm.bar[issued & 1];
    mbar_expect_tx(bar, (uint32_t)(hi - lo) * 16u);
    int start = 0;
#pragma unroll
    for (int p = 0; p < kPieces; ++p) {
      const int4* ptr = p < kSubs ? sm.bin0[0][p].ptr : sm.bin[0][p - kSubs + 1].ptr;
      const int np = pn(p);
      const int x = max(lo, start), y = min(hi, start + np);
      if (y > x) tma_load_1d(&sm.stage[issued & 1][x - lo], ptr + (x - start), (uint32_t)(y - x) * 16u, bar);
      start += np;
    }
    ++issued;
  };

  bool staged = false;

  // ---- CTA tiles that no valid face touches (40 % of them on the benchmark scene): the outputs are
  // constants, written as full 16-byte vectors row by row (9 stores per thread instead of 32)
  if (RASTER && !KLISTS && total == 0 && cta_x0 + kSide <= s.W && cta_y0 + kSide <= s.H && (s.W & 3) == 0 &&
      std::is_same<FT, float>::value && a.D == 3) {
    const int64_t pix_row0 = ((int64_t)b * s.H + cta_y0) * s.W + cta_x0;
    const int4 neg = make_int4(-1, -1, -1, -1);
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    constexpr int kIdxC = kSide * 8 / 16, kWC = kSide * 12 / 16, kSC = kSide * 4 / 16;   // 16-byte chunks per row
    for (int c = tid; c < kSide * kIdxC; c += kThreads) {
      const int r = c / kIdxC, ch = c - r * kIdxC;
      reinterpret_cast<int4*>(a.idx + pix_row0 + (int64_t)r * s.W)[ch] = neg;
    }
    for (int c = tid; c < kSide * kWC; c += kThreads) {
      const int r = c / kWC, ch = c - r * kWC;
      reinterpret_cast<float4*>(a.out_w + (pix_row0 + (int64_t)r * s.W) * 3)[ch] = zero;
      reinterpret_cast<float4*>(static_cast<float*>(a.out_feat) + (pix_row0 + (int64_t)r * s.W) * 3)[ch] = zero;
    }
    if (SOFT) {
      for (int c = tid; c < kSide * kSC; c += kThreads) {
        const int r = c / kSC, ch = c - r * kSC;
        reinterpret_cast<float4*>(a.out_soft + pix_row0 + (int64_t)r * s.W)[ch] = zero;   // uncovered, no neighbour yet
      }
      if (tid < kSubs) {   // every pixel is uncovered: file the sub-tiles an enlarged face can reach
        const int tx = ctx0 + tid % S, ty = cty0 + tid / S;
        const int nlarge = ((__ldg(s.tile_cnt + ((size_t)b * s.nty[0] + ty) * ((s.ntx[0] + 31) >> 5) + (tx >> 5)) >> (tx & 31)) & 1) +
                           __ldg(s.view_flag + b);
        if (nlarge > 0) {
          int* rec = s.band_list + (size_t)atomicAdd(s.band_ctr, 1) * kBandRec;
          const int4* ebase = s.entries + (size_t)4 * s.NF + 4 * fbase;
          rec[0] = (b * s.nty[0] + ty) * s.ntx[0] + tx;
          for (int q = 0; q < kThreads / 32; ++q) rec[1 + q] = -1;
          for (int l = 0; l < kMaxLevels; ++l) {
            const BinRef br = l == 0 ? sm.bin0[1][tid] : sm.bin[1][l];
            rec[9 + 2 * l] = br.n > 0 ? (int)(br.ptr - ebase) : 0;
            rec[10 + 2 * l] = br.n;
          }
        }
      }
    }
    return;
  }

  for (int sub = 0; sub < kSubs; ++sub) {
    const int sx = sub % S, sy = sub / S;
    const int tx = ctx0 + sx, ty = cty0 + sy;
    if (tx >= s.ntx[0] || ty >= s.nty[0]) continue;   // uniform: sub-tile outside the image
    const int lx = ((warp & 1) << 3) | (lane & 7);     // each warp owns an 8x4 pixel block
    const int ly = ((warp >> 1) << 2) | (lane >> 3);
    const int px = tx * kTile + lx, py = ty * kTile + ly;
    const bool in_img = px < s.W && py < s.H;
    const int64_t pix = ((int64_t)b * s.H + py) * s.W + px;
    int best_f;
    if (RASTER) {
      RasterOut o;
      o.z = -INFINITY; o.f = -1; o.w0 = o.w1 = o.w2 = 0.f;
      if (total > 0) {
        const float x0 = pix_x(s.grid, px), y0 = pix_y(s.grid, py);
        const int clx = sx * kTile + lx, cly = sy * kTile + ly;
        const float fbx0 = (float)(sx * kTile + ((warp & 1) << 3)), fbx1 = fbx0 + 7.f;
        const float fby0 = (float)(sy * kTile + ((warp >> 1) << 2)), fby1 = fby0 + 3.f;
        for (int k = 0; k < nrounds; ++k) {
          const int cnt = min(kChunk, total - k * kChunk);
          if (!(staged && nrounds == 1)) {
            // ---- stage round k: TMA -> cull against the CTA tile -> face records, edge tests, bit matrices
            if (tid == 0) {
              if (k == 0) issue(0);
              if (k + 1 < nrounds) issue(k + 1);   // its buffer was released by the barrier ending round k-1
            }
            const int buf = waited & 1;
            // only the warps that read the landing buffer poll the mbarrier; the others go
            // straight to the CTA barrier below and sleep there (256 polling threads cost 5 % of
            // the kernel's instructions in the first version)
            if ((tid & ~31) < cnt) mbar_wait(&sm.bar[buf], (uint32_t)((waited >> 1) & 1));
            ++waited;
            uint32_t cm = 0, rm = 0;
            if (tid < cnt) {
              const int4 e = sm.stage[buf][tid];
              const int x_lo = e.y & 0xffff, x_hi = (int)((unsigned)e.y >> 16);
              const int y_lo = e.z & 0xffff, y_hi = (int)((unsigned)e.z >> 16);
              bool take = true;
              if (S > 1) {
                // level-0 pieces: the face is also in the neighbouring bins it spans; take it from
                // the first of its bins inside this CTA only
                const int vi = k * kChunk + tid;
                int start = 0;
#pragma unroll
                for (int p = 0; p < kSubs; ++p) {
                  const int np = pn(p);
                  if (vi >= start && vi < start + np)
                    take = (ctx0 + p % S) == max(x_lo >> 4, ctx0) && (cty0 + p / S) == max(y_lo >> 4, cty0);
                  start += np;
                }
              }
              if (take) {
                const int cx0 = max(x_lo - cta_x0, 0), cx1 = min(x_hi - cta_x0, kSide);
                const int cy0 = max(y_lo - cta_y0, 0), cy1 = min(y_hi - cta_y0, kSide);
                if (cx1 > cx0 && cy1 > cy0) {
                  cm = (uint32_t)(((1ull << cx1) - 1ull) & ~((1ull << cx0) - 1ull));
                  rm = (uint32_t)(((1ull << cy1) - 1ull) & ~((1ull << cy0) - 1ull));
                }
              }
              if (cm) {
                const int64_t g = fbase + e.x;
                float v[6];
                load_xy(s, g, v);
                const float* zp = s.z + g * 3;
                sm.cxy0[tid] = make_float4(v[0], v[1], v[2], v[3]);
                sm.cxy1[tid] = make_float2(v[4], v[5]);
                sm.cz[tid] = make_float4(__ldg(zp), __ldg(zp + 1), __ldg(zp + 2), 0.f);
                sm.cface[tid] = e.x;
                float4 et[3];
                make_edge_tests(v, (double)pix_x(s.grid, cta_x0), (double)pix_y(s.grid, cta_y0),
                                2.0 * (double)s.grid.inv_w, 2.0 * (double)s.grid.inv_h, kSide, et);
                sm.cedge[tid][0] = et[0]; sm.cedge[tid][1] = et[1]; sm.cedge[tid][2] = et[2];
              }
            }
            if ((tid & ~31) < cnt) {
              // transpose the rectangle masks of this warp's 32 candidates into per-column / per-row words
              const int g = tid >> 5;
              if (__any_sync(kFull, cm != 0)) {
                uint32_t mine_c = 0, mine_r = 0;
#pragma unroll
                for (int q = 0; q < kSide; ++q) {
                  const uint32_t c = __ballot_sync(kFull, (cm >> q) & 1u);
                  const uint32_t r = __ballot_sync(kFull, (rm >> q) & 1u);
                  if (lane == (q & 31)) { mine_c = c; mine_r = r; }
                }
                if (lane < kSide) { sm.colbits[g][lane] = mine_c; sm.rowbits[g][lane] = mine_r; }
              } else if (lane < kSide) {
                sm.colbits[g][lane] = 0; sm.rowbits[g][lane] = 0;
              }
            }
            __syncthreads();
          }
          // ---- rasterize this sub-tile against the staged round
          const int ngroups = (cnt + 31) >> 5;
          for (int g = 0; g < ngroups; ++g) {
            const uint32_t mybits = sm.colbits[g][clx] & sm.rowbits[g][cly];
            const uint32_t uni = __reduce_or_sync(kFull, mybits);   // candidates whose rectangle meets the block
            if (!uni) continue;
            bool keep = false;
            if ((uni >> lane) & 1u) {                                 // lane j: candidate j against the block's corners
              const float4 e0 = sm.cedge[(g << 5) + lane][0], e1 = sm.cedge[(g << 5) + lane][1],
                           e2 = sm.cedge[(g << 5) + lane][2];
              const float h0 = e0.x + fmaxf(e0.y * fbx0, e0.y * fbx1) + fmaxf(e0.z * fby0, e0.z * fby1);
              const float h1 = e1.x + fmaxf(e1.y * fbx0, e1.y * fbx1) + fmaxf(e1.z * fby0, e1.z * fby1);
              const float h2 = e2.x + fmaxf(e2.y * fbx0, e2.y * fbx1) + fmaxf(e2.z * fby0, e2.z * fby1);
              keep = !(h0 < 0.f || h1 < 0.f || h2 < 0.f);
            }
            uint32_t surv = __ballot_sync(kFull, keep);
            while (surv) {                                            // warp-uniform loop
              const int jj = __ffs(surv) - 1;
              surv &= surv - 1;
              if (!((mybits >> jj) & 1u)) continue;
              const int j = (g << 5) + jj;
              const float4 q0 = sm.cxy0[j];
              const float2 q1 = sm.cxy1[j];
              float w0, w1, w2;
              if (!raster_weights(a.rc, x0, y0, q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, w0, w1, w2)) continue;
              const float4 zz = sm.cz[j];
              const float zv = raster_depth(zz.x, zz.y, zz.z, w0, w1, w2);
              const int f = sm.cface[j];
              // reference: strict '>' in ascending face order == (z, lowest index) maximum
              if (!(zv <= o.z) || (zv == o.z && f < o.f)) { o.z = zv; o.f = f; o.w0 = w0; o.w1 = w1; o.w2 = w2; }
            }
          }
          if (nrounds > 1) __syncthreads();   // the next round overwrites the staged arrays
        }
        staged = true;
      }
      best_f = o.f;
      if (in_img) {
        a.idx[pix] = (int64_t)o.f;
        float* wp = a.out_w + pix * 3;
        wp[0] = o.w0; wp[1] = o.w1; wp[2] = o.w2;
        FT* fp = static_cast<FT*>(a.out_feat) + pix * a.D;
        const FT* feat = static_cast<const FT*>(a.feat);
        if (a.D == 3) {  // the DIB-R tutorial shape (uv + mask), fully unrolled
          float r[3] = {0.f, 0.f, 0.f};
          if (o.f >= 0) {
            const FT* ff = feat + (fbase + o.f) * 9;
#pragma unroll
            for (int d = 0; d < 3; ++d)
              r[d] = raster_interp(Feat<FT>::ld(ff + d), Feat<FT>::ld(ff + 3 + d), Feat<FT>::ld(ff + 6 + d),
                                   o.w0, o.w1, o.w2);
          }
          Feat<FT>::st(fp, r[0]); Feat<FT>::st(fp + 1, r[1]); Feat<FT>::st(fp + 2, r[2]);
        } else if (o.f >= 0) {
          const FT* ff = feat + (fbase + o.f) * 3 * a.D;
          for (int d = 0; d < a.D; ++d)
            Feat<FT>::st(fp + d, raster_interp(Feat<FT>::ld(ff + d), Feat<FT>::ld(ff + a.D + d),
                                               Feat<FT>::ld(ff + 2 * a.D + d), o.w0, o.w1, o.w2));
        } else {
          for (int d = 0; d < a.D; ++d) Feat<FT>::st(fp + d, 0.f);
        }
      }
    } else {
      best_f = in_img ? (int)a.idx[pix] : 0;
    }
    if (SOFT) {
      // defaults (covered: 1; uncovered with no neighbour: 1 - 1 = 0) and K-list padding; tiles
      // where an uncovered pixel may lie under an enlarged face go to the soft-mask work list
      const bool uncovered = in_img && best_f < 0;
      if (in_img) {
        a.out_soft[pix] = uncovered ? 0.0f : 1.0f;
        if (KLISTS) {  // padding the reference gets from at::zeros / at::full(-1)
          for (int k = 0; k < a.K; ++k) {
            const int64_t o = pix * a.K + k;
            a.kl.prob[o] = 0.f; a.kl.idx[o] = -1; a.kl.type[o] = 0;
          }
        }
      }
      // no CTA barrier: warps retire independently; the last one to finish files the tile
      const unsigned wv = __ballot_sync(kFull, uncovered);
      if (lane == 0) {
        sm.uncmask[sub][warp] = wv;
        if (wv) atomicOr(&sm.any_uncovered[sub], 1);
        __threadfence_block();
        if (atomicAdd(&sm.warps_done[sub], 1) == kThreads / 32 - 1 && atomicOr(&sm.any_uncovered[sub], 0)) {
          const int nlarge = ((__ldg(s.tile_cnt + ((size_t)b * s.nty[0] + ty) * ((s.ntx[0] + 31) >> 5) + (tx >> 5)) >> (tx & 31)) & 1) +
                             __ldg(s.view_flag + b);
          if (nlarge > 0) {
            // work-list record: everything the soft-mask kernels need to start without
            // re-reading face_idx or the bin tables
            int* rec = s.band_list + (size_t)atomicAdd(s.band_ctr, 1) * kBandRec;
            const int4* ebase = s.entries + (size_t)4 * s.NF + 4 * fbase;
            rec[0] = (b * s.nty[0] + ty) * s.ntx[0] + tx;
            for (int q = 0; q < kThreads / 32; ++q) rec[1 + q] = (int)atomicOr(&sm.uncmask[sub][q], 0u);
            for (int l = 0; l < kMaxLevels; ++l) {
              const BinRef br = l == 0 ? sm.bin0[1][sub] : sm.bin[1][l];
              rec[9 + 2 * l] = br.n > 0 ? (int)(br.ptr - ebase) : 0;
              rec[10 + 2 * l] = br.n;
            }
          }
        }
      }
    }
  }
}

// Soft-mask forward over the work list (persistent CTAs).
template <bool KLISTS>
__global__ void __launch_bounds__(kThreads, 4) soft_tiles_fwd_kernel(const __grid_constant__ FwdArgs a) {
  extern __shared__ __align__(128) unsigned char soft_smem_raw[];
  SoftSmem& sm = *reinterpret_cast<SoftSmem*>(soft_smem_raw);
  const Scene& s = a.s;
  const int total = min(a.from_fb ? *s.fb_ctr : *s.band_ctr, s.ntx[0] * s.nty[0] * s.B);
  SoftIO io;
  io.out_soft = a.out_soft; io.kl = a.kl; io.grad_soft = nullptr; io.soft = nullptr; io.grad_xy = nullptr;
  for (int w = blockIdx.x; w < total; w += gridDim.x) {
    const TileCtx c = tile_ctx_from_linear(s, a.from_fb ? s.fb_list[w] : s.band_list[(size_t)w * kBandRec]);
    __syncthreads();  // previous tile's shared state fully consumed
    load_bin_table(s, c, sm);
    __syncthreads();
    soft_tile_fwd<KLISTS>(s, c, sm, c.in_img && a.idx[c.pix] < 0, a.sigmainv, a.K, !KLISTS && a.cache != 0, io);
  }
}

// ---------------------------------------------------------------------------
// Two-kernel soft-mask forward (knum <= 32, hit cache available):
//   soft_enum_kernel : per silhouette tile, decides WHICH (pixel, face) pairs exist
//                      (integer work only) and lays them out face-major in the tile's
//                      cache block, with each pixel's slot list in face order;
//   soft_eval_kernel : one thread per pair - the expensive distance / probability,
//                      dense - then each pixel folds its probabilities in face order
//                      (a tile's pairs are all evaluated by the CTA that folds them).
// Tiles that do not fit the cache go to fb_list and take the single-kernel path.
constexpr int kEnumK = 32;
constexpr int kRunHits = 8;   // consecutive cached pairs per thread in the run kernels

struct EnumSmem {
  unsigned long long list[kSoftCap];
  unsigned long long sorted[kSoftCap];
  int cface[kChunk];
  uint32_t colbits[kChunk / 32][16];
  uint32_t rowbits[kChunk / 32][16];
  int cnt_c[kChunk];
  int off_c[kChunk];
  uint16_t claim[kThreads][kEnumK];
  uint8_t apix[kThreads];
  BinRef bin[2][kMaxLevels];
  int wcount[kThreads / 32];
  int nsoft, nent, pool_slot, npairs;
};

#ifndef DIBR_ENUM_MINB
#define DIBR_ENUM_MINB 6   /* measured: 80 registers / 3 CTAs per SM 0.436 ms, 48 / 5: 0.388, 40 / 6: 0.374 */
#endif
__global__ void __launch_bounds__(kThreads, DIBR_ENUM_MINB) soft_enum_kernel(const __grid_constant__ FwdArgs a) {
  __shared__ __align__(128) EnumSmem sm;
  const Scene& s = a.s;
  const int K = a.K;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int total = min(*s.band_ctr, s.ntx[0] * s.nty[0] * s.B);
  const size_t E = (size_t)256 * s.pool_K;
  for (int w = blockIdx.x; w < total; w += gridDim.x) {
    // the work-list record carries the tile id, the uncovered-pixel ballots of the
    // rasterizer's 8 warps and the tile's large-bin table: one load latency, no
    // face_idx re-read, no barrier for the compaction
    const int* rec = s.band_list + (size_t)w * kBandRec;
    const TileCtx c = tile_ctx_from_linear(s, __ldg(rec));
    unsigned mymask = 0;
    int before = 0, na = 0;
#pragma unroll
    for (int q = 0; q < kThreads / 32; ++q) {
      const unsigned mq = (unsigned)__ldg(rec + 1 + q);
      if (q < warp) before += __popc(mq);
      if (q == warp) mymask = mq;
      na += __popc(mq);
    }
    __syncthreads();  // previous tile's shared state fully consumed
    bins_from_record(s, rec, c.fbase, sm);
    if ((mymask >> lane) & 1u) sm.apix[before + __popc(mymask & ((1u << lane) - 1u))] = (uint8_t)(c.lx | (c.ly << 4));
    const bool active = tid < na;
    int lx = 0, ly = 0;
    int kid = 0;
    const int maxf = s.first ? (int)(__ldg(s.first + c.b + 1) - c.fbase) : s.F;
    uint32_t* blk = nullptr;
    uint16_t* myslots = nullptr;
    bool first_window = true, cached = true;
    int lo = -1;
    while (true) {
      int hi;
      int n = soft_window(s, c, sm, lo, maxf, hi);
      if (first_window && active) { const int p = sm.apix[tid]; lx = p & 15; ly = p >> 4; }
      const bool alloc = first_window;
      if (first_window) {
        first_window = false;
        if (n == 0) { cached = false; break; }  // uncovered pixels, but no face near them: soft stays 0
        // cache block: one atomic, its round trip hidden behind the sort below
        if (tid == 0) {
          int slot = atomicAdd(s.pool_ctr, 1);
          if (slot >= s.pool_tiles) {   // cache full: single-kernel path + recompute in backward
            slot = -1;
            s.fb_list[atomicAdd(s.fb_ctr, 1)] = tile_linear(s, c);
          }
          sm.pool_slot = slot;
          sm.nent = 0;
        }
      }
      soft_sort(sm, n);  // by face index
      if (alloc) {
        if (sm.pool_slot < 0) { cached = false; break; }  // uniform: handed over to the single-kernel path
        blk = s.pool_data + (size_t)sm.pool_slot * 3 * E;
        myslots = s.pool_slots + ((size_t)sm.pool_slot * kThreads + tid) * kEnumK;
      }
      bool all_done = false;
      for (int c0 = 0; c0 < n && !all_done; c0 += kChunk) {
        const int cn = min(kChunk, n - c0);
        const int ngroups = (cn + 31) >> 5;
        uint32_t m = 0;
        if (tid < cn) {
          const unsigned long long key = sm.sorted[c0 + tid];
          m = (uint32_t)key;
          sm.cface[tid] = (int)(key >> 32);
        }
        if (warp < ngroups) store_bit_matrix(m, sm.colbits, sm.rowbits, warp);
        sm.cnt_c[tid] = 0;
        __syncthreads();
        // every uncovered pixel claims ALL its remaining faces of this chunk (index order, <= knum)
        // (a warp-uniform candidate loop with one ballot + one atomic per (warp, candidate) was
        // measured slower: 0.47 vs 0.37 ms)
        int took = 0;
        if (active) {
          for (int g = 0; g < ngroups && kid + took < K; ++g) {
            uint32_t bits = sm.colbits[g][lx] & sm.rowbits[g][ly];
            while (bits && kid + took < K) {
              const int j = (g << 5) + __ffs(bits) - 1;
              bits &= bits - 1;
              const int pos = atomicAdd(&sm.cnt_c[j], 1);
              sm.claim[tid][took] = (uint16_t)(j | (pos << 8));
              ++took;
            }
          }
        }
        __syncthreads();
        if (warp == 0) {  // face-major offsets
          int v[8], sum = 0;
#pragma unroll
          for (int i = 0; i < 8; ++i) { const int j = lane * 8 + i; v[i] = j < cn ? sm.cnt_c[j] : 0; sum += v[i]; }
          int x = sum;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(kFull, x, d); if (lane >= d) x += y; }
          int run = x - sum;
#pragma unroll
          for (int i = 0; i < 8; ++i) { const int j = lane * 8 + i; if (j < cn) sm.off_c[j] = run; run += v[i]; }
          if (lane == 31) sm.npairs = x;
        }
        __syncthreads();
        const int ebase = sm.nent;
        for (int i = 0; i < took; ++i) {
          const int cl = sm.claim[tid][i];
          const int j = cl & 0xff;
          const int slot = ebase + sm.off_c[j] + (cl >> 8);
          blk[slot] = (uint32_t)sm.cface[j];
          blk[2 * E + slot] = (uint32_t)lx | ((uint32_t)ly << 4);
          myslots[kid + i] = (uint16_t)slot;
        }
        kid += took;
        all_done = __syncthreads_and(!active || kid >= K);
        if (tid == 0) sm.nent = ebase + sm.npairs;
      }
      if (hi == 0x7fffffff || all_done) break;
      lo = hi;
    }
    if (cached) {
      __syncthreads();
      s.pool_aux[(size_t)sm.pool_slot * kThreads + tid] =
          active ? ((uint32_t)(lx | (ly << 4)) | ((uint32_t)kid << 8)) : 0u;
      if (tid == 0) {
        s.pool_hdr[sm.pool_slot] = make_int4(c.b, c.tx, c.ty, sm.nent);
        s.pool_na[sm.pool_slot] = na;
      }
    }
  }
}

__global__ void __launch_bounds__(kThreads) soft_eval_kernel(const __grid_constant__ FwdArgs a) {
  const Scene& s = a.s;
  const int used = min(*s.pool_ctr, s.pool_tiles);
  if ((int)blockIdx.x >= used) return;
  const int4 h = s.pool_hdr[blockIdx.x];  // b, tx, ty, hits
  const size_t E = (size_t)256 * s.pool_K;
  uint32_t* blk = s.pool_data + (size_t)blockIdx.x * 3 * E;
  const int64_t fbase = view_fbase(s, h.x);
  const int tid = threadIdx.x;
  uint32_t nface = 0, nmeta = 0;
  if (tid < h.w) { nface = blk[tid]; nmeta = blk[2 * E + tid]; }
  for (int t = tid; t < h.w; t += kThreads) {
    const uint32_t face = nface, meta = nmeta;
    if (t + kThreads < h.w) { nface = blk[t + kThreads]; nmeta = blk[2 * E + t + kThreads]; }
    const int px = h.y * kTile + (int)(meta & 15u), py = h.z * kTile + (int)((meta >> 4) & 15u);
    float v[6];
    load_xy(s, fbase + (int)face, v);
    int edgeid;
    const float d2 = soft_min_dist(pix_x(s.grid, px), pix_y(s.grid, py), v, s.multiplier, edgeid);
    const float prob = soft_prob(d2, a.sigmainv, s.multiplier);
    blk[E + t] = __float_as_uint(prob);
    blk[2 * E + t] = meta | ((uint32_t)(edgeid + 1) << 8);
  }
  // fold: each uncovered pixel multiplies its probabilities in face order
  // (dibr_soft_mask_cuda.cu:174-182); the tile's pairs were all evaluated by this CTA
  __syncthreads();
  if (tid >= s.pool_na[blockIdx.x]) return;
  const uint32_t aux = s.pool_aux[(size_t)blockIdx.x * kThreads + tid];
  const uint16_t* myslots = s.pool_slots + ((size_t)blockIdx.x * kThreads + tid) * kEnumK;
  const int cnt = (int)(aux >> 8);
  float allprob = 1.0f;
  for (int i = 0; i < cnt; ++i) allprob = soft_accumulate(allprob, __uint_as_float(blk[E + myslots[i]]));
  const int fx = h.y * kTile + (int)(aux & 15u), fy = h.z * kTile + (int)((aux >> 4) & 15u);
  a.out_soft[((int64_t)h.x * s.H + fy) * s.W + fx] = soft_finish(allprob);
}

// ---------------------------------------------------------------------------
// Soft-mask backward.  (1) dense kernel over the hit cache; (2) the recompute tile
// kernel for the tiles the cache could not hold (fb_list) or, with no forward state,
// for every tile.  Persistent CTAs walk the work list.
struct SoftBwdArgs {
  Scene s;
  float sigmainv; int K;
  int from_list;             // 1: tiles of fb_list only; 0: every tile
  int view_begin, view_end;  // only tiles / cache blocks of these views (dibr_b200_backward_views)
  const float* grad_soft; const float* soft; const int64_t* idx;
  float* grad_xy;
};

__global__ void __launch_bounds__(kThreads) dibr_tile_soft_bwd_kernel(const __grid_constant__ SoftBwdArgs a) {
  __shared__ __align__(128) TileSmem sm;
  const Scene& s = a.s;
  const int ntiles = s.ntx[0] * s.nty[0] * s.B;
  const int total = a.from_list ? min(*s.fb_ctr, ntiles) : ntiles;
  for (int w = blockIdx.x; w < total; w += gridDim.x) {
    const TileCtx c = tile_ctx_from_linear(s, a.from_list ? s.fb_list[w] : w);
    if (c.b < a.view_begin || c.b >= a.view_end) continue;   // uniform for the CTA
    __syncthreads();  // previous tile's shared state fully consumed
    load_bin_table(s, c, sm);
    __syncthreads();
    SoftIO io;
    io.out_soft = nullptr; io.kl = SoftFwdOut{nullptr, nullptr, nullptr};
    io.grad_soft = a.grad_soft; io.soft = a.soft; io.grad_xy = a.grad_xy;
    soft_tile<true, false>(s, c, sm, c.in_img && a.idx[c.pix] < 0, a.sigmainv, a.K, false, io);
  }
}

template <int N>
__device__ __forceinline__ void reduce_peers(unsigned peers, float (&v)[N]);

__global__ void __launch_bounds__(kThreads) soft_bwd_dense_kernel(const __grid_constant__ SoftBwdArgs a) {
  const Scene& s = a.s;
  const int used = min(*s.pool_ctr, s.pool_tiles);
  if ((int)blockIdx.x >= used) return;
  const int4 h = s.pool_hdr[blockIdx.x];  // b, tx, ty, hits
  if (h.x < a.view_begin || h.x >= a.view_end) return;
  const size_t E = (size_t)256 * s.pool_K;
  const uint32_t* blk = s.pool_data + (size_t)blockIdx.x * 3 * E;
  const int64_t fbase = view_fbase(s, h.x);
  const int tid = threadIdx.x, lane = tid & 31;
  uint32_t nface = 0, nprob = 0, nmeta = 0;
  if (tid < h.w) { nface = __ldcs(blk + tid); nprob = __ldcs(blk + E + tid); nmeta = __ldcs(blk + 2 * E + tid); }
  for (int base = 0; base < h.w; base += kThreads) {
    const int t = base + tid;
    const bool valid = t < h.w;
    const uint32_t cface = nface, cprob = nprob, meta = nmeta;
    if (t + kThreads < h.w) {  // next batch of hits: requested before this one is processed
      nface = __ldcs(blk + t + kThreads); nprob = __ldcs(blk + E + t + kThreads);
      nmeta = __ldcs(blk + 2 * E + t + kThreads);
    }
    int face = -1 - lane;
    float g[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) g[q] = 0.f;
    if (valid) {
      face = (int)cface;
      const float prob = __uint_as_float(cprob);
      const int px = h.y * kTile + (int)(meta & 15u), py = h.z * kTile + (int)((meta >> 4) & 15u);
      const int64_t pix = ((int64_t)h.x * s.H + py) * s.W + px;
      float v[6];
      load_xy(s, fbase + face, v);
      soft_backward_terms(pix_x(s.grid, px), pix_y(s.grid, py), v, (int)(meta >> 8) - 1, prob,
                          __ldg(a.soft + pix), __ldg(a.grad_soft + pix), a.sigmainv, s.multiplier, g);
    }
    // hits were appended candidate by candidate: neighbouring lanes mostly share the face
    const unsigned peers = __match_any_sync(kFull, face);
    reduce_peers<6>(peers, g);
    if (valid && (peers & ((1u << lane) - 1u)) == 0) {
      float2* gx = reinterpret_cast<float2*>(a.grad_xy + (fbase + face) * 6);
      if (g[0] != 0.f || g[1] != 0.f) atomicAdd(gx, make_float2(g[0], g[1]));
      if (g[2] != 0.f || g[3] != 0.f) atomicAdd(gx + 1, make_float2(g[2], g[3]));
      if (g[4] != 0.f || g[5] != 0.f) atomicAdd(gx + 2, make_float2(g[4], g[5]));
    }
  }
}

// Dense soft-mask backward, RUN variant: the hits of a tile lie face-major in its cache block, so
// a thread that takes 8 CONSECUTIVE hits (two LDG.128 per array, 32 bytes per lane, 1 KB per warp
// request) sees one or two faces.  It sums the six partials of a face in registers and flushes
// them with three RED.v2 when the face changes - no match/shuffle reduction (30 SHFL per warp at
// 1 SHFL per clock per SM in the kernel above) and one face-vertex load per run instead of per hit.
#ifndef DIBR_SBWD_MINB
#define DIBR_SBWD_MINB 4   /* 64 registers (12 B of spills), 32 warps/SM: 0.290 vs 0.303 ms at 3 */
#endif
__global__ void __launch_bounds__(kThreads, DIBR_SBWD_MINB) soft_bwd_runs_kernel(const __grid_constant__ SoftBwdArgs a) {
  const Scene& s = a.s;
  const int used = min(*s.pool_ctr, s.pool_tiles);
  if ((int)blockIdx.x >= used) return;
  const int4 h = s.pool_hdr[blockIdx.x];  // b, tx, ty, hits
  if (h.x < a.view_begin || h.x >= a.view_end) return;
  const size_t E = (size_t)256 * s.pool_K;
  const uint32_t* blk = s.pool_data + (size_t)blockIdx.x * 3 * E;
  const int64_t fbase = view_fbase(s, h.x);
  const float inv_m = 1.0f / s.multiplier;
  const int64_t pix_tile = ((int64_t)h.x * s.H + (int64_t)h.z * kTile) * s.W + h.y * kTile;
  for (int start = threadIdx.x * kRunHits; start < h.w; start += kThreads * kRunHits) {
    const int n = min(kRunHits, h.w - start);
    uint32_t face[kRunHits], prob[kRunHits], meta[kRunHits];
    {
      const uint4* pf = reinterpret_cast<const uint4*>(blk + start);
      const uint4* pp = reinterpret_cast<const uint4*>(blk + E + start);
      const uint4* pm = reinterpret_cast<const uint4*>(blk + 2 * E + start);
      // the block is sized 256*K entries: reading the (unused) tail of the last group of 8 stays inside it
      const uint4 f0 = __ldcs(pf), f1 = __ldcs(pf + 1), p0 = __ldcs(pp), p1 = __ldcs(pp + 1);
      const uint4 m0 = __ldcs(pm), m1 = __ldcs(pm + 1);
      face[0] = f0.x; face[1] = f0.y; face[2] = f0.z; face[3] = f0.w; face[4] = f1.x; face[5] = f1.y; face[6] = f1.z; face[7] = f1.w;
      prob[0] = p0.x; prob[1] = p0.y; prob[2] = p0.z; prob[3] = p0.w; prob[4] = p1.x; prob[5] = p1.y; prob[6] = p1.z; prob[7] = p1.w;
      meta[0] = m0.x; meta[1] = m0.y; meta[2] = m0.z; meta[3] = m0.w; meta[4] = m1.x; meta[5] = m1.y; meta[6] = m1.z; meta[7] = m1.w;
    }
    int cur = -1;
    float v[6], acc[6];
#pragma unroll
    for (int j = 0; j < kRunHits; ++j) {
      if (j < n) {
        const int f = (int)face[j];
        if (f != cur) {
          if (cur >= 0) {
            float2* gx = reinterpret_cast<float2*>(a.grad_xy + (fbase + cur) * 6);
            if (acc[0] != 0.f || acc[1] != 0.f) atomicAdd(gx, make_float2(acc[0], acc[1]));
            if (acc[2] != 0.f || acc[3] != 0.f) atomicAdd(gx + 1, make_float2(acc[2], acc[3]));
            if (acc[4] != 0.f || acc[5] != 0.f) atomicAdd(gx + 2, make_float2(acc[4], acc[5]));
          }
          cur = f;
          load_xy(s, fbase + f, v);
#pragma unroll
          for (int q = 0; q < 6; ++q) acc[q] = 0.f;
        }
        const int lx = (int)(meta[j] & 15u), ly = (int)((meta[j] >> 4) & 15u);
        const int64_t pix = pix_tile + (int64_t)ly * s.W + lx;
        float g[6];
        soft_backward_terms_fast(pix_x(s.grid, h.y * kTile + lx), pix_y(s.grid, h.z * kTile + ly), v,
                                 (int)(meta[j] >> 8) - 1, __uint_as_float(prob[j]), __ldg(a.soft + pix),
                                 __ldg(a.grad_soft + pix), a.sigmainv, inv_m, g);
#pragma unroll
        for (int q = 0; q < 6; ++q) acc[q] += g[q];
      }
    }
    if (cur >= 0) {
      float2* gx = reinterpret_cast<float2*>(a.grad_xy + (fbase + cur) * 6);
      if (acc[0] != 0.f || acc[1] != 0.f) atomicAdd(gx, make_float2(acc[0], acc[1]));
      if (acc[2] != 0.f || acc[3] != 0.f) atomicAdd(gx + 1, make_float2(acc[2], acc[3]));
      if (acc[4] != 0.f || acc[5] != 0.f) atomicAdd(gx + 2, make_float2(acc[4], acc[5]));
    }
  }
}

// ---------------------------------------------------------------------------
// Rasterize backward: pixel-parallel; lanes of a warp (an 8x4 pixel block) that
// hit the same face are summed with a segmented shuffle reduction, so a face
// costs one group of atomics per warp instead of 9*D per pixel
// (rasterization_cuda.cu:272-285,376-399).
template <int N>
__device__ __forceinline__ void reduce_peers(unsigned peers, float (&v)[N]) {
  const int lane = threadIdx.x & 31;
  int rel = __popc(peers & ((1u << lane) - 1u));
  peers &= (0xfffffffeu << lane);  // peers above me
  while (__any_sync(kFull, peers)) {
    const int next = __ffs(peers);  // 1-based lane of my next peer, 0 if none
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const float t = __shfl_sync(kFull, v[i], (next - 1) & 31);
      if (next) v[i] += t;
    }
    const unsigned done = __ballot_sync(kFull, rel & 1);
    peers &= ~done;
    rel >>= 1;
  }
}

struct RasterBwdArgs {
  int B, H, W, F, D;
  int ntx, nty;
  const void* grad_feat; const int64_t* idx; const float* w; const float* xy; const void* feat;  // FT
  float eps;
  float* grad_xy; float* grad_feat_out;
};

template <int DT, typename FT>  // DT > 0: feature dim known at compile time; 0: runtime loop
__global__ void __launch_bounds__(kThreads, 6) raster_bwd_kernel(const __grid_constant__ RasterBwdArgs a) {
  const FT* grad_feat = static_cast<const FT*>(a.grad_feat);
  const FT* feat = static_cast<const FT*>(a.feat);
  const int tx = blockIdx.x, ty = blockIdx.y, b = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int px = tx * kTile + (((warp & 1) << 3) | (lane & 7));
  const int py = ty * kTile + (((warp >> 1) << 2) | (lane >> 3));
  const bool in_img = px < a.W && py < a.H;
  const int64_t pix = ((int64_t)b * a.H + py) * a.W + px;
  const int D = DT > 0 ? DT : a.D;
  // all streaming operands of the pixel are requested together (weights and upstream
  // gradient do not depend on face_idx): one exposed HBM latency instead of two
  int f = -1;
  float w0 = 0.f, w1 = 0.f, w2 = 0.f;
  float gpre[DT > 0 ? DT : 1];
#pragma unroll
  for (int d = 0; d < (DT > 0 ? DT : 1); ++d) gpre[d] = 0.f;
  if (in_img) {
    const float* wp = a.w + pix * 3;
    f = (int)__ldcs(a.idx + pix);
    w0 = __ldcs(wp); w1 = __ldcs(wp + 1); w2 = __ldcs(wp + 2);
    if (DT > 0) {
#pragma unroll
      for (int d = 0; d < DT; ++d) gpre[d] = Feat<FT>::ld_stream(grad_feat + pix * DT + d);
    }
  }
  if (!__any_sync(kFull, f >= 0)) return;
  const bool cov = f >= 0;
  const int64_t face = (int64_t)b * a.F + (cov ? f : 0);

  RasterBwdGeom G;
  if (cov) {
    const float2* pp = reinterpret_cast<const float2*>(a.xy + face * 6);
    const float2 pa = __ldg(pp), pb = __ldg(pp + 1), pc = __ldg(pp + 2);
    const float p[6] = {pa.x, pa.y, pb.x, pb.y, pc.x, pc.y};
    raster_backward_geom(p, w0, w1, w2, a.eps, G);
  }
  // lanes without a face get unique negative keys so they never merge
  const unsigned peers = __match_any_sync(kFull, cov ? (int)f : -1 - lane);
  const bool leader = (peers & ((1u << lane) - 1u)) == 0;
  const FT* gp = grad_feat + pix * D;
  const FT* cf = feat + face * 3 * D;

  if (DT > 0) {
    float v[6 + 3 * (DT > 0 ? DT : 1)];
#pragma unroll
    for (int j = 0; j < 6; ++j) v[j] = 0.f;
#pragma unroll
    for (int d = 0; d < DT; ++d) {
      float g = 0.f;
      if (cov) {
        g = gpre[d];
        float t6[6];
        raster_backward_feature(G, g, Feat<FT>::ld(cf + d), Feat<FT>::ld(cf + DT + d), Feat<FT>::ld(cf + 2 * DT + d), t6);
#pragma unroll
        for (int j = 0; j < 6; ++j) v[j] += t6[j];
      }
      v[6 + d] = g * w0; v[6 + DT + d] = g * w1; v[6 + 2 * DT + d] = g * w2;
    }
    reduce_peers<6 + 3 * (DT > 0 ? DT : 1)>(peers, v);
    if (leader && cov) {
      float2* gx = reinterpret_cast<float2*>(a.grad_xy + face * 6);
      atomicAdd(gx, make_float2(v[0], v[1]));
      atomicAdd(gx + 1, make_float2(v[2], v[3]));
      atomicAdd(gx + 2, make_float2(v[4], v[5]));
      float* gf = a.grad_feat_out + face * 3 * DT;
#pragma unroll
      for (int j = 0; j < 3 * DT; ++j) atomicAdd(gf + j, v[6 + j]);
    }
  } else {
    float vx[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) vx[j] = 0.f;
    for (int d = 0; d < D; ++d) {
      float g = 0.f;
      if (cov) {
        g = Feat<FT>::ld_stream(gp + d);
        float t6[6];
        raster_backward_feature(G, g, Feat<FT>::ld(cf + d), Feat<FT>::ld(cf + D + d), Feat<FT>::ld(cf + 2 * D + d), t6);
#pragma unroll
        for (int j = 0; j < 6; ++j) vx[j] += t6[j];
      }
      float v[3] = {g * w0, g * w1, g * w2};
      reduce_peers<3>(peers, v);
      if (leader && cov) {
        float* gf = a.grad_feat_out + face * 3 * D;
        atomicAdd(gf + d, v[0]); atomicAdd(gf + D + d, v[1]); atomicAdd(gf + 2 * D + d, v[2]);
      }
    }
    reduce_peers<6>(peers, vx);
    if (leader && cov) {
      float2* gx = reinterpret_cast<float2*>(a.grad_xy + face * 6);
      atomicAdd(gx, make_float2(vx[0], vx[1]));
      atomicAdd(gx + 1, make_float2(vx[2], vx[3]));
      atomicAdd(gx + 2, make_float2(vx[4], vx[5]));
    }
  }
}

// ---------------------------------------------------------------------------
// Rasterize backward, ROW-WALK variant (the one the fused path uses when the feature
// dim is 1..4 fp32 and the image width a multiple of 4).
//
// Measured on B200 (scripts/microbench.cu): SHFL issues at 1 warp-instruction per
// clock per SM (a quarter of the FFMA rate), and a vector reduction RED.E.ADD.F32x4
// costs the same per lane as a scalar one (228 G lane-ops/s chip-wide).  The kernel
// above spends 75 shuffles per covered warp on its segmented reduction and 12 scalar /
// v2 reductions per (warp, face) group; this one uses neither:
//   * a warp owns 32 image rows x `strip` columns; LANE = ROW.  The lane walks along its
//     row and accumulates the 6 + 3*D partial sums of the current face in REGISTERS; when
//     face_idx changes it flushes them with (6+3D+3)/4 vector reductions into a padded
//     per-face accumulator (acc[face][16] for D = 3: 64-byte records, 16-byte aligned) and
//     reloads the face constants.  No shuffles, no match, no leader election;
//   * the pixel streams (face_idx 8 B, weights 12 B, upstream gradient 4*D B per pixel) are
//     staged per 4-column slab with 16-byte cp.async (LDGSTS) into rows padded to an odd
//     number of 16-byte chunks, double buffered, and read back with LDS.128 (conflict free:
//     8 consecutive rows cover the 32 banks).  9 KB of shared memory and <= 100 registers per
//     single-warp CTA keep ~20 warps per SM in flight (the first version, 8-column slabs at
//     162 registers, ran 9 warps per SM at 47 % issue utilisation: ncu, profiles/r2_*);
//   * raster_bwd_finalize_kernel unpacks acc into grad_face_vertices_image /
//     grad_face_features (which therefore need no memset).
// Per-pixel arithmetic is the reference's operation tree (dibr_math.cuh,
// raster_backward_geom / _feature) with the face-constant factors hoisted; the only
// change is g * (1 / k3^2) for g / k3^2 (<= 1 ulp per term).
constexpr int kRwSlab = 4;   // columns per staged slab (= the 4-pixel block a lane reads with LDS.128)

template <int DT>
struct RwCfg {
  // rows padded to an ODD number of 16-byte chunks: 8 consecutive rows then cover all 32 banks
  static constexpr int pad_odd(int bytes) { return ((bytes / 16) & 1) ? bytes : bytes + 16; }
  static constexpr int kIdxPitch = pad_odd(kRwSlab * 8);        // 32 -> 48
  static constexpr int kWPitch = pad_odd(kRwSlab * 12);         // 48
  static constexpr int kVals = 6 + 3 * DT;
  static constexpr int kAcc = (kVals + 3) & ~3;                 // floats per face record
};
// upstream-gradient rows: fp32 (16*D bytes, 16-byte chunks) or bf16 (8*D bytes; D odd -> 8-byte chunks,
// rows of 24 bytes are read with LDS.64: a half warp covers the 32 banks)
template <int DT, typename FT>
struct RwG {
  static constexpr int kRow = kRwSlab * DT * (int)sizeof(FT);
  static constexpr int kChunk = (kRow % 16) ? 8 : 16;
  static constexpr int kPitch = kChunk == 16 ? RwCfg<DT>::pad_odd(kRow) : kRow;
  static constexpr int kStage = 32 * (RwCfg<DT>::kIdxPitch + RwCfg<DT>::kWPitch + kPitch);
};
constexpr int kAccMax = 20;  // D = 4

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

struct RowBwdArgs {
  int B, H, W, F, strip, jobs_x, jobs_y;
  const void* grad_feat; const int64_t* idx; const float* w; const float* xy; const void* feat;   // FT: float | bf16
  float eps;
  float* acc;    // [B*F][RwCfg<D>::kAcc], zeroed
  int* job_ctr;  // [1] zeroed (lives right behind the records)
};

template <int DT>
struct RowFace {          // constants of the face a lane is currently accumulating
  float ax, ay, bx, by, cx, cy;
  float pp, n, m, q, k3, rk;
  float qk3, nk3n, ppk3n, mk3;  // q*k3, -(n*k3), -(pp*k3), m*k3  (dw1ds, dw1dt, dw2ds, dw2dt)
  float d1[DT], d2[DT];
};

template <int DT, typename FT>
__device__ __forceinline__ void row_face_load(const RowBwdArgs& a, int64_t face, RowFace<DT>& c) {
  const float2* pp = reinterpret_cast<const float2*>(a.xy + face * 6);
  const float2 pa = __ldg(pp), pb = __ldg(pp + 1), pc = __ldg(pp + 2);
  const FT* cf = static_cast<const FT*>(a.feat) + face * 3 * DT;
  float c0[DT], c1[DT], c2[DT];
#pragma unroll
  for (int d = 0; d < DT; ++d) { c0[d] = Feat<FT>::ld(cf + d); c1[d] = Feat<FT>::ld(cf + DT + d); c2[d] = Feat<FT>::ld(cf + 2 * DT + d); }
  c.ax = pa.x; c.ay = pa.y; c.bx = pb.x; c.by = pb.y; c.cx = pc.x; c.cy = pc.y;
  c.pp = fsub(c.by, c.ay); c.n = fsub(c.cx, c.ax); c.m = fsub(c.bx, c.ax); c.q = fsub(c.cy, c.ay);
  float k3 = ffma(c.m, c.q, -fmul(c.pp, c.n));
  {
    const double e = (f2u(k3) >> 31) ? -fabs((double)a.eps) : fabs((double)a.eps);
    k3 = d2f(dibr::dadd((double)k3, e));
  }
  c.k3 = k3;
  c.rk = fdiv(1.0f, fmul(k3, k3));
  c.qk3 = fmul(c.q, k3); c.nk3n = -fmul(c.n, k3); c.ppk3n = -fmul(c.pp, k3); c.mk3 = fmul(c.m, k3);
#pragma unroll
  for (int d = 0; d < DT; ++d) { c.d1[d] = fsub(c1[d], c0[d]); c.d2[d] = fsub(c2[d], c0[d]); }
}

template <int DT>
__device__ __forceinline__ void row_pixel(const RowFace<DT>& c, float aw, float bw, float cw, const float* g,
                                          float (&acc)[RwCfg<DT>::kAcc]) {
  const float y0 = ffma(c.cy, cw, ffma(c.ay, aw, fmul(c.by, bw)));
  const float x0 = ffma(c.cx, cw, ffma(c.ax, aw, fmul(c.bx, bw)));
  const float t = fsub(y0, c.ay), s = fsub(x0, c.ax);
  const float k1 = ffma(c.q, s, -fmul(c.n, t));
  const float k2 = ffma(c.m, t, -fmul(c.pp, s));
  const float tk3 = fmul(t, c.k3), sk3 = fmul(s, c.k3);
  const float dw1dm = -fmul(c.q, k1);
  const float dw2dm = ffma(-c.q, k2, tk3);
  const float dw1dn = ffma(c.pp, k1, -tk3);
  const float dw1dp = fmul(c.n, k1);
  const float dw1dq = ffma(-c.m, k1, sk3);
  const float dw2dp = ffma(c.n, k2, -sk3);
  const float dw2dn = fmul(c.pp, k2);
  const float dw2dq = -fmul(c.m, k2);
  const float n1ay = fadd(c.nk3n, fadd(dw1dp, dw1dq));
  const float n1ax = fadd(c.qk3, fadd(dw1dm, dw1dn));
  const float n2ax = fadd(c.ppk3n, fadd(dw2dm, dw2dn));
  const float n2ay = fadd(c.mk3, fadd(dw2dp, dw2dq));
#pragma unroll
  for (int d = 0; d < DT; ++d) {
    const float dl = fmul(g[d], c.rk);
    const float d1 = c.d1[d], d2 = c.d2[d];
    acc[0] = ffma(ffma(-n2ax, d2, -fmul(n1ax, d1)), dl, acc[0]);
    acc[1] = ffma(ffma(-n2ay, d2, -fmul(n1ay, d1)), dl, acc[1]);
    acc[2] = ffma(ffma(dw1dm, d1, fmul(dw2dm, d2)), dl, acc[2]);
    acc[3] = ffma(ffma(dw1dp, d1, fmul(dw2dp, d2)), dl, acc[3]);
    acc[4] = ffma(ffma(dw1dn, d1, fmul(dw2dn, d2)), dl, acc[4]);
    acc[5] = ffma(ffma(dw1dq, d1, fmul(dw2dq, d2)), dl, acc[5]);
    acc[6 + d] = ffma(g[d], aw, acc[6 + d]);
    acc[6 + DT + d] = ffma(g[d], bw, acc[6 + DT + d]);
    acc[6 + 2 * DT + d] = ffma(g[d], cw, acc[6 + 2 * DT + d]);
  }
}

#ifndef DIBR_ROWS_MINB
#define DIBR_ROWS_MINB 20
#endif
template <int DT, typename FT>
__global__ void __launch_bounds__(32, DIBR_ROWS_MINB) raster_bwd_rows_kernel(const __grid_constant__ RowBwdArgs a) {
  using C = RwCfg<DT>;
  using G = RwG<DT, FT>;
  __shared__ __align__(128) unsigned char smem[2 * G::kStage];
  const int lane = threadIdx.x;
  // persistent single-warp CTAs pull (view, 32-row band, column strip) jobs from a counter: the
  // jobs differ by 10x in cost (background vs dense mesh), so a static grid ends with a
  // ragged tail of half-empty SMs
  const int total_jobs = a.jobs_x * a.jobs_y * a.B;
  for (;;) {
  int job = 0;
  if (lane == 0) job = atomicAdd(a.job_ctr, 1);
  job = __shfl_sync(kFull, job, 0);
  if (job >= total_jobs) break;
  const int jx = job % a.jobs_x; job /= a.jobs_x;
  const int jy = job % a.jobs_y;
  const int b = job / a.jobs_y;
  const int row0 = jy * 32, col0 = jx * a.strip;
  const int col1 = min(a.W, col0 + a.strip);
  const int nslabs = (col1 - col0) / kRwSlab;
  const bool row_ok = row0 + lane < a.H;
  const int64_t pix0 = ((int64_t)b * a.H + row0) * a.W;  // first pixel of the job's first row
  const int64_t fbase = (int64_t)b * a.F;

  auto issue = [&](int s, int buf) {
    unsigned char* base = smem + buf * G::kStage;
    const int x = col0 + s * kRwSlab;
#pragma unroll
    for (int j = 0; j < 2; ++j) {           // face_idx: 2 chunks per row
      const int k = lane + 32 * j, r = k >> 1, ch = k & 1;
      if (row0 + r < a.H)
        cp_async16(base + r * C::kIdxPitch + ch * 16,
                   reinterpret_cast<const char*>(a.idx + pix0 + (int64_t)r * a.W + x) + ch * 16);
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {           // weights: 3 chunks per row
      const int k = lane + 32 * j, r = k / 3, ch = k - r * 3;
      if (row0 + r < a.H)
        cp_async16(base + 32 * C::kIdxPitch + r * C::kWPitch + ch * 16,
                   reinterpret_cast<const char*>(a.w + (pix0 + (int64_t)r * a.W + x) * 3) + ch * 16);
    }
    constexpr int GC = G::kRow / G::kChunk;   // upstream gradient: chunks per row
    const FT* gsrc = static_cast<const FT*>(a.grad_feat);
#pragma unroll
    for (int j = 0; j < GC; ++j) {
      const int k = lane + 32 * j, r = k / GC, ch = k - r * GC;
      if (row0 + r < a.H) {
        unsigned char* dst = base + 32 * (C::kIdxPitch + C::kWPitch) + r * G::kPitch + ch * G::kChunk;
        const char* src = reinterpret_cast<const char*>(gsrc + (pix0 + (int64_t)r * a.W + x) * DT) + ch * G::kChunk;
        if (G::kChunk == 16) cp_async16(dst, src); else cp_async8(dst, src);
      }
    }
    cp_async_commit();
  };

  int cur = -1;
  RowFace<DT> fc;
  float acc[C::kAcc];
#pragma unroll
  for (int i = 0; i < C::kAcc; ++i) acc[i] = 0.f;

  auto flush = [&]() {
    float4* p = reinterpret_cast<float4*>(a.acc + (fbase + cur) * C::kAcc);
#pragma unroll
    for (int i = 0; i < C::kAcc; i += 4) atomicAdd(p + (i >> 2), make_float4(acc[i], acc[i + 1], acc[i + 2], acc[i + 3]));
  };

  if (nslabs > 0) issue(0, 0);
  for (int s = 0; s < nslabs; ++s) {
    if (s + 1 < nslabs) { issue(s + 1, (s + 1) & 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncwarp();
    const unsigned char* base = smem + (s & 1) * G::kStage;
    if (row_ok) {
      do {
        const ulonglong2* ip = reinterpret_cast<const ulonglong2*>(base + lane * C::kIdxPitch);
        const ulonglong2 i01 = ip[0], i23 = ip[1];
        int f[4] = {(int)(long long)i01.x, (int)(long long)i01.y, (int)(long long)i23.x, (int)(long long)i23.y};
        bool any = cur >= 0;
#pragma unroll
        for (int p = 0; p < 4; ++p) { f[p] = f[p] < 0 ? -1 : f[p]; any = any || f[p] >= 0; }
        if (!any) break;
        // (prefetch.global.L1 of the block's upcoming face records here was measured slower: 0.319 vs 0.307 ms)
        const float4* wp = reinterpret_cast<const float4*>(base + 32 * C::kIdxPitch + lane * C::kWPitch);
        const float4 w0 = wp[0], w1 = wp[1], w2 = wp[2];
        const float wv[12] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w, w2.x, w2.y, w2.z, w2.w};
        float gv[4 * DT];
        {
          const unsigned char* grow = base + 32 * (C::kIdxPitch + C::kWPitch) + lane * G::kPitch;
          if (std::is_same<FT, float>::value) {
            const float4* gp = reinterpret_cast<const float4*>(grow);
#pragma unroll
            for (int k = 0; k < DT; ++k) { const float4 t = gp[k]; gv[4 * k] = t.x; gv[4 * k + 1] = t.y; gv[4 * k + 2] = t.z; gv[4 * k + 3] = t.w; }
          } else {   // bf16: 2 values per 32-bit word, low half first
            const uint2* gp = reinterpret_cast<const uint2*>(grow);
#pragma unroll
            for (int k = 0; k < DT; ++k) {
              const uint2 t = gp[k];
              gv[4 * k] = __uint_as_float(t.x << 16); gv[4 * k + 1] = __uint_as_float(t.x & 0xffff0000u);
              gv[4 * k + 2] = __uint_as_float(t.y << 16); gv[4 * k + 3] = __uint_as_float(t.y & 0xffff0000u);
            }
          }
        }
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          if (f[p] != cur) {
            if (cur >= 0) flush();
            cur = f[p];
            if (cur >= 0) {
              row_face_load<DT, FT>(a, fbase + cur, fc);
#pragma unroll
              for (int i = 0; i < C::kAcc; ++i) acc[i] = 0.f;
            }
          }
          if (cur >= 0) row_pixel<DT>(fc, wv[3 * p], wv[3 * p + 1], wv[3 * p + 2], &gv[DT * p], acc);
        }
      } while (false);
    }
    __syncwarp();  // everyone is done with this buffer before slab s+2 lands in it
  }
  if (cur >= 0) flush();
  __syncwarp();
  }  // job loop
}

// acc[face][kAcc] -> grad_face_vertices_image (NF,3,2) (= or +=) and grad_face_features (NF,3,D) (=).
// A CTA moves 256 face records through shared memory so that both the 64-byte records and the
// 24- / 12*D-byte output rows are read and written as contiguous, fully used lines.
template <int DT>
__global__ void __launch_bounds__(256) raster_bwd_finalize_kernel(const float* __restrict__ acc, int64_t NF,
                                                                 float* __restrict__ g_xy, float* __restrict__ g_ff,
                                                                 int accumulate_xy) {
  using C = RwCfg<DT>;
  constexpr int kFaces = 256;
  __shared__ __align__(16) float sm[kFaces * C::kAcc];
  const int64_t f0 = (int64_t)blockIdx.x * kFaces;
  const int nf = (int)min((int64_t)kFaces, NF - f0);
  const int tid = threadIdx.x;
  const float4* src = reinterpret_cast<const float4*>(acc + f0 * C::kAcc);
  for (int i = tid; i < nf * (C::kAcc / 4); i += 256) reinterpret_cast<float4*>(sm)[i] = __ldcs(src + i);
  __syncthreads();
  float2* gx = reinterpret_cast<float2*>(g_xy + f0 * 6);
  for (int i = tid; i < nf * 3; i += 256) {          // (face, vertex) -> float2
    const int f = i / 3, v = i - f * 3;
    float2 o = make_float2(sm[f * C::kAcc + 2 * v], sm[f * C::kAcc + 2 * v + 1]);
    if (accumulate_xy) { const float2 p = gx[i]; o.x += p.x; o.y += p.y; }
    gx[i] = o;
  }
  float* gf = g_ff + f0 * 3 * DT;
  for (int i = tid; i < nf * 3 * DT; i += 256) {
    const int f = i / (3 * DT), j = i - f * (3 * DT);
    gf[i] = sm[f * C::kAcc + 6 + j];
  }
}

// ---------------------------------------------------------------------------
// Soft-mask backward from stored K-lists (operator contract, dibr_soft_mask_cuda.cu:230-353).
struct SoftBwdListArgs {
  int B, H, W, F, K;
  PixelGrid grid;
  float sigmainv, multiplier;
  const float* grad_soft; const float* soft; const int64_t* idx;
  const float* prob; const int64_t* cidx; const uint8_t* ctype; const float* xy;
  float* grad_xy;
};

__global__ void __launch_bounds__(256) soft_bwd_lists_kernel(const __grid_constant__ SoftBwdListArgs a) {
  const int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t P = (int64_t)a.B * a.H * a.W;
  if (pix >= P) return;
  if (a.idx[pix] >= 0) return;
  const int ix = (int)(pix % a.W);
  const int iy = (int)((pix / a.W) % a.H);
  const int64_t b = pix / ((int64_t)a.W * a.H);
  const float x0 = pix_x(a.grid, ix), y0 = pix_y(a.grid, iy);
  const float dLdp = a.grad_soft[pix], allprob = a.soft[pix];
  for (int k = 0; k < a.K; ++k) {
    const int64_t f = a.cidx[pix * a.K + k];
    if (f < 0) break;
    const int64_t base = (b * a.F + f) * 6;
    float v[6], g[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) v[i] = __ldg(a.xy + base + i);
    soft_backward_terms(x0, y0, v, (int)a.ctype[pix * a.K + k] - 1, a.prob[pix * a.K + k], allprob,
                        dLdp, a.sigmainv, a.multiplier, g);
#pragma unroll
    for (int i = 0; i < 6; ++i)
      if (g[i] != 0.f) atomicAdd(a.grad_xy + base + i, g[i]);
  }
}

// ---------------------------------------------------------------------------
// Host side.
int levels_for(int H, int W) {
  int L = 1;
  while ((kTile << (2 * (L - 1))) < (H > W ? H : W)) ++L;
  return L;
}

int bins_per_view(int H, int W) {
  int nb = 0;
  const int L = levels_for(H, W);
  for (int l = 0; l < L; ++l) {
    const int t = kTile << (2 * l);
    nb += ((W + t - 1) / t) * ((H + t - 1) / t);
  }
  return nb;
}

// Workspace layout (all pieces 256-byte aligned):
//   cnt [2*B*NB] int + pool_ctr + fb_ctr + band_ctr | off [2*B*NB] int | fb_list, band_list [tiles] int |
//   entries [2*4*NF] int4 | acc [NF][<=20] f32 (rasterize backward) | pool_hdr [pool_tiles] int4 |
//   pool_data [pool_tiles][3][256*K] u32
struct Layout { size_t cnt, off, mode, ent, acc, base; };

Layout layout_for(int B, int64_t NF, int H, int W) {
  Layout L;
  const size_t tiles = (size_t)((W + kTile - 1) / kTile) * ((H + kTile - 1) / kTile) * B;
  L.cnt = align_up(((size_t)2 * B * bins_per_view(H, W) + 3 + B + tiles) * sizeof(int), 256);
  L.off = align_up((size_t)2 * B * bins_per_view(H, W) * sizeof(int), 256);
  L.mode = align_up(tiles * sizeof(int), 256) + align_up(tiles * kBandRec * sizeof(int), 256);
  L.ent = align_up((size_t)2 * 4 * (size_t)(NF > 0 ? NF : 1) * sizeof(int4), 256);
  L.acc = align_up((size_t)(NF > 0 ? NF : 1) * kAccMax * sizeof(float) + 16, 256);  // rasterize-backward face records + job counter
  L.base = L.cnt + L.off + L.mode + L.ent + L.acc + 256;
  return L;
}

size_t pool_aux_bytes(int K) {  // per-tile extras of the 3-kernel forward
  return K <= kEnumK ? sizeof(int) + 256 * sizeof(uint32_t) + (size_t)256 * kEnumK * sizeof(uint16_t) : 0;
}
size_t pool_block_bytes(int K) {
  return sizeof(int4) + pool_aux_bytes(K) + (size_t)3 * 256 * (size_t)K * sizeof(uint32_t);
}

int check_dims(int B, int64_t NF, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0 || NF < 0) return DIBR_B200_EINVAL;
  if (H > DIBR_B200_MAX_IMAGE_DIM || W > DIBR_B200_MAX_IMAGE_DIM || B > 65535) return DIBR_B200_ESIZE;
  if (NF > 0x3fffffffLL) return DIBR_B200_ESIZE;
  return 0;
}

// knum > 0 enables the hit cache in whatever the workspace holds beyond the minimum.
int setup_scene(Scene& s, int B, int64_t NF, int F, int H, int W, float multiplier, float margin,
                int knum, void* ws, size_t ws_bytes) {
  if (!(multiplier > 0.f)) return DIBR_B200_EINVAL;
  if (!ws) return DIBR_B200_EINVAL;
  const Layout Lo = layout_for(B, NF, H, W);
  char* p = (char*)align_up((size_t)ws, 256);
  char* const end = (char*)ws + ws_bytes;
  if (ws_bytes < Lo.base || p + Lo.cnt + Lo.off + Lo.mode + Lo.ent + Lo.acc > end) return DIBR_B200_EWORKSPACE;
  s.B = B; s.H = H; s.W = W; s.F = F; s.NF = NF;
  s.multiplier = multiplier; s.margin = margin;
  s.grid = make_grid(multiplier, W, H);
  s.L = levels_for(H, W);
  int nb = 0;
  for (int l = 0; l < kMaxLevels; ++l) {
    const int t = kTile << (2 * l);
    s.ntx[l] = l < s.L ? (W + t - 1) / t : 0;
    s.nty[l] = l < s.L ? (H + t - 1) / t : 0;
    s.bin_base[l] = nb;
    nb += s.ntx[l] * s.nty[l];
  }
  s.NB = nb;
  if ((int64_t)2 * B * nb >= 0x7fffffffLL) return DIBR_B200_ESIZE;  // counter ids are 32-bit
  s.cnt = (int*)p;
  s.pool_ctr = s.cnt + (size_t)2 * B * nb;
  s.fb_ctr = s.pool_ctr + 1;
  s.band_ctr = s.pool_ctr + 2;
  s.view_flag = s.pool_ctr + 3;
  s.tile_cnt = s.view_flag + B;
  p += Lo.cnt;
  s.off = (int*)p; p += Lo.off;
  s.fb_list = (int*)p;
  s.band_list = (int*)(p + align_up((size_t)s.ntx[0] * s.nty[0] * B * sizeof(int), 256));
  p += Lo.mode;
  s.entries = (int4*)p; p += Lo.ent;
  p += Lo.acc;
  s.pool_tiles = 0; s.pool_K = knum > 0 ? knum : 1; s.pool_hdr = nullptr; s.pool_data = nullptr;
  s.pool_na = nullptr; s.pool_aux = nullptr; s.pool_slots = nullptr;
  if (knum > 0) {
    const size_t left = (size_t)(end - p);
    const size_t data = (size_t)3 * 256 * (size_t)knum * sizeof(uint32_t);
    const bool aux = knum <= kEnumK;
    auto need = [&](size_t n) {
      size_t b = align_up(n * sizeof(int4), 256) + n * data;
      if (aux) b += align_up(n * sizeof(int), 256) + n * 256 * sizeof(uint32_t) +
                    align_up(n * 256 * kEnumK * sizeof(uint16_t), 256);
      return b;
    };
    size_t n = left / pool_block_bytes(knum);
    const size_t tiles = (size_t)s.ntx[0] * s.nty[0] * B;
    if (n > tiles) n = tiles;
    while (n > 0 && need(n) > left) --n;
    if (n > 0) {
      s.pool_tiles = (int)n;
      s.pool_hdr = (int4*)p; p += align_up(n * sizeof(int4), 256);
      if (aux) {
        s.pool_na = (int*)p; p += align_up(n * sizeof(int), 256);
        s.pool_aux = (uint32_t*)p; p += n * 256 * sizeof(uint32_t);
        s.pool_slots = (uint16_t*)p; p += align_up(n * 256 * kEnumK * sizeof(uint16_t), 256);
      }
      s.pool_data = (uint32_t*)p;
    }
  }
  return 0;
}

int build_bins(const Scene& s, int sets, cudaStream_t st) {
  const size_t zero_ints = (size_t)2 * s.B * s.NB + 3 + s.B + (size_t)s.ntx[0] * s.nty[0] * s.B;
  cudaError_t e = cudaMemsetAsync(s.cnt, 0, zero_ints * sizeof(int), st);
  if (e != cudaSuccess) return (int)e;
  if (s.NF > 0) {
    const bool agg = s.NF / s.B >= (int64_t)32 * s.ntx[0] * s.nty[0];
    const char* fb = getenv("DIBR_B200_BIN");          // "warp": match.any-aggregated atomics (measured SLOWER on
    const int warp_agg = (fb && fb[0] == 'w') ? 1 : 0; // the benchmark mesh: 98 + 89 vs 77 + 76 us; kept as an A/B switch)
    const int threads = agg ? kBinThreadsAgg : kBinThreadsPlain;
    const unsigned blocks = (unsigned)((s.NF + threads - 1) / threads);
    // dense meshes (tens of faces per 16x16 tile) hammer a few counters: aggregate per CTA
    {
      Span sp("bin_faces_kernel<count>", st);
      if (agg) bin_faces_kernel<false, true><<<blocks, threads, 0, st>>>(s, sets, 0);
      else bin_faces_kernel<false, false><<<blocks, threads, 0, st>>>(s, sets, warp_agg);
    }
    {
      Span sp("scan_bins_kernel", st);
      scan_bins_kernel<<<2 * s.B, 1024, 0, st>>>(s);
    }
    {
      Span sp("bin_faces_kernel<fill>", st);
      if (agg) bin_faces_kernel<true, true><<<blocks, threads, 0, st>>>(s, sets, 0);
      else bin_faces_kernel<true, false><<<blocks, threads, 0, st>>>(s, sets, warp_agg);
    }
  }
  return (int)cudaGetLastError();
}

dim3 tile_grid(const Scene& s) { return dim3((unsigned)s.ntx[0], (unsigned)s.nty[0], (unsigned)s.B); }

// Persistent kernels: one resident wave (SMs x CTAs that fit per SM), never more than the tiles.
// The wave size is a property of (device, kernel): queried once and cached in a per-instantiation
// table (idempotent writes of the same value, safe from any thread) - the occupancy / attribute
// queries cost ~0.1 ms of host time per step on small problems when repeated on every call.
struct WaveEntry { const void* kernel; int dev; int wave; };
constexpr int kWaveSlots = 64;
WaveEntry g_waves[kWaveSlots];   // append-only; a lost race re-queries and stores the same value again

template <typename Kernel>
unsigned persistent_grid(const Scene& s, Kernel kernel, size_t dyn_smem = 0) {
  int dev = 0;
  cudaGetDevice(&dev);
  const void* key = reinterpret_cast<const void*>(kernel);   // kernels with one signature share this template
  int wave = 0;
  for (int i = 0; i < kWaveSlots && g_waves[i].kernel; ++i)
    if (g_waves[i].kernel == key && g_waves[i].dev == dev) { wave = g_waves[i].wave; break; }
  if (wave == 0) {
    int sms = 148, per_sm = 2;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (dyn_smem > 48 * 1024)
      cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_smem);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, dyn_smem) != cudaSuccess ||
        per_sm < 1)
      per_sm = 2;
    wave = sms * per_sm;
    for (int i = 0; i < kWaveSlots; ++i)
      if (!g_waves[i].kernel) { g_waves[i].dev = dev; g_waves[i].wave = wave; g_waves[i].kernel = key; break; }
  }
  const int64_t ntiles = (int64_t)s.ntx[0] * s.nty[0] * s.B;
  return (unsigned)(ntiles < wave ? ntiles : wave);
}

template <bool R, bool S, bool K, typename FT = float>
void launch_fwd(const FwdArgs& a0, cudaStream_t st) {
  FwdArgs a = a0;
  a.from_fb = 0;
  {
    // S = 2 (32x32 px per CTA, candidates staged once for 4 tiles) when the mesh is sparse enough
    // for a 32x32 tile's candidates to fit one staging round and the grid still fills the GPU;
    // dense meshes / small images keep one tile per CTA.
    const char* force = getenv("DIBR_B200_FWD");   // "old" | "s1" | "s2": A/B switches
    const int64_t tiles32 = (int64_t)((a.s.W + 31) / 32) * ((a.s.H + 31) / 32);
    const int64_t faces_per_view = a.s.NF / (a.s.B > 0 ? a.s.B : 1);
    // ~ faces per 32x32 tile <= 40: c4 (20 k faces at 1024^2) has 20, c3 (512^2) 80, c2 80, c5 320;
    // measured: c4 0.86 (S=2) vs 0.90 ms (one tile per CTA), c3 0.75 vs 0.52 ms
    bool two = R && faces_per_view <= 40 * tiles32 && tiles32 * a.s.B >= 2048;
    if (force && force[0] == 's') two = force[1] == '2';
    const bool v2_single = force && force[0] == 's' && force[1] == '1';
    if ((force && force[0] == 'o') || (!two && !v2_single)) {
      // one 16x16 tile per CTA: dense meshes (hundreds of candidates per tile) and small images;
      // measured faster there than the v2 kernel with S = 1 (0.90 vs 1.17 ms on the benchmark mesh)
      Span sp("dibr_tile_fwd_kernel", st);
      dibr_tile_fwd_kernel<R, S, K, FT><<<tile_grid(a.s), kThreads, 0, st>>>(a);
    } else if (two) {
      Span sp("dibr_fwd2_kernel<S=2>", st);
      const dim3 grid((unsigned)((a.s.ntx[0] + 1) / 2), (unsigned)((a.s.nty[0] + 1) / 2), (unsigned)a.s.B);
      dibr_fwd2_kernel<R, S, K, FT, 2><<<grid, kThreads, 0, st>>>(a);
    } else {
      Span sp("dibr_fwd2_kernel<S=1>", st);
      dibr_fwd2_kernel<R, S, K, FT, 1><<<tile_grid(a.s), kThreads, 0, st>>>(a);
    }
  }
  if (S) {
    const unsigned g1 = persistent_grid(a.s, soft_tiles_fwd_kernel<K>, sizeof(SoftSmem));   // (sets the smem attribute once)
    if (!K && a.cache && a.s.pool_tiles > 0 && a.s.pool_slots != nullptr) {
      // enumerate -> evaluate densely -> fold; tiles beyond the cache take the single-kernel path
      {
        Span sp("soft_enum_kernel", st);
        soft_enum_kernel<<<persistent_grid(a.s, soft_enum_kernel), kThreads, 0, st>>>(a);
      }
      {
        Span sp("soft_eval_kernel", st);
        soft_eval_kernel<<<(unsigned)a.s.pool_tiles, kThreads, 0, st>>>(a);
      }
      a.from_fb = 1;
      a.cache = 0;
      Span sp("soft_tiles_fwd_kernel<leftovers>", st);
      soft_tiles_fwd_kernel<K><<<g1, kThreads, sizeof(SoftSmem), st>>>(a);
    } else {
      Span sp("soft_tiles_fwd_kernel", st);
      soft_tiles_fwd_kernel<K><<<g1, kThreads, sizeof(SoftSmem), st>>>(a);
    }
  }
}

template <typename FT>
int launch_raster_bwd(const RasterBwdArgs& a, cudaStream_t st) {
  const dim3 grid((unsigned)a.ntx, (unsigned)a.nty, (unsigned)a.B);
  Span sp("raster_bwd_kernel", st);
  switch (a.D) {
    case 1: raster_bwd_kernel<1, FT><<<grid, kThreads, 0, st>>>(a); break;
    case 2: raster_bwd_kernel<2, FT><<<grid, kThreads, 0, st>>>(a); break;
    case 3: raster_bwd_kernel<3, FT><<<grid, kThreads, 0, st>>>(a); break;
    case 4: raster_bwd_kernel<4, FT><<<grid, kThreads, 0, st>>>(a); break;
    default: raster_bwd_kernel<0, FT><<<grid, kThreads, 0, st>>>(a); break;
  }
  return (int)cudaGetLastError();
}

// The face-record region of a workspace (nullptr: none / too small -> warp-reduction kernel).
float* acc_region(void* ws, size_t ws_bytes, int B, int64_t NF, int H, int W) {
  if (!ws) return nullptr;
  const Layout Lo = layout_for(B, NF, H, W);
  char* p = (char*)align_up((size_t)ws, 256);
  if (ws_bytes < Lo.base || p + Lo.cnt + Lo.off + Lo.mode + Lo.ent + Lo.acc > (char*)ws + ws_bytes) return nullptr;
  return (float*)(p + Lo.cnt + Lo.off + Lo.mode + Lo.ent);
}

template <int DT, typename FT>
int launch_rows_t(const RowBwdArgs& a0, int64_t NF, float* g_xy, float* g_ff, int accumulate_xy, cudaStream_t st) {
  RowBwdArgs a = a0;
  a.job_ctr = reinterpret_cast<int*>(a.acc + (size_t)NF * RwCfg<DT>::kAcc);   // kAcc <= 16 < kAccMax: room behind the records
  cudaError_t e = cudaMemsetAsync(a.acc, 0, (size_t)NF * RwCfg<DT>::kAcc * sizeof(float) + sizeof(int), st);
  if (e != cudaSuccess) return (int)e;
  {
    Span sp("raster_bwd_rows_kernel", st);
    // resident single-warp CTAs per device: a property of (device, kernel), cached after the first
    // query (idempotent writes of the same value: safe from any thread)
    static int slots_of[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    int slots = slots_of[dev & 63];
    if (slots == 0) {
      int sms = 148, per_sm = 16;
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, raster_bwd_rows_kernel<DT, FT>, 32, 0) != cudaSuccess || per_sm < 1)
        per_sm = 16;
      slots = sms * per_sm;
      slots_of[dev & 63] = slots;
    }
    const int64_t jobs = (int64_t)a.jobs_x * a.jobs_y * a.B;
    raster_bwd_rows_kernel<DT, FT><<<(unsigned)(jobs < slots ? jobs : slots), 32, 0, st>>>(a);
  }
  {
    Span sp("raster_bwd_finalize_kernel", st);
    raster_bwd_finalize_kernel<DT><<<(unsigned)((NF + 255) / 256), 256, 0, st>>>(a.acc, NF, g_xy, g_ff, accumulate_xy);
  }
  return (int)cudaGetLastError();
}

// Row-walk rasterize backward: one warp per 32 rows x strip columns; the strip is as long as
// still leaves a few waves of single-warp CTAs (longer strips = fewer cut face runs).
template <typename FT>
int launch_raster_bwd_rows(const RasterBwdArgs& r, float* acc, int accumulate_xy, cudaStream_t st) {
  RowBwdArgs a;
  a.B = r.B; a.H = r.H; a.W = r.W; a.F = r.F;
  a.grad_feat = r.grad_feat; a.idx = r.idx; a.w = r.w; a.xy = r.xy;
  a.feat = r.feat; a.eps = r.eps; a.acc = acc;
  a.jobs_y = (r.H + 31) / 32;
  int strip = 32;   // measured on the benchmark scene: 128 -> 0.494, 64 -> 0.526, 32 -> 0.542 of HBM peak
  if (const char* fs = getenv("DIBR_B200_ROWS_STRIP")) { const int v = atoi(fs); if (v >= kRwSlab && v % kRwSlab == 0) strip = v; }
  while (strip > kRwSlab && (int64_t)r.B * a.jobs_y * ((r.W + strip - 1) / strip) < 8192) strip >>= 1;
  a.strip = strip;
  a.jobs_x = (r.W + strip - 1) / strip;
  const int64_t NF = (int64_t)r.B * r.F;
  switch (r.D) {
    case 1: return launch_rows_t<1, FT>(a, NF, r.grad_xy, r.grad_feat_out, accumulate_xy, st);
    case 2: return launch_rows_t<2, FT>(a, NF, r.grad_xy, r.grad_feat_out, accumulate_xy, st);
    case 3: return launch_rows_t<3, FT>(a, NF, r.grad_xy, r.grad_feat_out, accumulate_xy, st);
    case 4: return launch_rows_t<4, FT>(a, NF, r.grad_xy, r.grad_feat_out, accumulate_xy, st);
    default: return DIBR_B200_EINVAL;
  }
}

#include "dibr_f64.cuh"

}  // namespace

// ===========================================================================
extern "C" {

size_t dibr_b200_workspace_bytes_f64(int batch, int64_t total_faces, int height, int width) {
  if (check_dims(batch, total_faces, height, width)) return 0;
  return f64_layout(batch, total_faces, height, width).total;
}

int dibr_b200_forward_f64(int batch, int num_faces, int height, int width, int feat_dim,
                          const double* face_vertices_z, const double* face_vertices_image,
                          const double* face_features, const double* face_normals_z, const uint8_t* valid_faces,
                          float multiplier, float eps, int mode, float sigmainv, double boxlen_m, int knum,
                          double* interpolated_features, int64_t* face_idx, double* output_weights,
                          double* soft_mask, void* workspace, size_t workspace_bytes_, dibr_b200_stream_t stream) {
  const int64_t NF = (int64_t)batch * num_faces;
  int rc = check_dims(batch, NF, height, width);
  if (rc) return rc;
  const bool raster = mode & DIBR_B200_RASTER, soft = mode & DIBR_B200_SOFT_MASK;
  if ((!raster && !soft) || num_faces < 0 || feat_dim < 0 || !face_idx || !(multiplier > 0.f)) return DIBR_B200_EINVAL;
  if (num_faces > 0 && !face_vertices_image) return DIBR_B200_EINVAL;
  if (raster && (!output_weights || (feat_dim > 0 && (!interpolated_features || (num_faces > 0 && !face_features))) ||
                 (num_faces > 0 && !face_vertices_z)))
    return DIBR_B200_EINVAL;
  if (soft && (!soft_mask || knum <= 0)) return DIBR_B200_EINVAL;
  if (misaligned(face_vertices_z, face_vertices_image, face_features, face_normals_z, valid_faces,
                 interpolated_features, face_idx, output_weights, soft_mask))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  F64Args a;
  rc = f64_setup(a, batch, num_faces, height, width, face_vertices_image, face_normals_z, valid_faces, multiplier,
                 boxlen_m, (raster ? 1 : 0) | (soft ? 2 : 0), true, workspace, workspace_bytes_, st);
  if (rc) return rc;
  a.D = feat_dim; a.K = knum; a.mode = mode; a.eps = eps; a.sigmainv = sigmainv; a.multiplier = multiplier;
  a.margin = boxlen_m; a.xy = face_vertices_image; a.z = face_vertices_z; a.feat = face_features;
  a.out_feat = interpolated_features; a.idx = face_idx; a.out_w = output_weights; a.out_soft = soft_mask;
  a.g_feat = nullptr; a.g_soft = nullptr; a.soft = nullptr; a.g_xy = nullptr; a.g_ff = nullptr;
  Span sp("dibr_f64_kernel<forward>", st);
  dibr_f64_kernel<false><<<tile_grid(a.s), kThreads, 0, st>>>(a);
  return (int)cudaGetLastError();
}

int dibr_b200_backward_f64(int batch, int num_faces, int height, int width, int feat_dim,
                           const double* grad_features, const double* grad_soft_mask, const int64_t* face_idx,
                           const double* output_weights, const double* soft_mask, const double* face_vertices_image,
                           const double* face_features, float multiplier, float eps, float sigmainv, double boxlen_m,
                           int knum, double* grad_face_vertices_image, double* grad_face_features, void* workspace,
                           size_t workspace_bytes_, int flags, dibr_b200_stream_t stream) {
  const int64_t NF = (int64_t)batch * num_faces;
  int rc = check_dims(batch, NF, height, width);
  if (rc) return rc;
  if (!face_idx || !grad_face_vertices_image || num_faces < 0 || feat_dim < 0 || !(multiplier > 0.f)) return DIBR_B200_EINVAL;
  if (num_faces > 0 && !face_vertices_image) return DIBR_B200_EINVAL;
  const bool run_raster = grad_features && feat_dim > 0;
  if (run_raster && NF > 0 && (!output_weights || !face_features || !grad_face_features)) return DIBR_B200_EINVAL;
  if (grad_soft_mask && (!soft_mask || knum <= 0)) return DIBR_B200_EINVAL;
  if (misaligned(grad_features, grad_soft_mask, face_idx, output_weights, soft_mask, face_vertices_image,
                 face_features, grad_face_vertices_image, grad_face_features))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(grad_face_vertices_image, 0, (size_t)NF * 6 * sizeof(double), st);
  if (e != cudaSuccess) return (int)e;
  if (grad_face_features && feat_dim > 0) {
    e = cudaMemsetAsync(grad_face_features, 0, (size_t)NF * 3 * feat_dim * sizeof(double), st);
    if (e != cudaSuccess) return (int)e;
  }
  if (NF == 0 || (!run_raster && !grad_soft_mask)) return 0;
  F64Args a;
  // the soft-mask branch needs the enlarged bins: forward's (BINS_VALID) or rebuilt here
  rc = f64_setup(a, batch, num_faces, height, width, face_vertices_image, nullptr, nullptr, multiplier, boxlen_m, 2,
                 grad_soft_mask && !(flags & DIBR_B200_BINS_VALID), workspace, workspace_bytes_, st);
  if (rc) return rc;
  a.D = feat_dim; a.K = knum; a.mode = 0; a.eps = eps; a.sigmainv = sigmainv; a.multiplier = multiplier;
  a.margin = boxlen_m; a.xy = face_vertices_image; a.z = nullptr; a.feat = face_features;
  a.out_feat = nullptr; a.idx = const_cast<int64_t*>(face_idx); a.out_w = const_cast<double*>(output_weights);
  a.out_soft = nullptr; a.g_feat = run_raster ? grad_features : nullptr; a.g_soft = grad_soft_mask; a.soft = soft_mask;
  a.g_xy = grad_face_vertices_image; a.g_ff = grad_face_features;
  Span sp("dibr_f64_kernel<backward>", st);
  dibr_f64_kernel<true><<<tile_grid(a.s), kThreads, 0, st>>>(a);
  return (int)cudaGetLastError();
}

int dibr_b200_packed_rasterize_forward_f64(int batch, int64_t total_faces, int height, int width, int feat_dim,
                                           const double* face_vertices_z, const double* face_vertices_image,
                                           const double* face_bboxes, const double* face_features,
                                           const int64_t* first_idx_face_per_mesh, float multiplier, float eps,
                                           double* interpolated_features, int64_t* selected_face_idx,
                                           double* output_weights, void* workspace, size_t workspace_bytes_,
                                           dibr_b200_stream_t stream) {
  int rc = check_dims(batch, total_faces, height, width);
  if (rc) return rc;
  if (!selected_face_idx || !output_weights || !first_idx_face_per_mesh || feat_dim < 0 || !(multiplier > 0.f))
    return DIBR_B200_EINVAL;
  if (feat_dim > 0 && (!interpolated_features || (total_faces > 0 && !face_features))) return DIBR_B200_EINVAL;
  if (total_faces > 0 && (!face_vertices_z || !face_vertices_image || !face_bboxes)) return DIBR_B200_EINVAL;
  if (misaligned(face_vertices_z, face_vertices_image, face_bboxes, face_features, first_idx_face_per_mesh,
                 interpolated_features, selected_face_idx, output_weights))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  F64OpArgs a;
  a.D = feat_dim; a.K = 0; a.eps = eps; a.sigmainv = 0.f; a.multiplier = multiplier;
  a.xy = face_vertices_image; a.z = face_vertices_z; a.feat = face_features; a.box = face_bboxes;
  a.out_feat = interpolated_features; a.idx = selected_face_idx; a.out_w = output_weights; a.out_soft = nullptr;
  a.prob = nullptr; a.cidx = nullptr; a.ctype = nullptr;
  rc = f64_op_setup(a, batch, total_faces, 0, height, width, first_idx_face_per_mesh, multiplier, 1, workspace,
                    workspace_bytes_, st);
  if (rc) return rc;
  Span sp("f64_raster_op_kernel", st);
  f64_raster_op_kernel<<<tile_grid(a.s), kThreads, 0, st>>>(a);
  return (int)cudaGetLastError();
}

int dibr_b200_rasterize_backward_f64(int batch, int num_faces, int height, int width, int feat_dim,
                                     const double* grad_interpolated_features, const int64_t* selected_face_idx,
                                     const double* output_weights, const double* face_vertices_image,
                                     const double* face_features, float eps, double* grad_face_vertices_image,
                                     double* grad_face_features, dibr_b200_stream_t stream) {
  const int64_t NF = (int64_t)batch * num_faces;
  int rc = check_dims(batch, NF, height, width);
  if (rc) return rc;
  if (!selected_face_idx || !grad_face_vertices_image || num_faces < 0 || feat_dim < 0) return DIBR_B200_EINVAL;
  if (feat_dim > 0 && (!grad_interpolated_features || !output_weights || !grad_face_features ||
                       (num_faces > 0 && !face_features)))
    return DIBR_B200_EINVAL;
  if (num_faces > 0 && !face_vertices_image) return DIBR_B200_EINVAL;
  if (misaligned(grad_interpolated_features, selected_face_idx, output_weights, face_vertices_image, face_features,
                 grad_face_vertices_image, grad_face_features))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(grad_face_vertices_image, 0, (size_t)NF * 6 * sizeof(double), st);
  if (e != cudaSuccess) return (int)e;
  if (feat_dim > 0) {
    e = cudaMemsetAsync(grad_face_features, 0, (size_t)NF * 3 * feat_dim * sizeof(double), st);
    if (e != cudaSuccess) return (int)e;
  }
  if (NF == 0 || feat_dim == 0) return 0;
  F64Args a = {};
  a.s.B = batch; a.s.H = height; a.s.W = width; a.s.F = num_faces;
  a.D = feat_dim; a.eps = eps; a.xy = face_vertices_image; a.feat = face_features;
  a.idx = const_cast<int64_t*>(selected_face_idx); a.out_w = const_cast<double*>(output_weights);
  a.g_feat = grad_interpolated_features; a.g_xy = grad_face_vertices_image; a.g_ff = grad_face_features;
  const int64_t P = (int64_t)batch * height * width;
  Span sp("f64_raster_bwd_op_kernel", st);
  f64_raster_bwd_op_kernel<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(a);
  return (int)cudaGetLastError();
}

int dibr_b200_soft_mask_forward_f64(int batch, int num_faces, int height, int width, int knum,
                                    const double* face_vertices_image, const double* face_large_bboxes,
                                    const int64_t* selected_face_idx, float sigmainv, float multiplier,
                                    double* soft_mask, double* close_face_prob, int64_t* close_face_idx,
                                    uint8_t* close_face_dist_type, void* workspace, size_t workspace_bytes_,
                                    dibr_b200_stream_t stream) {
  const int64_t NF = (int64_t)batch * num_faces;
  int rc = check_dims(batch, NF, height, width);
  if (rc) return rc;
  if (!selected_face_idx || !soft_mask || knum <= 0 || num_faces < 0 || !(multiplier > 0.f)) return DIBR_B200_EINVAL;
  if (num_faces > 0 && (!face_vertices_image || !face_large_bboxes)) return DIBR_B200_EINVAL;
  const bool lists = close_face_prob || close_face_idx || close_face_dist_type;
  if (lists && !(close_face_prob && close_face_idx && close_face_dist_type)) return DIBR_B200_EINVAL;
  if (lists && (int64_t)batch * height * width * knum < 0) return DIBR_B200_ESIZE;
  if (misaligned(face_vertices_image, face_large_bboxes, selected_face_idx, soft_mask, close_face_prob,
                 close_face_idx, close_face_dist_type))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  F64OpArgs a;
  a.D = 0; a.K = knum; a.eps = 0.f; a.sigmainv = sigmainv; a.multiplier = multiplier;
  a.xy = face_vertices_image; a.z = nullptr; a.feat = nullptr; a.box = face_large_bboxes;
  a.out_feat = nullptr; a.idx = const_cast<int64_t*>(selected_face_idx); a.out_w = nullptr; a.out_soft = soft_mask;
  a.prob = close_face_prob; a.cidx = close_face_idx; a.ctype = close_face_dist_type;
  rc = f64_op_setup(a, batch, NF, num_faces, height, width, nullptr, multiplier, 2, workspace, workspace_bytes_, st);
  if (rc) return rc;
  Span sp("f64_soft_op_kernel", st);
  f64_soft_op_kernel<<<tile_grid(a.s), kThreads, 0, st>>>(a);
  return (int)cudaGetLastError();
}

int dibr_b200_soft_mask_backward_f64(int batch, int num_faces, int height, int width, int knum,
                                     const double* grad_soft_mask, const double* soft_mask,
                                     const int64_t* selected_face_idx, const double* close_face_prob,
                                     const int64_t* close_face_idx, const uint8_t* close_face_dist_type,
                                     const double* face_vertices_image, float sigmainv, float multiplier,
                                     double* grad_face_vertices_image, dibr_b200_stream_t stream) {
  const int64_t NF = (int64_t)batch * num_faces;
  int rc = check_dims(batch, NF, height, width);
  if (rc) return rc;
  if (!grad_soft_mask || !soft_mask || !selected_face_idx || !close_face_prob || !close_face_idx ||
      !close_face_dist_type || !grad_face_vertices_image || knum <= 0 || num_faces < 0 || !(multiplier > 0.f))
    return DIBR_B200_EINVAL;
  if (num_faces > 0 && !face_vertices_image) return DIBR_B200_EINVAL;
  if (misaligned(grad_soft_mask, soft_mask, selected_face_idx, close_face_prob, close_face_idx,
                 close_face_dist_type, face_vertices_image, grad_face_vertices_image))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(grad_face_vertices_image, 0, (size_t)NF * 6 * sizeof(double), st);
  if (e != cudaSuccess) return (int)e;
  if (NF == 0) return 0;
  F64SoftBwdArgs a;
  a.B = batch; a.H = height; a.W = width; a.F = num_faces; a.K = knum;
  a.grid = make_grid(multiplier, width, height);
  a.sigmainv = sigmainv; a.multiplier = multiplier;
  a.grad_soft = grad_soft_mask; a.soft = soft_mask; a.idx = selected_face_idx;
  a.prob = close_face_prob; a.cidx = close_face_idx; a.ctype = close_face_dist_type;
  a.xy = face_vertices_image; a.grad_xy = grad_face_vertices_image;
  const int64_t P = (int64_t)batch * height * width;
  Span sp("f64_soft_bwd_op_kernel", st);
  f64_soft_bwd_op_kernel<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(a);
  return (int)cudaGetLastError();
}

int dibr_b200_trace_begin(void) {
  g_trace.on = true;
  g_trace.used = 0;
  g_trace.names.clear();
  return 0;
}

int dibr_b200_trace_end(char* names, size_t names_bytes, float* ms, int capacity) {
  TraceState& t = g_trace;
  t.on = false;
  const int n = t.used / 2;
  std::string joined;
  for (int i = 0; i < n; ++i) {
    if (cudaEventSynchronize(t.pool[2 * i + 1]) != cudaSuccess) return DIBR_B200_EINVAL;
    float v = 0.f;
    if (cudaEventElapsedTime(&v, t.pool[2 * i], t.pool[2 * i + 1]) != cudaSuccess) return DIBR_B200_EINVAL;
    if (ms && i < capacity) ms[i] = v;
    joined += t.names[i];
    joined += '\n';
  }
  if (names && names_bytes > 0) {
    const size_t c = joined.size() < names_bytes - 1 ? joined.size() : names_bytes - 1;
    memcpy(names, joined.data(), c);
    names[c] = 0;
  }
  t.used = 0;
  t.names.clear();
  return n;
}

int dibr_b200_version(void) { return 200; }

size_t dibr_b200_workspace_bytes(int batch, int64_t total_faces, int height, int width) {
  if (check_dims(batch, total_faces, height, width)) return 0;
  return layout_for(batch, total_faces, height, width).base;
}

size_t dibr_b200_workspace_bytes_cached(int batch, int64_t total_faces, int height, int width,
                                        int knum, int64_t cache_tiles) {
  if (check_dims(batch, total_faces, height, width) || knum <= 0 || cache_tiles < 0) return 0;
  const int64_t tiles = (int64_t)((width + kTile - 1) / kTile) * ((height + kTile - 1) / kTile) * batch;
  if (cache_tiles > tiles) cache_tiles = tiles;
  return layout_for(batch, total_faces, height, width).base + 512 +
         (size_t)cache_tiles * pool_block_bytes(knum);
}

static int forward_impl(int batch, int num_faces, int height, int width, int feat_dim,
                        const float* face_vertices_z, const float* face_vertices_image,
                        const void* face_features, const float* face_normals_z,
                        const uint8_t* valid_faces, float multiplier, float eps, int mode,
                        float sigmainv, float boxlen_m, int knum, void* interpolated_features,
                        int64_t* face_idx, float* output_weights, float* soft_mask, void* workspace,
                        size_t workspace_bytes_, dibr_b200_stream_t stream, bool bf16) {
  const int64_t NF = (int64_t)batch * num_faces;
  int rc = check_dims(batch, NF, height, width);
  if (rc) return rc;
  const bool raster = mode & DIBR_B200_RASTER, soft = mode & DIBR_B200_SOFT_MASK;
  if ((!raster && !soft) || num_faces < 0 || feat_dim < 0 || !face_idx) return DIBR_B200_EINVAL;
  if (num_faces > 0 && !face_vertices_image) return DIBR_B200_EINVAL;
  if (raster && (!output_weights || (feat_dim > 0 && (!interpolated_features || (num_faces > 0 && !face_features))) ||
                 (num_faces > 0 && !face_vertices_z)))
    return DIBR_B200_EINVAL;
  if (soft && (!soft_mask || knum <= 0)) return DIBR_B200_EINVAL;
  if (misaligned(face_vertices_z, face_vertices_image, face_features, face_normals_z, valid_faces,
                 interpolated_features, face_idx, output_weights, soft_mask))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  FwdArgs a;
  Scene& s = a.s;
  rc = setup_scene(s, batch, NF, num_faces, height, width, multiplier, boxlen_m, soft ? knum : 0,
                   workspace, workspace_bytes_);
  if (rc) return rc;
  s.first = nullptr; s.xy = face_vertices_image; s.z = face_vertices_z; s.premultiplied = 0;
  s.fnz = face_normals_z; s.valid = valid_faces; s.bbox_tight = nullptr; s.bbox_large = nullptr;
  rc = build_bins(s, (raster ? 1 : 0) | (soft ? 2 : 0), st);
  if (rc) return rc;
  a.rc = make_raster_const(eps);
  a.D = feat_dim; a.feat = face_features; a.sigmainv = sigmainv; a.K = knum;
  a.cache = soft ? 1 : 0;   // hits are cached while blocks last; other tiles go to fb_list
  a.out_feat = interpolated_features; a.idx = face_idx; a.out_w = output_weights; a.out_soft = soft_mask;
  a.kl = SoftFwdOut{nullptr, nullptr, nullptr};
  if (raster && soft) { if (bf16) launch_fwd<true, true, false, __nv_bfloat16>(a, st); else launch_fwd<true, true, false>(a, st); }
  else if (raster) { if (bf16) launch_fwd<true, false, false, __nv_bfloat16>(a, st); else launch_fwd<true, false, false>(a, st); }
  else launch_fwd<false, true, false>(a, st);
  return (int)cudaGetLastError();
}

int dibr_b200_forward(int batch, int num_faces, int height, int width, int feat_dim,
                      const float* face_vertices_z, const float* face_vertices_image,
                      const float* face_features, const float* face_normals_z,
                      const uint8_t* valid_faces, float multiplier, float eps, int mode,
                      float sigmainv, float boxlen_m, int knum, float* interpolated_features,
                      int64_t* face_idx, float* output_weights, float* soft_mask, void* workspace,
                      size_t workspace_bytes_, dibr_b200_stream_t stream) {
  return forward_impl(batch, num_faces, height, width, feat_dim, face_vertices_z, face_vertices_image,
                      face_features, face_normals_z, valid_faces, multiplier, eps, mode, sigmainv, boxlen_m,
                      knum, interpolated_features, face_idx, output_weights, soft_mask, workspace,
                      workspace_bytes_, stream, false);
}

int dibr_b200_forward_bf16(int batch, int num_faces, int height, int width, int feat_dim,
                           const float* face_vertices_z, const float* face_vertices_image,
                           const uint16_t* face_features, const float* face_normals_z,
                           const uint8_t* valid_faces, float multiplier, float eps, int mode,
                           float sigmainv, float boxlen_m, int knum, uint16_t* interpolated_features,
                           int64_t* face_idx, float* output_weights, float* soft_mask, void* workspace,
                           size_t workspace_bytes_, dibr_b200_stream_t stream) {
  return forward_impl(batch, num_faces, height, width, feat_dim, face_vertices_z, face_vertices_image,
                      face_features, face_normals_z, valid_faces, multiplier, eps, mode, sigmainv, boxlen_m,
                      knum, interpolated_features, face_idx, output_weights, soft_mask, workspace,
                      workspace_bytes_, stream, true);
}


static int backward_impl(int batch, int num_faces, int height, int width, int feat_dim,
                         const void* grad_features, const float* grad_soft_mask,
                         const int64_t* face_idx, const float* output_weights, const float* soft_mask,
                         const float* face_vertices_image, const void* face_features,
                         float multiplier, float eps, float sigmainv, float boxlen_m, int knum,
                         float* grad_face_vertices_image, float* grad_face_features, void* workspace,
                         size_t workspace_bytes_, int flags, dibr_b200_stream_t stream, bool bf16,
                         int view_begin, int view_end) {
  const int64_t NF = (int64_t)batch * num_faces;
  const bool bins_valid = (flags & DIBR_B200_BINS_VALID) != 0;
  int rc = check_dims(batch, NF, height, width);
  if (rc) return rc;
  if (!face_idx || !grad_face_vertices_image || num_faces < 0 || feat_dim < 0) return DIBR_B200_EINVAL;
  if (num_faces > 0 && !face_vertices_image) return DIBR_B200_EINVAL;
  if (view_begin < 0 || view_end > batch || view_begin >= view_end) return DIBR_B200_EINVAL;
  if (misaligned(grad_features, grad_soft_mask, face_idx, output_weights, soft_mask, face_vertices_image,
                 face_features, grad_face_vertices_image, grad_face_features))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaSuccess;
  const bool run_raster = grad_features && feat_dim > 0;
  // the views of this call: rows [view_begin, view_end) of every per-view tensor
  const int nv = view_end - view_begin;
  const int64_t NFv = (int64_t)nv * num_faces;
  const size_t fsz = bf16 ? 2 : 4;
  float* const g_xy_v = grad_face_vertices_image + (size_t)view_begin * num_faces * 6;
  float* const g_ff_v = grad_face_features ? grad_face_features + (size_t)view_begin * num_faces * 3 * feat_dim : nullptr;
  // row-walk kernel: fp32 or bf16 features, D <= 4, rows a multiple of 4 px, a workspace with the face records
  float* acc = nullptr;
  if (run_raster && feat_dim <= 4 && (width % kRwSlab) == 0 && NF > 0) {
    const char* force = getenv("DIBR_B200_RASTER_BWD");   // "warp": A/B against the warp-reduction kernel
    if (!(force && force[0] == 'w')) acc = acc_region(workspace, workspace_bytes_, batch, NF, height, width);
  }
  if (!(flags & DIBR_B200_ACCUMULATE) && !acc) {
    e = cudaMemsetAsync(g_xy_v, 0, (size_t)NFv * 6 * sizeof(float), st);
    if (e != cudaSuccess) return (int)e;
  }
  if (grad_face_features && feat_dim > 0 && (grad_features || !(flags & DIBR_B200_ACCUMULATE)) && !acc) {
    e = cudaMemsetAsync(g_ff_v, 0, (size_t)NFv * 3 * feat_dim * sizeof(float), st);
    if (e != cudaSuccess) return (int)e;
  }
  if (NF == 0) return 0;
  if (run_raster) {
    if (!output_weights || !face_features || !grad_face_features) return DIBR_B200_EINVAL;
    RasterBwdArgs a;
    const size_t px0 = (size_t)view_begin * height * width;
    a.B = nv; a.H = height; a.W = width; a.F = num_faces; a.D = feat_dim;
    a.ntx = (width + kTile - 1) / kTile; a.nty = (height + kTile - 1) / kTile;
    a.grad_feat = static_cast<const char*>(grad_features) + px0 * feat_dim * fsz;
    a.idx = face_idx + px0; a.w = output_weights + px0 * 3;
    a.xy = face_vertices_image + (size_t)view_begin * num_faces * 6;
    a.feat = static_cast<const char*>(face_features) + (size_t)view_begin * num_faces * 3 * feat_dim * fsz;
    a.eps = eps; a.grad_xy = g_xy_v;
    a.grad_feat_out = g_ff_v;
    if (acc) rc = bf16 ? launch_raster_bwd_rows<__nv_bfloat16>(a, acc, (flags & DIBR_B200_ACCUMULATE) ? 1 : 0, st)
                       : launch_raster_bwd_rows<float>(a, acc, (flags & DIBR_B200_ACCUMULATE) ? 1 : 0, st);
    else rc = bf16 ? launch_raster_bwd<__nv_bfloat16>(a, st) : launch_raster_bwd<float>(a, st);
    if (rc) return rc;
  }
  if (grad_soft_mask) {
    if (!soft_mask || knum <= 0) return DIBR_B200_EINVAL;
    SoftBwdArgs a;
    rc = setup_scene(a.s, batch, NF, num_faces, height, width, multiplier, boxlen_m, knum, workspace,
                     workspace_bytes_);
    if (rc) return rc;
    Scene& s = a.s;
    s.first = nullptr; s.xy = face_vertices_image; s.z = nullptr; s.premultiplied = 0;
    s.fnz = nullptr; s.valid = nullptr; s.bbox_tight = nullptr; s.bbox_large = nullptr;
    a.sigmainv = sigmainv; a.K = knum; a.grad_soft = grad_soft_mask; a.soft = soft_mask;
    a.idx = face_idx; a.grad_xy = grad_face_vertices_image;
    a.view_begin = view_begin; a.view_end = view_end;
    const unsigned persistent = persistent_grid(s, dibr_tile_soft_bwd_kernel);
    if (!bins_valid) {
      // no forward state: rebuild the large bins and recompute every tile
      rc = build_bins(s, 2, st);
      if (rc) return rc;
      a.from_list = 0;
      Span sp("dibr_tile_soft_bwd_kernel<all tiles>", st);
      dibr_tile_soft_bwd_kernel<<<persistent, kThreads, 0, st>>>(a);
    } else {
      // forward left the bins, the hit cache and the list of tiles it could not cache
      a.from_list = 1;
      if (s.pool_tiles > 0) {
        const char* force = getenv("DIBR_B200_SOFT_BWD");   // "dense": A/B against the shuffle-reduction kernel
        if (force && force[0] == 'd') {
          Span sp("soft_bwd_dense_kernel", st);
          soft_bwd_dense_kernel<<<(unsigned)s.pool_tiles, kThreads, 0, st>>>(a);
        } else {
          Span sp("soft_bwd_runs_kernel", st);
          soft_bwd_runs_kernel<<<(unsigned)s.pool_tiles, kThreads, 0, st>>>(a);
        }
      }
      Span sp("dibr_tile_soft_bwd_kernel<leftovers>", st);
      dibr_tile_soft_bwd_kernel<<<persistent, kThreads, 0, st>>>(a);
    }
    return (int)cudaGetLastError();
  }
  return 0;
}

int dibr_b200_backward(int batch, int num_faces, int height, int width, int feat_dim,
                       const float* grad_features, const float* grad_soft_mask,
                       const int64_t* face_idx, const float* output_weights, const float* soft_mask,
                       const float* face_vertices_image, const float* face_features,
                       float multiplier, float eps, float sigmainv, float boxlen_m, int knum,
                       float* grad_face_vertices_image, float* grad_face_features, void* workspace,
                       size_t workspace_bytes_, int flags, dibr_b200_stream_t stream) {
  return backward_impl(batch, num_faces, height, width, feat_dim, grad_features, grad_soft_mask, face_idx,
                       output_weights, soft_mask, face_vertices_image, face_features, multiplier, eps,
                       sigmainv, boxlen_m, knum, grad_face_vertices_image, grad_face_features, workspace,
                       workspace_bytes_, flags, stream, false, 0, batch);
}

int dibr_b200_backward_views(int batch, int num_faces, int height, int width, int feat_dim,
                             const void* grad_features, const float* grad_soft_mask,
                             const int64_t* face_idx, const float* output_weights, const float* soft_mask,
                             const float* face_vertices_image, const void* face_features, int features_bf16,
                             float multiplier, float eps, float sigmainv, float boxlen_m, int knum,
                             float* grad_face_vertices_image, float* grad_face_features, void* workspace,
                             size_t workspace_bytes_, int flags, int view_begin, int view_end,
                             dibr_b200_stream_t stream) {
  return backward_impl(batch, num_faces, height, width, feat_dim, grad_features, grad_soft_mask, face_idx,
                       output_weights, soft_mask, face_vertices_image, face_features, multiplier, eps,
                       sigmainv, boxlen_m, knum, grad_face_vertices_image, grad_face_features, workspace,
                       workspace_bytes_, flags, stream, features_bf16 != 0, view_begin, view_end);
}

int dibr_b200_backward_bf16(int batch, int num_faces, int height, int width, int feat_dim,
                            const uint16_t* grad_features, const float* grad_soft_mask,
                            const int64_t* face_idx, const float* output_weights, const float* soft_mask,
                            const float* face_vertices_image, const uint16_t* face_features,
                            float multiplier, float eps, float sigmainv, float boxlen_m, int knum,
                            float* grad_face_vertices_image, float* grad_face_features, void* workspace,
                            size_t workspace_bytes_, int flags, dibr_b200_stream_t stream) {
  return backward_impl(batch, num_faces, height, width, feat_dim, grad_features, grad_soft_mask, face_idx,
                       output_weights, soft_mask, face_vertices_image, face_features, multiplier, eps,
                       sigmainv, boxlen_m, knum, grad_face_vertices_image, grad_face_features, workspace,
                       workspace_bytes_, flags, stream, true, 0, batch);
}

int dibr_b200_packed_rasterize_forward(int batch, int64_t total_faces, int height, int width,
                                       int feat_dim, const float* face_vertices_z,
                                       const float* face_vertices_image, const float* face_bboxes,
                                       const float* face_features,
                                       const int64_t* first_idx_face_per_mesh, float multiplier,
                                       float eps, float* interpolated_features,
                                       int64_t* selected_face_idx, float* output_weights,
                                       void* workspace, size_t workspace_bytes_,
                                       dibr_b200_stream_t stream) {
  int rc = check_dims(batch, total_faces, height, width);
  if (rc) return rc;
  if (!selected_face_idx || !output_weights || !first_idx_face_per_mesh || feat_dim < 0) return DIBR_B200_EINVAL;
  if (feat_dim > 0 && (!interpolated_features || (total_faces > 0 && !face_features))) return DIBR_B200_EINVAL;
  if (total_faces > 0 && (!face_vertices_z || !face_vertices_image || !face_bboxes)) return DIBR_B200_EINVAL;
  if (misaligned(face_vertices_z, face_vertices_image, face_bboxes, face_features, first_idx_face_per_mesh,
                 interpolated_features, selected_face_idx, output_weights))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  FwdArgs a;
  Scene& s = a.s;
  rc = setup_scene(s, batch, total_faces, 0, height, width, multiplier, 0.f, 0, workspace, workspace_bytes_);
  if (rc) return rc;
  s.first = first_idx_face_per_mesh; s.xy = face_vertices_image; s.z = face_vertices_z;
  s.premultiplied = 1; s.fnz = nullptr; s.valid = nullptr; s.bbox_tight = face_bboxes; s.bbox_large = nullptr;
  rc = build_bins(s, 1, st);
  if (rc) return rc;
  a.rc = make_raster_const(eps);
  a.D = feat_dim; a.feat = face_features; a.sigmainv = 0.f; a.K = 0;
  a.out_feat = interpolated_features; a.idx = selected_face_idx; a.out_w = output_weights; a.out_soft = nullptr;
  a.cache = 0;
  a.kl = SoftFwdOut{nullptr, nullptr, nullptr};
  launch_fwd<true, false, false>(a, st);
  return (int)cudaGetLastError();
}

int dibr_b200_rasterize_backward(int batch, int num_faces, int height, int width, int feat_dim,
                                 const float* grad_interpolated_features,
                                 const int64_t* selected_face_idx, const float* output_weights,
                                 const float* face_vertices_image, const float* face_features,
                                 float eps, float* grad_face_vertices_image,
                                 float* grad_face_features, dibr_b200_stream_t stream) {
  if (!grad_interpolated_features && feat_dim > 0) return DIBR_B200_EINVAL;
  // workspace is not needed for the rasterize branch
  return dibr_b200_backward(batch, num_faces, height, width, feat_dim, grad_interpolated_features,
                            nullptr, selected_face_idx, output_weights, nullptr, face_vertices_image,
                            face_features, 1.f, eps, 0.f, 0.f, 0, grad_face_vertices_image,
                            grad_face_features, nullptr, 0, 0, stream);
}

int dibr_b200_soft_mask_forward(int batch, int num_faces, int height, int width, int knum,
                                const float* face_vertices_image, const float* face_large_bboxes,
                                const int64_t* selected_face_idx, float sigmainv, float multiplier,
                                float* soft_mask, float* close_face_prob, int64_t* close_face_idx,
                                uint8_t* close_face_dist_type, void* workspace,
                                size_t workspace_bytes_, dibr_b200_stream_t stream) {
  const int64_t NF = (int64_t)batch * num_faces;
  int rc = check_dims(batch, NF, height, width);
  if (rc) return rc;
  if (!selected_face_idx || !soft_mask || knum <= 0 || num_faces < 0) return DIBR_B200_EINVAL;
  if (num_faces > 0 && (!face_vertices_image || !face_large_bboxes)) return DIBR_B200_EINVAL;
  const bool lists = close_face_prob || close_face_idx || close_face_dist_type;
  if (lists && !(close_face_prob && close_face_idx && close_face_dist_type)) return DIBR_B200_EINVAL;
  if (lists && (int64_t)batch * height * width * knum < 0) return DIBR_B200_ESIZE;
  if (misaligned(face_vertices_image, face_large_bboxes, selected_face_idx, soft_mask, close_face_prob,
                 close_face_idx, close_face_dist_type))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  FwdArgs a;
  Scene& s = a.s;
  rc = setup_scene(s, batch, NF, num_faces, height, width, multiplier, 0.f, 0, workspace, workspace_bytes_);
  if (rc) return rc;
  s.first = nullptr; s.xy = face_vertices_image; s.z = nullptr; s.premultiplied = 1;
  s.fnz = nullptr; s.valid = nullptr; s.bbox_tight = nullptr; s.bbox_large = face_large_bboxes;
  rc = build_bins(s, 2, st);
  if (rc) return rc;
  a.rc = make_raster_const(0.f);
  a.D = 0; a.feat = nullptr; a.sigmainv = sigmainv; a.K = knum;
  a.out_feat = nullptr; a.idx = const_cast<int64_t*>(selected_face_idx); a.out_w = nullptr; a.out_soft = soft_mask;
  a.cache = 0;
  a.kl = SoftFwdOut{close_face_prob, close_face_idx, close_face_dist_type};
  if (lists) launch_fwd<false, true, true>(a, st);
  else launch_fwd<false, true, false>(a, st);
  return (int)cudaGetLastError();
}

int dibr_b200_soft_mask_backward(int batch, int num_faces, int height, int width, int knum,
                                 const float* grad_soft_mask, const float* soft_mask,
                                 const int64_t* selected_face_idx, const float* close_face_prob,
                                 const int64_t* close_face_idx, const uint8_t* close_face_dist_type,
                                 const float* face_vertices_image, float sigmainv, float multiplier,
                                 float* grad_face_vertices_image, dibr_b200_stream_t stream) {
  const int64_t NF = (int64_t)batch * num_faces;
  int rc = check_dims(batch, NF, height, width);
  if (rc) return rc;
  if (!grad_soft_mask || !soft_mask || !selected_face_idx || !close_face_prob || !close_face_idx ||
      !close_face_dist_type || !grad_face_vertices_image || knum <= 0 || !(multiplier > 0.f))
    return DIBR_B200_EINVAL;
  if (num_faces > 0 && !face_vertices_image) return DIBR_B200_EINVAL;
  if (misaligned(grad_soft_mask, soft_mask, selected_face_idx, close_face_prob, close_face_idx,
                 close_face_dist_type, face_vertices_image, grad_face_vertices_image))
    return DIBR_B200_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(grad_face_vertices_image, 0, (size_t)NF * 6 * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  if (NF == 0) return 0;
  SoftBwdListArgs a;
  a.B = batch; a.H = height; a.W = width; a.F = num_faces; a.K = knum;
  a.grid = make_grid(multiplier, width, height);
  a.sigmainv = sigmainv; a.multiplier = multiplier;
  a.grad_soft = grad_soft_mask; a.soft = soft_mask; a.idx = selected_face_idx;
  a.prob = close_face_prob; a.cidx = close_face_idx; a.ctype = close_face_dist_type;
  a.xy = face_vertices_image; a.grad_xy = grad_face_vertices_image;
  const int64_t P = (int64_t)batch * height * width;
  Span sp("soft_bwd_lists_kernel", st);
  soft_bwd_lists_kernel<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(a);
  return (int)cudaGetLastError();
}

}  // extern "C"
