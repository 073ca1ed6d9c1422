// GAT edge phase kernels (ops 3-13 in one pass, genGraphOP.py:52-62; block [4,5,6,7,8] alone) and the er statistics
// of the bound-shifted softmax.  Work list, chain, cursor and launch helpers: aggregate_common.cuh; mapping and
// determinism: the header of aggregate.cu.
#include "aggregate_common.cuh"

namespace gta {

// ----------------------------------------------------------------------------------------
// GAT edge phase, single pass
// ----------------------------------------------------------------------------------------
template <int H>
__device__ __forceinline__ void load_heads(const float* __restrict__ p, float (&v)[H]) {
  if (H % 4 == 0) {
#pragma unroll
    for (int q = 0; q < H / 4; ++q) {
      float4 t = __ldg(reinterpret_cast<const float4*>(p) + q);
      v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
    }
  } else if (H % 2 == 0) {
#pragma unroll
    for (int q = 0; q < H / 2; ++q) {
      float2 t = __ldg(reinterpret_cast<const float2*>(p) + q);
      v[2 * q] = t.x; v[2 * q + 1] = t.y;
    }
  } else {
#pragma unroll
    for (int q = 0; q < H; ++q) v[q] = __ldg(p + q);
  }
}

template <int H>
__device__ __forceinline__ float pick(const float (&v)[H], int h) {
  float r = v[0];
#pragma unroll
  for (int q = 1; q < H; ++q) r = (h == q) ? v[q] : r;
  return r;
}

// ---- softmax shift from a BOUND instead of the running maximum -----------------------------------
// leaky_relu is monotonic, so for every edge of row i whose source lies in column block cb
//     e = leaky(el[i,h] + er[j,h])  <=  leaky(el[i,h] + max_{j in cb} er[j,h])  =: bound(i, cb, h).
// Softmax is invariant under the shift, so p = exp(e - bound) needs no running maximum: no warp
// reductions, no rescale of the accumulator, one exp per edge and head instead of two (round 2 ncu: the 20
// shuffles per 32-edge batch were 0.9 L1/TEX data-pipe wavefronts per edge, the exps 0.6 ms of 5.0).
// A loose bound only costs exponent range, never precision: as long as max er - min er of the block is
// below kBoundRange every p stays above exp(-kBoundRange) relative to the row's largest term.  er_stats
// (gta_er_stats: ordered-int coded max er and max -er per column block and head) says so; blocks that
// fail the test, heads counts that are no power of two and calls that want the true row maximum back
// take the online path below.
constexpr float kBoundRange = 60.f;
// er_stats[cb*pitch + h] = code(max er), er_stats[cb*pitch + heads + h] = code(max -er); 0 = "no source seen".
// pitch = 2*heads for a gta_er_stats buffer, 64 for the statistics of a signal block (exchange.cuh).
__device__ __forceinline__ bool block_bound(const uint32_t* er_stats, int64_t cb0, int64_t cb1, int pitch, int heads,
                                            int h, float* er_max) {
  // an item may span several statistics blocks (an exchange groups its peers' slots): the bound and the
  // range test are taken over their union
  uint32_t cmax = 0u, cneg = 0u;
  bool seen = true;
  for (int64_t cb = cb0; cb <= cb1; ++cb) {
    const uint32_t a = __ldcg(er_stats + cb * pitch + h), b = __ldcg(er_stats + cb * pitch + heads + h);
    seen = seen && a != 0u && b != 0u;
    cmax = a > cmax ? a : cmax;
    cneg = b > cneg ? b : cneg;
  }
  const float hi = ordered_decode(cmax), lo = -ordered_decode(cneg);
  *er_max = hi;
  return seen && (hi - lo) < kBoundRange;      // NaN compares false
}

// ---- the bound, looked up per item -----------------------------------------------------------------
// Round-2 ncu of the GAT kernel on a low-degree shape (items of 20 edges, profiles/r02_gat_lowdeg_*): computing the
// bound cost about 230 of an item's 1 180 warp instructions and 12 % of its stall samples -- two emulated 64-bit
// divisions for the statistics blocks of the first and last source, then, head by head, a loop over those blocks
// whose two L2 loads are consumed inside the loop: H serialised L2 round trips in front of every item's first batch.
// Consecutive items of a warp almost always touch the same statistics blocks, so the warp (each lane group of it)
// keeps the last answer in shared memory, keyed by (first block, last block): the bound stays a pure function of the
// item, hence bitwise the same whoever computes it, and a hit costs two multiply-high divisions and one LDS.
template <int MAXH>
struct __align__(16) BoundCache {
  int32_t cb0, cb1, ok, pad;
  float hi[MAXH];
};
struct BlockDivider {          // source id -> statistics block, without the 64-bit division
  uint32_t d, magic;
  __device__ __forceinline__ explicit BlockDivider(int64_t col_block)
      : d(col_block > 0 ? uint32_t(col_block) : 0u), magic(d > 1u ? uint32_t((uint64_t(1) << 32) / d) : 0u) {}
  __device__ __forceinline__ int operator()(int src) const {
    if (d <= 1u) return d == 0u ? 0 : src;
    uint32_t q = __umulhi(uint32_t(src), magic);          // floor(2^32 / d): never above the quotient, at most 2 below
    uint32_t r = uint32_t(src) - q * d;
    while (r >= d) { ++q; r -= d; }
    return int(q);
  }
};
template <int LANES, int MAXH>
__device__ __forceinline__ void bound_lookup(BoundCache<MAXH>* bc, const uint32_t* er_stats, int cb0, int cb1, int pitch,
                                             int heads, int l, uint32_t gmask) {
  if (bc->cb0 != cb0 || bc->cb1 != cb1) {          // the same answer in every lane of the group
    __syncwarp(gmask);          // everybody has read the old key
    bool ok = true;
    for (int h = l; h < heads; h += LANES) {
      float hi;
      ok = block_bound(er_stats, cb0, cb1, pitch, heads, h, &hi) && ok;
      bc->hi[h] = hi;
    }
    ok = __all_sync(gmask, ok);
    if (l == 0) { bc->cb0 = cb0; bc->cb1 = cb1; bc->ok = ok ? 1 : 0; }
    __syncwarp(gmask);
  }
}

template <typename P, int LANES, int H>
__global__ void __launch_bounds__(kAggThreads, (H <= 4) ? GTA_GAT_MINBLOCKS : (GTA_GAT_MINBLOCKS + 1) / 2)
gat_aggregate_kernel(const WorkList wl, const Exchange ex, const float* __restrict__ el, const float* __restrict__ er,
                     int64_t lder, float slope, const typename P::T* __restrict__ z, const uint32_t row_bytes,
                     float* __restrict__ out, int64_t ldo, int f, int epilogue, float* __restrict__ rowmax,
                     float* __restrict__ rowsum, const uint32_t* er_stats, int stats_pitch, int64_t col_block) {
  // per warp: H rows of 32 staged edges, entry = {source id, softmax numerator}.  Row pitch kS = 34
  // entries: a lane's STS.64 lands beside its neighbour's (2 wavefronts per head, no conflicts) and the
  // LDS.128 of the gather loop -- two consecutive edges of one head, the 4 heads of a warp at once --
  // hits 4 disjoint bank quads (68 words = 4 mod 32).  Round 1 staged [edge][head]: 4-way conflicts on
  // every store, 27 % of the L1/TEX data-pipe wavefronts of the kernel.
  constexpr int kS = 34;
  using Raw = typename P::Raw;
  constexpr int KP = P::kPer;
  constexpr int kWindow = LANES * KP;
  __shared__ __align__(16) uint2 s_e[kAggWarps][H * kS];
  __shared__ BoundCache<H> s_bound[kAggWarps][32 / LANES];
  __shared__ __align__(16) NextItem s_next[kAggWarps][32 / LANES];
  if (ex.world > 1 && blockIdx.y == 0 && blockIdx.x < ex.copy_ctas) {
    exchange_pull(ex, blockIdx.x);          // these CTAs move the peers' slots; everybody else reduces
    return;
  }
  const int lane = threadIdx.x & 31;
  const int l = lane & (LANES - 1);
  const int gbase = lane & ~(LANES - 1);          // first lane of my group inside the warp
  BoundCache<H>* bc = &s_bound[threadIdx.x >> 5][lane / LANES];
  if (l == 0) { bc->cb0 = -1; bc->cb1 = -1; bc->ok = 0; }
  __syncwarp();
  const BlockDivider block_of(col_block);
  const int fo = blockIdx.y * kWindow + KP * l;
  const int head = (fo < f) ? fo / (f / H) : 0;
  uint2* se = s_e[threadIdx.x >> 5];
  const uint2* mine = se + head * kS + gbase;
  const uint4* mine2 = reinterpret_cast<const uint4*>(mine);
  int32_t* counter = wl.work_counter + blockIdx.y;
  int32_t* flags = wl.chain_flags + int64_t(blockIdx.y) * wl.num_slots;
  const uint64_t pol_stream = wl.pol_stream, pol_keep = wl.pol_keep;
  const int pstride = gat_partial_stride(f, H);
  const int stats = f + int(blockIdx.y) * gat_stats_stride(H);
  const char* zf = reinterpret_cast<const char*>(z + (fo < f ? fo : 0));

  const ItemCursor first = cursor_begin<LANES>(wl, ex, counter, lane);
  int32_t landed = 0;          // exchange_gate: highest peer slot this lane has seen complete
  // what an item needs before its first batch: the record, the row's el, the ids of its first two batches and its
  // last id (sources ascend: the last id names the highest slot / statistics block the item touches)
  float elr[H];
  int idx_cur = 0, idx_nxt = 0, last_src = 0;
  const bool want_last = ex.world > 1 || er_stats != nullptr;
  auto request_inputs = [&](const int4& t, bool hv) {
    const int cnt = hv ? t.z : 0;
    const int32_t* ib = wl.indices + t.y;
#pragma unroll
    for (int h = 0; h < H; ++h) elr[h] = 0.f;
    if (hv) load_heads<H>(el + int64_t(t.x) * H, elr);
    idx_cur = 0;
    idx_nxt = 0;
    if (l < cnt) idx_cur = ld_stream_i32(ib + l, pol_stream);
    if (LANES + l < cnt) idx_nxt = ld_stream_i32(ib + LANES + l, pol_stream);
    last_src = (cnt > 0 && want_last) ? __ldg(ib + cnt - 1) : 0;
  };
  ItemStage<LANES> stage(wl, first, lane, &s_next[threadIdx.x >> 5][lane / LANES]);
  request_inputs(stage.it, stage.have);
  while (stage.cur.first < wl.num_items) {
    // claim the next item now and let its record (and this row's slot range) travel into shared memory under the gathers
    stage.claim(wl, counter, lane);
    const int4 it = stage.it;
    const bool have = stage.have;
    const bool active = have && fo < f;
    const int count = have ? it.z : 0;
    const int max_count = (LANES == 32) ? count : warp_max_i32(count);
    const int32_t* idx_base = wl.indices + it.y;

    float m[H], s[H];      // s: this lane's share of the running sum (reduced at the end)
#pragma unroll
    for (int h = 0; h < H; ++h) { m[h] = -INFINITY; s[h] = 0.f; }
    float acc[KP];
#pragma unroll
    for (int c = 0; c < KP; ++c) acc[c] = 0.f;

    // software pipeline: source ids are loaded two batches ahead and the er rows one batch ahead, so
    // the id -> er -> softmax dependency chain of batch b+1 hides under the row gathers of batch b
    float er_cur[H];
#pragma unroll
    for (int h = 0; h < H; ++h) er_cur[h] = 0.f;
    if (ex.world > 1) {          // the item's slots (z, er and their er range) may still be on their way from the peers
      if (l == 0 && count > 0) exchange_gate(ex, last_src, landed);
      __syncwarp();
    }
    if (l < count) load_heads<H>(er + int64_t(idx_cur) * lder, er_cur);

    // bound path: the whole warp or nobody (the online path reduces with full-warp shuffles)
    bool bounded = false;
    if (er_stats != nullptr) {
      bool ok = true;
      const int first_src = __shfl_sync(0xffffffffu, idx_cur, gbase);
      if (count > 0) {
        bound_lookup<LANES, H>(bc, er_stats, block_of(first_src), block_of(last_src), stats_pitch, H, l, group_mask<LANES>(lane));
        ok = bc->ok != 0;
#pragma unroll
        for (int h = 0; h < H; ++h) m[h] = leaky(elr[h] + bc->hi[h], slope);
      }
      bounded = __all_sync(0xffffffffu, ok);
      if (!bounded) {
#pragma unroll
        for (int h = 0; h < H; ++h) m[h] = -INFINITY;
      }
    }

    for (int base = 0; base < max_count; base += LANES) {
      int n = count - base;
      n = n < 0 ? 0 : (n > LANES ? LANES : n);
      float e[H];
      const int my_idx = idx_cur;
#pragma unroll
      for (int h = 0; h < H; ++h) e[h] = (l < n) ? leaky(elr[h] + er_cur[h], slope) : -INFINITY;
      // prefetch: er of the next batch (its ids arrived during the previous iteration), ids of the one after
      idx_cur = idx_nxt;
      if (base + LANES + l < count) load_heads<H>(er + int64_t(idx_cur) * lder, er_cur);
      if (base + 2 * LANES + l < count) idx_nxt = ld_stream_i32(idx_base + base + 2 * LANES + l, pol_stream);
      if (bounded) {
#pragma unroll
        for (int h = 0; h < H; ++h) {
          const float p = (l < n) ? softmax_exp(e[h] - m[h]) : 0.f;
          s[h] += p;
          se[h * kS + lane] = make_uint2(uint32_t(my_idx), __float_as_uint(p));
        }
      } else {
        float my_scale = 1.f;
#pragma unroll
        for (int h = 0; h < H; ++h) {
          const float mn = fmaxf(m[h], group_max<LANES>(e[h]));
          // mn stays -inf only while this group has seen no edge (another group in the warp is running)
          const float sc = (mn == -INFINITY) ? 1.f : softmax_exp(m[h] - mn);
          const float p = (l < n) ? softmax_exp(e[h] - mn) : 0.f;
          s[h] = fmaf(s[h], sc, p);
          m[h] = mn;
          my_scale = (h == head) ? sc : my_scale;
          se[h * kS + lane] = make_uint2(uint32_t(my_idx), __float_as_uint(p));
        }
#pragma unroll
        for (int c = 0; c < KP; ++c) acc[c] *= my_scale;
      }
      __syncwarp();
      const bool full = (LANES == 32) ? (n == LANES) : __all_sync(0xffffffffu, n == LANES && active);
      if (full) {
        if (LANES < 32 || active) {
#pragma unroll 1
          for (int j = 0; j < LANES; j += kGatUnroll) {
            uint4 ed[kGatUnroll / 2];
            Raw raw[kGatUnroll];
#pragma unroll
            for (int u = 0; u < kGatUnroll / 2; ++u)
              if (j + 2 * u < LANES) ed[u] = mine2[(j >> 1) + u];
#pragma unroll
            for (int u = 0; u < kGatUnroll / 2; ++u) {
              if (j + 2 * u < LANES) {
                raw[2 * u] = P::load(row_addr(zf, ed[u].x, row_bytes), pol_keep);
                raw[2 * u + 1] = P::load(row_addr(zf, ed[u].z, row_bytes), pol_keep);
              }
            }
#pragma unroll
            for (int u = 0; u < kGatUnroll / 2; ++u) {
              if (j + 2 * u < LANES) {
                fma_row<P>(acc, __uint_as_float(ed[u].y), raw[2 * u]);
                fma_row<P>(acc, __uint_as_float(ed[u].w), raw[2 * u + 1]);
              }
            }
          }
        }
      } else {
        const int nmax = (LANES == 32) ? n : LANES;
        for (int j = 0; j < nmax; j += kGatUnroll) {
          Raw raw[kGatUnroll];
          float pv[kGatUnroll];
#pragma unroll
          for (int u = 0; u < kGatUnroll; ++u) {
            if (j + u < LANES) {
              const uint2 ed = mine[j + u];
              pv[u] = __uint_as_float(ed.y);
              raw[u] = P::zero();
              if (active && (j + u) < n) raw[u] = P::load(row_addr(zf, ed.x, row_bytes), pol_keep);
            }
          }
#pragma unroll
          for (int u = 0; u < kGatUnroll; ++u)
            if (j + u < LANES) fma_row<P>(acc, pv[u], raw[u]);
        }
      }
      __syncwarp();
    }
#pragma unroll
    for (int h = 0; h < H; ++h) s[h] = group_sum<LANES>(s[h]);
    const bool chained = have && it.w >= 0;
    // the gather loop is over: elr / idx_* are free, the staged record has long arrived.  Request the next item's
    // inputs now; they travel while this item's chain fold waits for its predecessor and writes its state.
    const int4 next = stage.land(chained);
    request_inputs(next, stage.next_have);
    chain_step<LANES>(flags, lane, it, chained, [&]() { return stage.slots; },
        [&](int prev_slot) {
          // fold the state of slots [s0, it.w) in: (max, sum, acc) triples merge like the online softmax itself
          const float* prev = wl.partials + int64_t(prev_slot) * pstride;
          float a_mine = 1.f, b_mine = 1.f;
#pragma unroll
          for (int h = 0; h < H; ++h) {
            const float pm = ld_state_f32(prev + stats + h), ps = ld_state_f32(prev + stats + H + h);
            const float mn = fmaxf(pm, m[h]);
            // one of the two factors is exp(0) = 1: a single exp per head (bit-identical to computing both)
            const float t = (mn == -INFINITY) ? 0.f : expf(fminf(pm, m[h]) - mn);
            const float a = (pm == -INFINITY) ? 0.f : (pm == mn ? 1.f : t);
            const float b = (m[h] == -INFINITY) ? 0.f : (m[h] == mn ? 1.f : t);
            s[h] = fmaf(ps, a, s[h] * b);
            m[h] = mn;
            a_mine = (h == head) ? a : a_mine;
            b_mine = (h == head) ? b : b_mine;
          }
          if (active) {
            float p[KP];
            ld_state<KP>(prev + fo, p);
#pragma unroll
            for (int c = 0; c < KP; ++c) acc[c] = fmaf(p[c], a_mine, acc[c] * b_mine);
          }
        },
        [&](int slot) {
          float* part = wl.partials + int64_t(slot) * pstride;
          if (active) st_state<KP>(part + fo, acc);
          if (l < H) {
            part[stats + l] = pick<H>(m, l);
            part[stats + H + l] = pick<H>(s, l);
          }
        },
        [&]() {
          if (!have) return;
          if (active) {
            const float sh = pick<H>(s, head);
            st_out<KP>(out + int64_t(it.x) * ldo + fo, acc, sh > 0.f ? 1.f / sh : 0.f, epilogue);
          }
          if (blockIdx.y == 0 && l < H) {
            const float ml = pick<H>(m, l);
            if (rowmax) rowmax[int64_t(it.x) * H + l] = (count > 0 || it.w >= 0) && ml != -INFINITY ? ml : 0.f;
            if (rowsum) rowsum[int64_t(it.x) * H + l] = pick<H>(s, l);
          }
        });
    stage.advance(next);
  }
}

// ----------------------------------------------------------------------------------------
// GAT edge phase, lane-local-head variant (any H whose per-head width F/H is a multiple of 4, or 2, or 1;
// used for H >= 8 and for the narrow heads of the reference's third GAT layer, F = H = 16)
//
// The staged kernel above keeps el/max/sum/er for ALL heads in every lane (5H registers: H = 16
// spills and runs at a quarter of the H = 4 speed).  Here a lane tracks only the heads its own 4
// features belong to -- HPL = 1 head when the per-head width is a multiple of 4, 2 heads of width 2, 4 heads
// of width 1: one er gather of HPL floats per edge (the lanes of a row read the H consecutive floats of
// er[j]: one wavefront), softmax over groups of a few edges, no arrays over all heads, no shuffles.  Lanes
// of one head see the same edges in the same order, so their (max, sum) are bit-identical.
// ----------------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void ldg_vec(const float* p, float (&v)[N]) {
  if constexpr (N == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else if constexpr (N == 2) {
    const float2 t = __ldg(reinterpret_cast<const float2*>(p));
    v[0] = t.x; v[1] = t.y;
  } else {
    v[0] = __ldg(p);
  }
}
// which of a lane's HPL heads its feature c (0..3) belongs to
template <int HPL>
__device__ __forceinline__ constexpr int head_of(int c) { return HPL == 1 ? 0 : (HPL == 2 ? c / 2 : c); }

template <int LANES, int HPL>
__global__ void __launch_bounds__(kAggThreads, GTA_LLH_MINBLOCKS)
gat_aggregate_llh_kernel(const WorkList wl, const Exchange ex, const float* __restrict__ el,
                         const float* __restrict__ er, int64_t lder, int heads, float slope,
                         const float* __restrict__ z, const uint32_t row_bytes, float* __restrict__ out, int64_t ldo,
                         int f, int epilogue, float* __restrict__ rowmax, float* __restrict__ rowsum,
                         const uint32_t* er_stats, int stats_pitch, int64_t col_block) {
  constexpr int kU = kLlhUnroll / HPL > 2 ? kLlhUnroll / HPL : 2;      // edges per softmax group: e / p are HPL wide
  __shared__ uint32_t s_id[kAggWarps][32];
  __shared__ BoundCache<32> s_bound[kAggWarps][32 / LANES];          // er_stats are only passed for heads <= 32
  if (ex.world > 1 && blockIdx.y == 0 && blockIdx.x < ex.copy_ctas) {
    exchange_pull(ex, blockIdx.x);          // these CTAs move the peers' slots; everybody else reduces
    return;
  }
  const int lane = threadIdx.x & 31;
  const int l = lane & (LANES - 1);
  BoundCache<32>* bc = &s_bound[threadIdx.x >> 5][lane / LANES];
  if (l == 0) { bc->cb0 = -1; bc->cb1 = -1; bc->ok = 0; }
  __syncwarp();
  const BlockDivider block_of(col_block);
  const int fo = blockIdx.y * 128 + 4 * l;
  const int d = f / heads;          // HPL == 1: a multiple of 4;  HPL == 2: 2;  HPL == 4: 1
  const int head = (fo < f) ? fo / d : 0;          // the lane's first head (a multiple of HPL)
  const char* erh = reinterpret_cast<const char*>(er + head);
  const uint32_t er_bytes = uint32_t(lder) * 4u;
  uint32_t* sid = s_id[threadIdx.x >> 5];
  const uint32_t* mine = sid + (lane & ~(LANES - 1));
  int32_t* counter = wl.work_counter + blockIdx.y;
  int32_t* flags = wl.chain_flags + int64_t(blockIdx.y) * wl.num_slots;
  const uint64_t pol_stream = wl.pol_stream, pol_keep = wl.pol_keep;
  const int pstride = gat_partial_stride(f, heads);
  const int stats = f + int(blockIdx.y) * gat_stats_stride(heads);

  ItemCursor cur = cursor_begin<LANES>(wl, ex, counter, lane);
  int32_t landed = 0;          // exchange_gate: highest peer slot this lane has seen complete
  while (cur.first < wl.num_items) {
    const int64_t group = int64_t(cur.first) + lane / LANES;
    const bool have = group < wl.num_items;
    const bool active = have && fo < f;
    const int4 it = have ? __ldg(wl.items + group) : make_int4(0, 0, 0, -1);
    const int count = have ? it.z : 0;
    const int max_count = (LANES == 32) ? count : warp_max_i32(count);
    const int32_t* idx_base = wl.indices + it.y;
    const char* zf = reinterpret_cast<const char*>(z + (active ? fo : 0));
    float elh[HPL], m[HPL], s[HPL];
#pragma unroll
    for (int k = 0; k < HPL; ++k) { elh[k] = 0.f; m[k] = -INFINITY; s[k] = 0.f; }
    if (active) ldg_vec<HPL>(el + int64_t(it.x) * heads + head, elh);

    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int idx_nxt = 0;
    if (l < count) idx_nxt = ld_stream_i32(idx_base + l, pol_stream);
    const int last_src = (count > 0 && (ex.world > 1 || er_stats != nullptr)) ? __ldg(idx_base + count - 1) : 0;
    if (ex.world > 1) {
      if (l == 0 && count > 0) exchange_gate(ex, last_src, landed);
      __syncwarp();
    }
    // bound path (see gat_aggregate_kernel): a lane only needs the bound of its own heads; the choice is
    // per lane group here, nothing below synchronises across groups on it
    bool bounded = false;
    int first_src = 0;
    if (er_stats != nullptr) first_src = __shfl_sync(0xffffffffu, idx_nxt, lane & ~(LANES - 1));
    if (er_stats != nullptr && count > 0) {          // every head of the block must pass: lanes of one item agree
      bound_lookup<LANES, 32>(bc, er_stats, block_of(first_src), block_of(last_src), stats_pitch, heads, l, group_mask<LANES>(lane));
      bounded = bc->ok != 0;
#pragma unroll
      for (int k = 0; k < HPL; ++k) m[k] = bounded ? leaky(elh[k] + bc->hi[head + k], slope) : -INFINITY;
    }
    for (int base = 0; base < max_count; base += LANES) {
      int n = count - base;
      n = n < 0 ? 0 : (n > LANES ? LANES : n);
      sid[lane] = uint32_t(idx_nxt);
      if (base + LANES + l < count) idx_nxt = ld_stream_i32(idx_base + base + LANES + l, pol_stream);
      __syncwarp();
      const int nmax = (LANES == 32) ? n : LANES;
#pragma unroll 1
      for (int j = 0; j < nmax; j += kU) {
        float e[kU][HPL];
        float4 v[kU];
        uint32_t id[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) id[u] = (j + u < LANES) ? mine[(j + u) & (LANES - 1)] : 0u;
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          const bool ok = (j + u) < n;
          float erv[HPL];
#pragma unroll
          for (int k = 0; k < HPL; ++k) erv[k] = 0.f;
          if (ok) ldg_vec<HPL>(reinterpret_cast<const float*>(row_addr(erh, id[u], er_bytes)), erv);
#pragma unroll
          for (int k = 0; k < HPL; ++k) e[u][k] = ok ? leaky(elh[k] + erv[k], slope) : -INFINITY;
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (active && (j + u) < n) v[u] = F32x4::unpack(F32x4::load(row_addr(zf, id[u], row_bytes), pol_keep));
        }
        if (!bounded) {
          // online softmax: new running maximum per head, rescale what has been accumulated.  A head that has
          // seen no edge yet (mn = -inf) keeps its zeros.
          float sc[HPL];
#pragma unroll
          for (int k = 0; k < HPL; ++k) {
            float bm = e[0][k];
#pragma unroll
            for (int u = 1; u < kU; ++u) bm = fmaxf(bm, e[u][k]);
            const float mn = fmaxf(m[k], bm);
            sc[k] = (mn == -INFINITY) ? 1.f : expf(m[k] - mn);          // m = -inf on the first group: sc = 0, acc and s are 0 anyway
            s[k] *= sc[k];
            m[k] = mn;
          }
          acc.x *= sc[head_of<HPL>(0)]; acc.y *= sc[head_of<HPL>(1)];
          acc.z *= sc[head_of<HPL>(2)]; acc.w *= sc[head_of<HPL>(3)];
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          // e = -inf for the padding of the last group: p = 0
          float p[HPL];
#pragma unroll
          for (int k = 0; k < HPL; ++k) {
            p[k] = (m[k] == -INFINITY) ? 0.f : softmax_exp(e[u][k] - m[k]);
            s[k] += p[k];
          }
          acc.x = fmaf(p[head_of<HPL>(0)], v[u].x, acc.x); acc.y = fmaf(p[head_of<HPL>(1)], v[u].y, acc.y);
          acc.z = fmaf(p[head_of<HPL>(2)], v[u].z, acc.z); acc.w = fmaf(p[head_of<HPL>(3)], v[u].w, acc.w);
        }
      }
      __syncwarp();
    }
    // who publishes a head's statistics: the first lane of the head (width >= 4), or the one lane that owns it.
    // A chained item's successor folds max and sum from the statistics of ITS window, so there the first lane of the
    // window saves them too: a head whose width does not divide 128 (f = 144, H = 12) starts in the window before.
    const bool head_leader = active && (HPL > 1 || (fo % d) == 0);
    const bool window_leader = head_leader || (active && l == 0);
    const bool chained = have && it.w >= 0;
    chain_step<LANES>(flags, lane, it, chained,
        [&]() { return make_int2(__ldg(wl.row_slots + it.x), __ldg(wl.row_slots + it.x + 1)); },
        [&](int prev_slot) {
          if (active) {
            const float* prev = wl.partials + int64_t(prev_slot) * pstride;
            float a[HPL], b[HPL];
#pragma unroll
            for (int k = 0; k < HPL; ++k) {
              const float pm = ld_state_f32(prev + stats + head + k), ps = ld_state_f32(prev + stats + heads + head + k);
              const float mn = fmaxf(pm, m[k]);
              const float t = (mn == -INFINITY) ? 0.f : expf(fminf(pm, m[k]) - mn);      // the other factor is exp(0) = 1
              a[k] = (pm == -INFINITY) ? 0.f : (pm == mn ? 1.f : t);
              b[k] = (m[k] == -INFINITY) ? 0.f : (m[k] == mn ? 1.f : t);
              s[k] = fmaf(ps, a[k], s[k] * b[k]);
              m[k] = mn;
            }
            const float4 p = ld_state_f32x4(prev + fo);
            acc.x = fmaf(p.x, a[head_of<HPL>(0)], acc.x * b[head_of<HPL>(0)]);
            acc.y = fmaf(p.y, a[head_of<HPL>(1)], acc.y * b[head_of<HPL>(1)]);
            acc.z = fmaf(p.z, a[head_of<HPL>(2)], acc.z * b[head_of<HPL>(2)]);
            acc.w = fmaf(p.w, a[head_of<HPL>(3)], acc.w * b[head_of<HPL>(3)]);
          }
        },
        [&](int slot) {
          float* part = wl.partials + int64_t(slot) * pstride;
          if (active) *reinterpret_cast<float4*>(part + fo) = acc;
          if (window_leader) {
#pragma unroll
            for (int k = 0; k < HPL; ++k) {
              part[stats + head + k] = m[k];
              part[stats + heads + head + k] = s[k];
            }
          }
        },
        [&]() {
          if (!active) return;
          float inv[HPL];
#pragma unroll
          for (int k = 0; k < HPL; ++k) inv[k] = s[k] > 0.f ? 1.f / s[k] : 0.f;
          st_stream_f32x4(out + int64_t(it.x) * ldo + fo,
                          make_float4(apply_epilogue(acc.x * inv[head_of<HPL>(0)], epilogue), apply_epilogue(acc.y * inv[head_of<HPL>(1)], epilogue),
                                      apply_epilogue(acc.z * inv[head_of<HPL>(2)], epilogue), apply_epilogue(acc.w * inv[head_of<HPL>(3)], epilogue)));
          if (head_leader) {
#pragma unroll
            for (int k = 0; k < HPL; ++k) {
              if (rowmax) rowmax[int64_t(it.x) * heads + head + k] = (count > 0 || it.w >= 0) && m[k] != -INFINITY ? m[k] : 0.f;
              if (rowsum) rowsum[int64_t(it.x) * heads + head + k] = s[k];
            }
          }
        });
    cursor_next<LANES>(cur, wl, counter, lane);
  }
}

// ----------------------------------------------------------------------------------------
// er_stats: per column block and head, max er and max -er as ordered-int codes (atomicMax on zeroed words)
// ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
er_stats_kernel(const float* __restrict__ er, int64_t lder, int64_t num_sources, int64_t col_block, int heads,
                uint32_t* __restrict__ stats) {
  // lane -> head (heads is a power of two <= 32), 32/heads rows per warp step
  const int lane = threadIdx.x & 31;
  const int h = lane & (heads - 1);
  const int rows_per_step = 32 / heads;
  const int64_t cb = blockIdx.y;
  const int64_t lo = col_block > 0 ? cb * col_block : 0;
  const int64_t hi = col_block > 0 ? (lo + col_block < num_sources ? lo + col_block : num_sources) : num_sources;
  const int64_t warp = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  const int64_t warps = (int64_t(gridDim.x) * blockDim.x) >> 5;
  float mx = -INFINITY, mn = INFINITY;
  bool seen = false;
  for (int64_t r = lo + warp * rows_per_step + lane / heads; r < hi; r += warps * rows_per_step) {
    const float v = __ldg(er + r * lder + h);
    mx = fmaxf(mx, v);
    mn = fminf(mn, v);
    seen = true;
  }
  // lanes with the same head: xor offsets heads, 2*heads, ...
  for (int o = heads; o < 32; o <<= 1) {
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    seen = __shfl_xor_sync(0xffffffffu, int(seen), o) || seen;
  }
  if (lane < heads && seen) {
    atomicMax(stats + (cb * 2) * heads + h, ordered_code(mx));
    atomicMax(stats + (cb * 2 + 1) * heads + h, ordered_code(-mn));
  }
}

// ----------------------------------------------------------------------------------------
// GAT block [4,5,6,7,8]: numerators p[E,H] (STORE_E) and row sums S[N,H]; warp per row
// ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gat_logits_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices, int64_t row_begin,
                  int64_t row_end, const float* __restrict__ el, const float* __restrict__ er, int heads,
                  float slope, int stabilize, float* __restrict__ p, float* __restrict__ rowmax,
                  float* __restrict__ rowsum) {
  const int lane = threadIdx.x & 31;
  const int64_t r = row_begin + ((blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5);
  if (r >= row_end) return;
  const int64_t b = indptr[r], e = indptr[r + 1];
  const int64_t lr = r - row_begin;
  for (int h = 0; h < heads; ++h) {
    const float elv = el[lr * heads + h];
    float mx = -INFINITY;
    if (stabilize) {
      for (int64_t k = b + lane; k < e; k += 32)
        mx = fmaxf(mx, leaky(elv + er[int64_t(indices[k]) * heads + h], slope));
      mx = group_max<32>(mx);
    }
    if (!stabilize || mx == -INFINITY) mx = 0.f;
    // deterministic sum: fixed lane-strided partial sums, then a fixed butterfly
    float sum = 0.f;
    for (int64_t k = b + lane; k < e; k += 32) {
      float v = expf(leaky(elv + er[int64_t(indices[k]) * heads + h], slope) - mx);
      p[k * heads + h] = v;
      sum += v;
    }
    sum = group_sum<32>(sum);
    if (lane == 0) {
      if (rowmax) rowmax[lr * heads + h] = mx;
      rowsum[lr * heads + h] = sum;
    }
  }
}

template <typename P, int H>
static int dispatch_gat(int lanes, cudaStream_t st, const WorkList& wl, const Exchange& ex, const float* el,
                        const float* er, int64_t lder, float slope, const typename P::T* z, int64_t ldz, float* out, int64_t ldo,
                        int f, int epi, float* rowmax, float* rowsum, const uint32_t* er_stats, int stats_pitch,
                        int64_t col_block) {
  auto launch = [&](auto kernel, int lanes_c) {
    launch_persistent(kernel, wl, ex, lanes_c, (f + lanes_c * P::kPer - 1) / (lanes_c * P::kPer), st, el, er, lder, slope, z,
                      uint32_t(ldz * sizeof(typename P::T)), out, ldo, f, epi, rowmax, rowsum, er_stats, stats_pitch,
                      col_block);
  };
  if constexpr (P::kPer == 8) {          // Bf16x8 only takes rows wider than 128 features: always 32 lanes
    if (lanes == 32) { launch(gat_aggregate_kernel<P, 32, H>, 32); return GTA_OK; }
  } else {
    switch (lanes) {
      case 4: if (H <= 4) { launch(gat_aggregate_kernel<P, 4, H>, 4); return GTA_OK; } break;
      case 8: if (H <= 8) { launch(gat_aggregate_kernel<P, 8, H>, 8); return GTA_OK; } break;
      case 16: launch(gat_aggregate_kernel<P, 16, H>, 16); return GTA_OK;
      case 32: launch(gat_aggregate_kernel<P, 32, H>, 32); return GTA_OK;
    }
  }
  return GTA_ERR_UNSUPPORTED;
}

template <typename P>
static int gat_run(const char* who, int heads, cudaStream_t st, const WorkList& wl, const Exchange& ex, const float* el,
                   const float* er, int64_t lder, float slope, const typename P::T* z, int64_t ldz, float* out, int64_t ldo,
                   int f, int epilogue, float* rowmax, float* rowsum, const uint32_t* er_stats, int stats_pitch,
                   int64_t col_block) {
  constexpr int KP = P::kPer;
  if (f % KP != 0 || (f / heads) % KP != 0) {
    set_error("%s: per-head width f/heads=%d is not a multiple of %d", who, f / heads, KP);
    return GTA_ERR_UNSUPPORTED;
  }
  const int lanes = lanes_for(f, KP);
  int rc = GTA_ERR_UNSUPPORTED;
#define GTA_GAT_H(HH) rc = dispatch_gat<P, HH>(lanes, st, wl, ex, el, er, lder, slope, z, ldz, out, ldo, f, epilogue, rowmax, rowsum, er_stats, stats_pitch, col_block)
  switch (heads) {
    case 1: GTA_GAT_H(1); break;
    case 2: GTA_GAT_H(2); break;
    default: GTA_GAT_H(4); break;
  }
#undef GTA_GAT_H
  if (rc != GTA_OK) set_error("%s: no kernel for heads=%d, f=%d", who, heads, f);
  return rc;
}

template <typename T>
static int gat_aggregate_impl(const char* who, const int32_t* items_, int64_t num_items, const int32_t* row_slots,
                              int64_t num_slots, const int32_t* indices, const float* el, const float* er, int64_t lder,
                              int32_t heads, float slope, const T* z, int64_t ldz, float* out, int64_t ldo, int32_t f,
                              int32_t epilogue, float* rowmax, float* rowsum, float* partials, int32_t* chain_state,
                              const uint32_t* er_stats, int64_t col_block, const gta_exchange_t* exchange,
                              int32_t phases, void* stream_) {
  constexpr int kRow = 16 / int(sizeof(T));
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  GTA_REQUIRE(f > 0 && f % 4 == 0, "%s: f=%d must be a positive multiple of 4", who, f);
  WorkList wl;
  bool launch = false;
  int rc = prepare_worklist(who, items_, num_items, row_slots, num_slots, indices, partials, chain_state, f, phases, st,
                            &wl, &launch);
  if (rc != GTA_OK || !launch) return rc;
  GTA_REQUIRE(items_ && indices && el && er && z && out, "%s: null pointer", who);
  GTA_REQUIRE(ldz % kRow == 0 && ldo % 4 == 0 && ldz >= f && ldo >= f && ldz * int64_t(sizeof(T)) < (int64_t(1) << 32),
              "%s: leading dimensions must be whole 16-byte pieces, >= f, and a row below 4 GiB", who);
  GTA_REQUIRE((reinterpret_cast<uintptr_t>(z) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
              (reinterpret_cast<uintptr_t>(er) & 15) == 0 && (reinterpret_cast<uintptr_t>(el) & 15) == 0,
              "%s: tables must be 16-byte aligned", who);
  GTA_REQUIRE(heads >= 1 && f % heads == 0, "%s: heads=%d must divide f=%d", who, heads, f);
  GTA_REQUIRE(lder >= heads && (heads % 4 != 0 || lder % 4 == 0) && (heads % 2 != 0 || lder % 2 == 0),
              "%s: er row stride %lld breaks the vector alignment of %d heads", who, (long long)lder, heads);
  Exchange ex;
  rc = make_exchange(who, exchange, wl.work_counter + (f + 127) / 128, ldz * int64_t(sizeof(T)), &ex);
  if (rc != GTA_OK) return rc;
  int stats_pitch = 2 * heads;
  if (ex.world > 1) {
    GTA_REQUIRE(ex.table == reinterpret_cast<const char*>(z), "%s: z is not the exchange table", who);
    // the slot owners published their er range with the step; a slot's statistics are valid once it has landed
    er_stats = &ex.signals->stats[ex.step & 1][0][0];
    stats_pitch = 64;
    col_block = ex.slot_rows;
    if ((heads & (heads - 1)) != 0 || heads > 32) er_stats = nullptr;
  }
  // the bound path does not track the true row maximum: callers that want it back run the online softmax
  if (rowmax != nullptr) er_stats = nullptr;
  // H <= 4 with whole pieces per head: staged kernel (all heads per lane, softmax once per 32-edge batch);  H >= 8, an
  // unusual H or heads narrower than a piece: lane-local-head kernel (per-head width a multiple of 4, or 2, or 1;
  // constant register footprint; fp32 tables only)
  bool staged = heads == 1 || heads == 2 || heads == 4;
  if constexpr (sizeof(T) == 4) staged = staged && (f / heads) % 4 == 0;
  if (staged) {
    if constexpr (sizeof(T) == 4) {
      rc = gat_run<F32x4>(who, heads, st, wl, ex, el, er, lder, slope, z, ldz, out, ldo, f, epilogue, rowmax, rowsum,
                          er_stats, stats_pitch, col_block);
    } else if (f <= 128 || f % 8 != 0 || (f / heads) % 8 != 0) {
      // 8-byte pieces of 4 features: every per-head width of whole pieces of 4, in windows of 128 above 128 features
      rc = gat_run<Bf16x4>(who, heads, st, wl, ex, el, er, lder, slope, z, ldz, out, ldo, f, epilogue, rowmax, rowsum,
                           er_stats, stats_pitch, col_block);
    } else {
      rc = gat_run<Bf16x8>(who, heads, st, wl, ex, el, er, lder, slope, z, ldz, out, ldo, f, epilogue, rowmax, rowsum,
                           er_stats, stats_pitch, col_block);
    }
    if (rc != GTA_OK) return rc;
  } else if constexpr (sizeof(T) == 4) {
    const int width = f / heads;
    const int hpl = width % 4 == 0 ? 1 : (width == 2 ? 2 : (width == 1 ? 4 : 0));      // heads per 4-feature lane
    if (hpl == 0) {
      set_error("%s: per-head width f/heads=%d is neither a multiple of 4 nor 2 nor 1", who, width);
      return GTA_ERR_UNSUPPORTED;
    }
    const int lanes = lanes_for(f, 4);
    auto launch_llh = [&](auto kernel) {
      launch_persistent(kernel, wl, ex, lanes, (f + 127) / 128, st, el, er, lder, heads, slope, z, uint32_t(ldz) * 4u, out,
                        ldo, f, epilogue, rowmax, rowsum, er_stats, stats_pitch, col_block);
    };
    auto for_heads_per_lane = [&](auto lanes_c) {
      constexpr int L = decltype(lanes_c)::value;
      if (hpl == 1) launch_llh(gat_aggregate_llh_kernel<L, 1>);
      else if (hpl == 2) launch_llh(gat_aggregate_llh_kernel<L, 2>);
      else launch_llh(gat_aggregate_llh_kernel<L, 4>);
    };
    switch (lanes) {
      case 4: for_heads_per_lane(std::integral_constant<int, 4>()); break;
      case 8: for_heads_per_lane(std::integral_constant<int, 8>()); break;
      case 16: for_heads_per_lane(std::integral_constant<int, 16>()); break;
      default: for_heads_per_lane(std::integral_constant<int, 32>()); break;
    }
  } else {
    set_error("%s: %d heads on a bf16 table has no kernel yet (fp32 tables: any head count)", who, heads);
    return GTA_ERR_UNSUPPORTED;
  }
  GTA_CHECK_LAUNCH("gat_aggregate_kernel");
  return GTA_OK;
}

}  // namespace gta

using namespace gta;

extern "C" {

int32_t gta_gat_partial_stride(int32_t f, int32_t heads) { return gat_partial_stride(f, heads); }

int gta_er_stats(const float* er, int64_t lder, int64_t num_sources, int64_t col_block, int32_t heads,
                 uint32_t* stats, void* stream_) {
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  GTA_REQUIRE(er && stats && num_sources >= 0 && lder >= heads, "gta_er_stats: bad arguments");
  if (heads < 1 || heads > 32 || (heads & (heads - 1)) != 0) {
    set_error("gta_er_stats: heads=%d is not a power of two <= 32 (run the aggregation without er_stats)", heads);
    return GTA_ERR_UNSUPPORTED;
  }
  const int64_t n_cb = (col_block > 0 && col_block < num_sources) ? (num_sources + col_block - 1) / col_block : 1;
  GTA_REQUIRE(n_cb <= 65535, "gta_er_stats: %lld column blocks", (long long)n_cb);
  GTA_CUDA(cudaMemsetAsync(stats, 0, size_t(n_cb) * 2 * heads * sizeof(uint32_t), st));
  count_launch();
  if (num_sources == 0) return GTA_OK;
  const int64_t rows_per_block = n_cb > 1 ? col_block : num_sources;
  int64_t ctas = (rows_per_block * heads + 256 * 8 - 1) / (256 * 8);        // about 8 rows per thread
  if (ctas < 1) ctas = 1;
  if (ctas > 4 * kNumSMs) ctas = 4 * kNumSMs;
  er_stats_kernel<<<dim3((unsigned)ctas, (unsigned)n_cb), 256, 0, st>>>(er, lder, num_sources, n_cb > 1 ? col_block : 0,
                                                                         heads, stats);
  GTA_CHECK_LAUNCH("er_stats_kernel");
  return GTA_OK;
}

int gta_gat_aggregate_f32(const int32_t* items, int64_t num_items, const int32_t* row_slots, int64_t num_slots,
                          const int32_t* indices, const float* el, const float* er, int64_t lder, int32_t heads,
                          float slope, const float* z, int64_t ldz, float* out, int64_t ldo, int32_t f,
                          int32_t epilogue, float* rowmax, float* rowsum, float* partials, int32_t* chain_state,
                          const uint32_t* er_stats, int64_t col_block, const gta_exchange_t* exchange,
                          int32_t phases, void* stream) {
  return gat_aggregate_impl<float>("gta_gat_aggregate_f32", items, num_items, row_slots, num_slots, indices, el, er, lder,
                                   heads, slope, z, ldz, out, ldo, f, epilogue, rowmax, rowsum, partials, chain_state,
                                   er_stats, col_block, exchange, phases, stream);
}

int gta_gat_aggregate_bf16(const int32_t* items, int64_t num_items, const int32_t* row_slots, int64_t num_slots,
                           const int32_t* indices, const float* el, const float* er, int64_t lder, int32_t heads,
                           float slope, const void* z, int64_t ldz, float* out, int64_t ldo, int32_t f,
                           int32_t epilogue, float* rowmax, float* rowsum, float* partials, int32_t* chain_state,
                           const uint32_t* er_stats, int64_t col_block, const gta_exchange_t* exchange,
                           int32_t phases, void* stream) {
  return gat_aggregate_impl<__nv_bfloat16>("gta_gat_aggregate_bf16", items, num_items, row_slots, num_slots, indices, el,
                                           er, lder, heads, slope, static_cast<const __nv_bfloat16*>(z), ldz, out, ldo, f,
                                           epilogue, rowmax, rowsum, partials, chain_state, er_stats, col_block, exchange,
                                           phases, stream);
}

int gta_gat_logits_f32(const int64_t* indptr, const int32_t* indices, int64_t row_begin, int64_t row_end,
                       const float* el, const float* er, int32_t heads, float slope, int32_t stabilize, float* p,
                       float* rowmax, float* rowsum, void* stream_) {
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  GTA_REQUIRE(indptr && indices && el && er && p && rowsum, "gta_gat_logits_f32: null pointer");
  GTA_REQUIRE(heads >= 1, "gta_gat_logits_f32: heads must be >= 1");
  int64_t rows = row_end - row_begin;
  if (rows <= 0) return GTA_OK;
  gat_logits_kernel<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, st>>>(indptr, indices, row_begin, row_end, el, er,
                                                                         heads, slope, stabilize, p, rowmax, rowsum);
  GTA_CHECK_LAUNCH("gat_logits_kernel");
  return GTA_OK;
}

}  // extern "C"
