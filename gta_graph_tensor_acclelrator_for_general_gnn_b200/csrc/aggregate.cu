// Segmented scatter-reduce kernels: the HBM/L2-bound heart of the hot path.
//
//   aggregate_kernel      COMP_MUL_COMP_ADD / COMP_ADD gather  (interpreter.py:575-638, 85-106)        this file
//   edge_sum_kernel       PNA ops 5-8 in one pass (genGraphOP.py:110-147)                               this file
//   gat_aggregate_kernel  GAT ops 3-13 in one pass (genGraphOP.py:52-62), gat_aggregate_llh_kernel      gat_aggregate.cu
//   gat_logits_kernel     GAT block [4,5,6,7,8] alone (STORE_E p, STORE_N S), er_stats_kernel           gat_aggregate.cu
//   work list, item cursor, slot chain, piece types, launch helpers                                      aggregate_common.cuh
//
// Mapping.  A work item (<= chunk edges of one destination row inside one column block, see
// schedule.cu) is owned by a GROUP of LANES = min(F,128)/4 lanes; each lane owns 4 consecutive
// features, so one gathered source row is ONE 128-bit load per lane and a full 512 B row per 32
// lanes.  Wider rows (F > 128) are covered by blockIdx.y feature windows of 128.  Source ids (and
// scalar edge weights) are read once per group, coalesced and streaming (L1 no-allocate, L2
// evict_first), then handed round the group by shuffle / shared memory.  Gathered rows use the
// coherent path without L1 allocation (no reuse inside an SM) and with an L2 evict_last policy; L2
// residency comes from the column-block order of the work list.  Not the non-coherent (.nc) path: in
// an exchange the copy CTAs write the peers' slots of the table during the same launch, and .nc is
// only valid for data that no thread writes while the kernel runs.  kUnroll independent row loads are
// in flight per lane and a full batch runs without a single predicate.
//
// Rows that own several items (long rows cut at `chunk` edges, and every row when the table is walked
// in column blocks) form a CHAIN in slot order: an item reduces its own edges first, then waits for
// its predecessor's published state (a release/acquire flag per slot), folds it in, and either
// publishes the folded state or -- last item of the row -- normalises and writes the output.  The
// wait is at the END of an item and whoever holds the predecessor took it from the item counter earlier
// and is running, so it almost never spins and cannot deadlock; there is no separate merge launch and the
// last partial of every row is never written (round 1: a combine kernel re-read 507 MB in 0.24 ms).
//
// Determinism.  Every item is reduced by exactly one group in ascending source order and the chain
// is a left fold in slot order: a fixed-shape reduction, bitwise reproducible run to run, no atomics.
#include "aggregate_common.cuh"

namespace gta {

// ----------------------------------------------------------------------------------------
// weighted aggregate
//   WKIND 0: no weight, 1: scalar weight per edge (wh == 1), 2: per-head weight (wh > 1,
//   (f / wh) % kPer == 0 so a lane's features share a head; V == 1 only)
//   V: 16-byte pieces per lane and gathered row.  V = 2 lets one warp take a whole 1 KB row (256 fp32
//   features, the RMAT config) in one pass instead of walking the work list once per 128-feature window:
//   the indices, the item records and the page-table entries of a row are then touched once, not twice.
// ----------------------------------------------------------------------------------------
template <typename P, int V, int LANES, int WKIND, bool DIV>
__global__ void __launch_bounds__(kAggThreads, (V == 1 && P::kPer == 4) ? GTA_AGG_MINBLOCKS : 8)
aggregate_kernel(const WorkList wl, const Exchange ex, const float* __restrict__ w, int wh,
                 const float* __restrict__ rowden, const typename P::T* __restrict__ x, const uint32_t row_bytes,
                 float* __restrict__ out, int64_t ldo, int f, int epilogue) {
  static_assert(V == 1 || (LANES == 32 && WKIND != 2), "two pieces per lane: full warps, no per-head weights");
  using Raw = typename P::Raw;
  constexpr int KP = P::kPer;
  constexpr int kWindow = LANES * KP * V;          // features one pass of a group covers
  constexpr int kEdges = kAggUnroll;      // edges whose loads (V each) are in flight together
  __shared__ __align__(16) uint2 s_a[kAggWarps][32];        // per warp: {source id, weight} of the staged batch
  __shared__ __align__(16) NextItem s_next[kAggWarps][32 / LANES];
  if (ex.world > 1 && blockIdx.y == 0 && blockIdx.x < ex.copy_ctas) {
    exchange_pull(ex, blockIdx.x);          // these CTAs move the peers' slots; everybody else reduces
    return;
  }
  const int lane = threadIdx.x & 31;
  const int l = lane & (LANES - 1);
  const int fo = blockIdx.y * kWindow + KP * l;          // piece v sits at fo + v * LANES * KP
  uint2* se = s_a[threadIdx.x >> 5];
  const uint2* mine = se + (lane & ~(LANES - 1));
  const uint4* mine2 = reinterpret_cast<const uint4*>(mine);      // two staged edges per LDS.128
  int32_t* counter = wl.work_counter + blockIdx.y;
  int32_t* flags = wl.chain_flags + int64_t(blockIdx.y) * wl.num_slots;
  const uint64_t pol_stream = wl.pol_stream, pol_keep = wl.pol_keep;
  bool on[V];
#pragma unroll
  for (int v = 0; v < V; ++v) on[v] = fo + v * LANES * KP < f;
  const char* xf = reinterpret_cast<const char*>(x + (on[0] ? fo : 0));

  const ItemCursor first = cursor_begin<LANES>(wl, ex, counter, lane);
  int32_t landed = 0;          // exchange_gate: highest peer slot this lane has seen complete
  const int head = (WKIND == 2 && on[0]) ? fo / (f / wh) : 0;
  // what an item needs before its first batch (see NextItem): record, first ids (and scalar weights), the row's
  // denominator, and -- in an exchange -- its last id, which names the highest slot it touches
  int idx_nxt = 0, last_src = 0;
  float w_nxt = 0.f, den = 1.f;
  auto request_inputs = [&](const int4& t, bool hv) {
    const int cnt = hv ? t.z : 0;
    const int32_t* ib = wl.indices + t.y;
    idx_nxt = 0;
    w_nxt = 0.f;
    den = 1.f;
    if (l < cnt) {
      idx_nxt = ld_stream_i32(ib + l, pol_stream);
      if (WKIND == 1) w_nxt = ld_stream_f32(w + int64_t(t.y) * wh + l, pol_stream);
    }
    if (DIV && hv) den = rowden[int64_t(t.x) * wh + head];
    last_src = (ex.world > 1 && cnt > 0) ? __ldg(ib + cnt - 1) : 0;
  };
  ItemStage<LANES> stage(wl, first, lane, &s_next[threadIdx.x >> 5][lane / LANES]);
  request_inputs(stage.it, stage.have);
  while (stage.cur.first < wl.num_items) {
    stage.claim(wl, counter, lane);
    const int4 it = stage.it;
    const bool have = stage.have;
    const bool active = have && on[0];
    const int count = have ? it.z : 0;
    const int max_count = (LANES == 32) ? count : warp_max_i32(count);
    const int32_t* idx_base = wl.indices + it.y;
    const float* w_base = (WKIND != 0) ? w + int64_t(it.y) * wh : nullptr;
    const float den_cur = den;          // the next item's denominator replaces `den` before this item is folded

    float acc[V][KP];
#pragma unroll
    for (int v = 0; v < V; ++v)
#pragma unroll
      for (int c = 0; c < KP; ++c) acc[v][c] = 0.f;
    // software pipeline: ids (and scalar weights) of batch b+1 are in flight under the gathers of batch b
    if (ex.world > 1) {          // the item's slots may still be on their way from the peers
      if (l == 0 && count > 0) exchange_gate(ex, last_src, landed);
      __syncwarp();
    }
    for (int base = 0; base < max_count; base += LANES) {
      int n = count - base;
      n = n < 0 ? 0 : (n > LANES ? LANES : n);
      const int my_idx = idx_nxt;
      float my_w = (l < n) ? w_nxt : 0.f;
      // divide only where an edge exists: a neighbouring group's empty row has den = 0 (0/0 = NaN)
      if (WKIND == 1 && DIV && l < n) my_w = my_w / den_cur;
      if (base + LANES + l < count) {
        idx_nxt = ld_stream_i32(idx_base + base + LANES + l, pol_stream);
        if (WKIND == 1) w_nxt = ld_stream_f32(w_base + base + LANES + l, pol_stream);
      }
      // stage {source id, weight} of the batch in shared memory: one LDS.128 per two edges in the gather loop
      se[lane] = make_uint2(uint32_t(my_idx), __float_as_uint(WKIND == 1 ? my_w : 1.f));
      __syncwarp();
      const bool full = (LANES == 32) ? (n == LANES) : __all_sync(0xffffffffu, n == LANES && active);
      if (full && (V == 1 || on[V - 1])) {
        // whole batch, no predicates: kEdges * V loads in flight, then their FMAs (the outer loop stays
        // rolled: unrolled, ptxas hoists every load of the batch and spills)
        if (LANES < 32 || active) {
#pragma unroll 1
          for (int j = 0; j < LANES; j += kEdges) {
            uint4 ed[kEdges / 2];
            Raw raw[kEdges][V];
#pragma unroll
            for (int u = 0; u < kEdges / 2; ++u)
              if (j + 2 * u < LANES) ed[u] = mine2[(j >> 1) + u];
#pragma unroll
            for (int u = 0; u < kEdges; ++u) {
              if (j + u < LANES) {
                const char* rp = row_addr(xf, (u & 1) ? ed[u / 2].z : ed[u / 2].x, row_bytes);
#pragma unroll
                for (int v = 0; v < V; ++v) raw[u][v] = P::load(rp + v * LANES * P::kBytes, pol_keep);
              }
            }
#pragma unroll
            for (int u = 0; u < kEdges; ++u) {
              if (j + u < LANES) {
                float ws = __uint_as_float((u & 1) ? ed[u / 2].w : ed[u / 2].y);
                if (WKIND == 2) {
                  ws = __ldg(w_base + int64_t(base + j + u) * wh + head);
                  if (DIV) ws = ws / den_cur;
                }
#pragma unroll
                for (int v = 0; v < V; ++v) fma_row<P>(acc[v], ws, raw[u][v]);
              }
            }
          }
        }
      } else {
        const int nmax = (LANES == 32) ? n : LANES;
        for (int j = 0; j < nmax; j += kEdges) {
          Raw raw[kEdges][V];
          float wv[kEdges];
#pragma unroll
          for (int u = 0; u < kEdges; ++u) {
            if (j + u < LANES) {
              const uint2 ed = mine[j + u];
              const bool ok = have && (j + u) < n;
              float ws = ok ? __uint_as_float(ed.y) : 0.f;
              const char* rp = row_addr(xf, ed.x, row_bytes);
#pragma unroll
              for (int v = 0; v < V; ++v) {
                raw[u][v] = P::zero();
                if (ok && on[v]) raw[u][v] = P::load(rp + v * LANES * P::kBytes, pol_keep);
              }
              if (WKIND == 2) {
                ws = 0.f;
                if (ok && active) {
                  ws = __ldg(w_base + int64_t(base + j + u) * wh + head);
                  if (DIV) ws = ws / den_cur;
                }
              }
              wv[u] = ws;
            }
          }
#pragma unroll
          for (int u = 0; u < kEdges; ++u)
            if (j + u < LANES)
#pragma unroll
              for (int v = 0; v < V; ++v) fma_row<P>(acc[v], wv[u], raw[u][v]);
        }
      }
      __syncwarp();
    }
    const bool chained = have && it.w >= 0;
    const int4 next = stage.land(chained);
    request_inputs(next, stage.next_have);
    chain_step<LANES>(flags, lane, it, chained, [&]() { return stage.slots; },
        [&](int prev) {
#pragma unroll
          for (int v = 0; v < V; ++v) {
            if (have && on[v]) {
              float p[KP];
              ld_state<KP>(wl.partials + int64_t(prev) * f + fo + v * LANES * KP, p);
#pragma unroll
              for (int c = 0; c < KP; ++c) acc[v][c] = p[c] + acc[v][c];
            }
          }
        },
        [&](int slot) {
#pragma unroll
          for (int v = 0; v < V; ++v)
            if (have && on[v]) st_state<KP>(wl.partials + int64_t(slot) * f + fo + v * LANES * KP, acc[v]);
        },
        [&]() {
#pragma unroll
          for (int v = 0; v < V; ++v)
            if (have && on[v]) st_out<KP>(out + int64_t(it.x) * ldo + fo + v * LANES * KP, acc[v], 1.f, epilogue);
        });
    stage.advance(next);
  }
}

// ----------------------------------------------------------------------------------------
// Edge phase "sum of three, then a unary, then the row sum" in one pass (PNA ops 5-8,
// genGraphOP.py:110-147:  gather_R( SF( edge + scatterC(a) + scatterR(b) ) )):
//     out[i, :] = epilogue( sum_{k in row i} unary( edge[k, :] + x[src_k, :] + rowterm[i, :] ) )
// Any of the three terms may be absent.  The generic path materialises three E x F tensors (two adds and the
// unary) before the segment sum; here the E x F operand is read once, streaming, and nothing E x F is written.
// Same work list, dynamic item fetch and slot chain as aggregate_kernel; the reduction is the plain ascending
// edge order per lane.  A lane moves one 16-byte piece of every row it touches.
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ float edge_unary_value(float v, int unary, float slope) {
  if (unary == GTA_UN_RELU) return fmaxf(v, 0.f);
  if (unary == GTA_UN_ELU) return elu1(v);
  if (unary == GTA_UN_EXP_LEAKY_RELU) return expf(leaky(v, slope));
  return v;
}
template <int LANES, bool HAS_X, bool HAS_E>
__global__ void __launch_bounds__(kAggThreads, 8)
edge_sum_kernel(const WorkList wl, const Exchange ex, const float* __restrict__ edge, int64_t lde,
                const float* __restrict__ x, const uint32_t row_bytes, const float* __restrict__ rowterm, int64_t ldr,
                int unary, float slope, float* __restrict__ out, int64_t ldo, int f, int epilogue) {
  constexpr int kU = 4;
  __shared__ uint32_t s_id[kAggWarps][32];
  const int lane = threadIdx.x & 31;
  const int l = lane & (LANES - 1);
  const int fo = blockIdx.y * (LANES * 4) + 4 * l;
  uint32_t* sid = s_id[threadIdx.x >> 5];
  const uint32_t* mine = sid + (lane & ~(LANES - 1));
  int32_t* counter = wl.work_counter + blockIdx.y;
  int32_t* flags = wl.chain_flags + int64_t(blockIdx.y) * wl.num_slots;
  const uint64_t pol_stream = wl.pol_stream, pol_keep = wl.pol_keep;

  ItemCursor cur = cursor_begin<LANES>(wl, ex, counter, lane);
  while (cur.first < wl.num_items) {
    const int64_t group = int64_t(cur.first) + lane / LANES;
    const bool have = group < wl.num_items;
    const bool active = have && fo < f;
    const int4 it = have ? __ldg(wl.items + group) : make_int4(0, 0, 0, -1);
    const int count = have ? it.z : 0;
    const int max_count = (LANES == 32) ? count : warp_max_i32(count);
    const int32_t* idx_base = wl.indices + it.y;
    const char* xf = HAS_X ? reinterpret_cast<const char*>(x + (active ? fo : 0)) : nullptr;
    const float* ef = HAS_E ? edge + int64_t(it.y) * lde + (active ? fo : 0) : nullptr;
    float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (active && rowterm != nullptr) r4 = __ldg(reinterpret_cast<const float4*>(rowterm + int64_t(it.x) * ldr + fo));
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int idx_nxt = 0;
    if (HAS_X && l < count) idx_nxt = ld_stream_i32(idx_base + l, pol_stream);
    for (int base = 0; base < max_count; base += LANES) {
      int n = count - base;
      n = n < 0 ? 0 : (n > LANES ? LANES : n);
      if (HAS_X) {
        sid[lane] = uint32_t(idx_nxt);
        if (base + LANES + l < count) idx_nxt = ld_stream_i32(idx_base + base + LANES + l, pol_stream);
        __syncwarp();
      }
      const int nmax = (LANES == 32) ? n : LANES;
#pragma unroll 1
      for (int j = 0; j < nmax; j += kU) {
        float4 xv[kU], ev[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          const bool ok = active && (j + u) < n;
          xv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
          ev[u] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (HAS_X && ok) xv[u] = F32x4::unpack(F32x4::load(row_addr(xf, mine[(j + u) & (LANES - 1)], row_bytes), pol_keep));
          if (HAS_E && ok) ev[u] = ld_gather_f32x4(ef + int64_t(base + j + u) * lde, pol_stream);          // streamed: read once, evict first
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          if ((j + u) < n) {          // a padded slot would contribute unary(rowterm), not 0
            acc.x += edge_unary_value(ev[u].x + xv[u].x + r4.x, unary, slope);
            acc.y += edge_unary_value(ev[u].y + xv[u].y + r4.y, unary, slope);
            acc.z += edge_unary_value(ev[u].z + xv[u].z + r4.z, unary, slope);
            acc.w += edge_unary_value(ev[u].w + xv[u].w + r4.w, unary, slope);
          }
        }
      }
      if (HAS_X) __syncwarp();
    }
    const bool chained = have && it.w >= 0;
    chain_step<LANES>(flags, lane, it, chained,
        [&]() { return make_int2(__ldg(wl.row_slots + it.x), __ldg(wl.row_slots + it.x + 1)); },
        [&](int prev) {
          if (active) {
            const float4 p = ld_state_f32x4(wl.partials + int64_t(prev) * f + fo);
            acc.x = p.x + acc.x; acc.y = p.y + acc.y; acc.z = p.z + acc.z; acc.w = p.w + acc.w;
          }
        },
        [&](int slot) { if (active) *reinterpret_cast<float4*>(wl.partials + int64_t(slot) * f + fo) = acc; },
        [&]() { if (active) st_stream_f32x4(out + int64_t(it.x) * ldo + fo, epilogue4(acc, 1.f, epilogue)); });
    cursor_next<LANES>(cur, wl, counter, lane);
  }
}

// ----------------------------------------------------------------------------------------
// Roofline denominator of the gather kernels: random whole-row gathers from a table that fits L2, with the
// kernels' own load instruction (one 128-bit load per lane, L1 no-allocate, L2 evict_last), 8 in flight per
// lane, ids from a hash so nothing else touches memory.  bench.py reports gather bytes / time of the real
// kernel against this measured peak (roofline.l2_frac): the HBM roofline says little about a kernel whose
// 96 % of the traffic is L2 hits.
// ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kAggThreads, 8)
gather_peak_kernel(const float* __restrict__ table, uint32_t rows, uint32_t row_bytes, int lanes_per_row,
                   int64_t gathers_per_group, float4* __restrict__ sink, const uint64_t pol_keep) {
  const int lane = threadIdx.x & 31;
  const int l = lane % lanes_per_row;
  const uint64_t group = (uint64_t(blockIdx.x) * blockDim.x + threadIdx.x) / lanes_per_row;
  const char* base = reinterpret_cast<const char*>(table + 4 * l);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  uint32_t state = uint32_t(group * 2654435761u) | 1u;
  for (int64_t i = 0; i < gathers_per_group; i += 8) {
    float4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      state = state * 1664525u + 1013904223u;            // LCG: the lanes of a group draw the same ids
      const uint32_t id = uint32_t((uint64_t(state) * rows) >> 32);
      v[u] = F32x4::unpack(F32x4::load(row_addr(base, id, row_bytes), pol_keep));
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
  }
  if (acc.x == 1.2345e38f) sink[group] = acc;          // keeps the loads alive, never true in practice
}

template <typename P, int V, int LANES>
static void dispatch_aggregate(int wkind, bool div, cudaStream_t st, const WorkList& wl, const Exchange& ex,
                               const float* w, int wh, const float* rowden, const typename P::T* x, int64_t ldx,
                               float* out, int64_t ldo, int f, int epi) {
  using T = typename P::T;
  constexpr int kWin = LANES * P::kPer * V;
  const int grid_y = (f + kWin - 1) / kWin;
  auto launch = [&](auto kernel) {
    launch_persistent(kernel, wl, ex, LANES, grid_y, st, w, wh, rowden, x, uint32_t(ldx * sizeof(T)), out, ldo, f, epi);
  };
  if (wkind == 0) launch(aggregate_kernel<P, V, LANES, 0, false>);
  else if (wkind == 1 && !div) launch(aggregate_kernel<P, V, LANES, 1, false>);
  else if (wkind == 1 && div) launch(aggregate_kernel<P, V, LANES, 1, true>);
  else if constexpr (V == 1) {
    if (!div) launch(aggregate_kernel<P, V, LANES, 2, false>);
    else launch(aggregate_kernel<P, V, LANES, 2, true>);
  }
}

// ---- the two aggregation entry points, for either storage type of the gathered table ---------------
template <typename P>
static int aggregate_run(const char* who, int wkind, bool div, cudaStream_t st, const WorkList& wl, const Exchange& ex,
                         const float* w, int wh, const float* rowden, const typename P::T* x, int64_t ldx, float* out,
                         int64_t ldo, int f, int epilogue) {
  constexpr int KP = P::kPer;
  GTA_REQUIRE(f % KP == 0, "%s: f=%d must be a multiple of %d (pad the table)", who, f, KP);
  if (wkind == 2 && (f / wh) % KP != 0) {
    set_error("%s: per-head width f/wh=%d is not a multiple of %d", who, f / wh, KP);
    return GTA_ERR_UNSUPPORTED;
  }
  // rows wider than one 32-lane pass of single pieces: two pieces per lane (one walk of the work list, not two)
  if (f > 32 * KP && wkind != 2) {
    dispatch_aggregate<P, 2, 32>(wkind, div, st, wl, ex, w, wh, rowden, x, ldx, out, ldo, f, epilogue);
  } else if constexpr (KP == 8) {          // Bf16x8 only takes rows wider than 128 features: always 32 lanes
    dispatch_aggregate<P, 1, 32>(wkind, div, st, wl, ex, w, wh, rowden, x, ldx, out, ldo, f, epilogue);
  } else {
    switch (lanes_for(f, KP)) {
      case 4: dispatch_aggregate<P, 1, 4>(wkind, div, st, wl, ex, w, wh, rowden, x, ldx, out, ldo, f, epilogue); break;
      case 8: dispatch_aggregate<P, 1, 8>(wkind, div, st, wl, ex, w, wh, rowden, x, ldx, out, ldo, f, epilogue); break;
      case 16: dispatch_aggregate<P, 1, 16>(wkind, div, st, wl, ex, w, wh, rowden, x, ldx, out, ldo, f, epilogue); break;
      default: dispatch_aggregate<P, 1, 32>(wkind, div, st, wl, ex, w, wh, rowden, x, ldx, out, ldo, f, epilogue); break;
    }
  }
  return GTA_OK;
}

template <typename T>
static int aggregate_impl(const char* who, const int32_t* items_, int64_t num_items, const int32_t* row_slots,
                          int64_t num_slots, const int32_t* indices, int32_t wmode, const float* w, int32_t wh,
                          const float* rowden, const T* x, int64_t ldx, float* out, int64_t ldo, int32_t f,
                          int32_t epilogue, float* partials, int32_t* chain_state, const gta_exchange_t* exchange,
                          int32_t phases, void* stream_) {
  constexpr int kRow = 16 / int(sizeof(T));          // elements per 16 bytes: the row pitch granule
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  GTA_REQUIRE(f > 0 && f % 4 == 0, "%s: f=%d must be a positive multiple of 4 (pad the table)", who, f);
  WorkList wl;
  bool launch = false;
  int rc = prepare_worklist(who, items_, num_items, row_slots, num_slots, indices, partials, chain_state, f, phases, st,
                            &wl, &launch);
  if (rc != GTA_OK || !launch) return rc;
  GTA_REQUIRE(items_ && indices && x && out, "%s: null pointer", who);
  GTA_REQUIRE(ldx % kRow == 0 && ldo % 4 == 0 && ldx >= f && ldo >= f && ldx * int64_t(sizeof(T)) < (int64_t(1) << 32),
              "%s: leading dimensions must be whole 16-byte pieces, >= f, and a row below 4 GiB", who);
  GTA_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "%s: tables must be 16-byte aligned", who);
  GTA_REQUIRE(wmode >= GTA_W_NONE && wmode <= GTA_W_EDGE_DIV, "%s: bad wmode %d", who, wmode);
  int wkind = 0;
  bool div = wmode == GTA_W_EDGE_DIV;
  if (wmode != GTA_W_NONE) {
    GTA_REQUIRE(w && wh >= 1 && f % wh == 0, "%s: weight width %d must divide f=%d", who, wh, f);
    GTA_REQUIRE(!div || rowden, "%s: rowden required for GTA_W_EDGE_DIV", who);
    wkind = wh == 1 ? 1 : 2;
  }
  Exchange ex;
  rc = make_exchange(who, exchange, wl.work_counter + (f + 127) / 128, ldx * int64_t(sizeof(T)), &ex);
  if (rc != GTA_OK) return rc;
  GTA_REQUIRE(ex.world <= 1 || ex.table == reinterpret_cast<const char*>(x), "%s: x is not the exchange table", who);
  // bf16: 16-byte pieces of 8 features for rows wider than 128 whose width (and per-head width) is whole pieces of 8;
  // every other width of whole 4-feature pieces takes 8-byte pieces of 4 (two per lane above 128 features)
  if constexpr (sizeof(T) == 4) {
    rc = aggregate_run<F32x4>(who, wkind, div, st, wl, ex, w, wh, rowden, x, ldx, out, ldo, f, epilogue);
  } else if (f <= 128 || f % 8 != 0 || (wkind == 2 && (f / wh) % 8 != 0)) {
    rc = aggregate_run<Bf16x4>(who, wkind, div, st, wl, ex, w, wh, rowden, x, ldx, out, ldo, f, epilogue);
  } else {
    rc = aggregate_run<Bf16x8>(who, wkind, div, st, wl, ex, w, wh, rowden, x, ldx, out, ldo, f, epilogue);
  }
  if (rc != GTA_OK) return rc;
  GTA_CHECK_LAUNCH("aggregate_kernel");
  return GTA_OK;
}

}  // namespace gta

using namespace gta;

extern "C" {

int gta_aggregate_f32(const int32_t* items, int64_t num_items, const int32_t* row_slots, int64_t num_slots,
                      const int32_t* indices, int32_t wmode, const float* w, int32_t wh, const float* rowden,
                      const float* x, int64_t ldx, float* out, int64_t ldo, int32_t f, int32_t epilogue,
                      float* partials, int32_t* chain_state, const gta_exchange_t* exchange, int32_t phases,
                      void* stream) {
  return aggregate_impl<float>("gta_aggregate_f32", items, num_items, row_slots, num_slots, indices, wmode, w, wh, rowden,
                               x, ldx, out, ldo, f, epilogue, partials, chain_state, exchange, phases, stream);
}

int gta_aggregate_bf16(const int32_t* items, int64_t num_items, const int32_t* row_slots, int64_t num_slots,
                       const int32_t* indices, int32_t wmode, const float* w, int32_t wh, const float* rowden,
                       const void* x, int64_t ldx, float* out, int64_t ldo, int32_t f, int32_t epilogue,
                       float* partials, int32_t* chain_state, const gta_exchange_t* exchange, int32_t phases,
                       void* stream) {
  return aggregate_impl<__nv_bfloat16>("gta_aggregate_bf16", items, num_items, row_slots, num_slots, indices, wmode, w, wh,
                                       rowden, static_cast<const __nv_bfloat16*>(x), ldx, out, ldo, f, epilogue, partials,
                                       chain_state, exchange, phases, stream);
}

int gta_aggregate_edge_sum_f32(const int32_t* items_, int64_t num_items, const int32_t* row_slots, int64_t num_slots,
                               const int32_t* indices, const float* edge, int64_t lde, const float* x, int64_t ldx,
                               const float* rowterm, int64_t ldr, int32_t unary, float slope, float* out, int64_t ldo,
                               int32_t f, int32_t epilogue, float* partials, int32_t* chain_state, int32_t phases,
                               void* stream_) {
  const char* who = "gta_aggregate_edge_sum_f32";
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  GTA_REQUIRE(f > 0 && f % 4 == 0, "%s: f=%d must be a positive multiple of 4 (pad the table)", who, f);
  WorkList wl;
  bool launch = false;
  int rc = prepare_worklist(who, items_, num_items, row_slots, num_slots, indices, partials, chain_state, f, phases, st,
                            &wl, &launch);
  if (rc != GTA_OK || !launch) return rc;
  GTA_REQUIRE(items_ && out && (edge || x || rowterm), "%s: null pointer (at least one of edge / x / rowterm is needed)", who);
  GTA_REQUIRE(!x || indices, "%s: indices are required to gather x", who);
  GTA_REQUIRE(unary >= GTA_UN_EXP_LEAKY_RELU && unary <= GTA_UN_COPY, "%s: bad unary %d", who, unary);
  GTA_REQUIRE(ldo % 4 == 0 && ldo >= f && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "%s: out must be 16-byte aligned rows >= f", who);
  GTA_REQUIRE(!edge || (lde % 4 == 0 && lde >= f && (reinterpret_cast<uintptr_t>(edge) & 15) == 0),
              "%s: edge must be 16-byte aligned rows >= f", who);
  GTA_REQUIRE(!x || (ldx % 4 == 0 && ldx >= f && ldx * 4 < (int64_t(1) << 32) && (reinterpret_cast<uintptr_t>(x) & 15) == 0),
              "%s: x must be 16-byte aligned rows >= f, a row below 4 GiB", who);
  GTA_REQUIRE(!rowterm || (ldr % 4 == 0 && ldr >= f && (reinterpret_cast<uintptr_t>(rowterm) & 15) == 0),
              "%s: rowterm must be 16-byte aligned rows >= f", who);
  Exchange ex;
  memset(&ex, 0, sizeof(ex));
  const int lanes = lanes_for(f, 4);
  auto launch_es = [&](auto kernel) {
    launch_persistent(kernel, wl, ex, lanes, (f + 127) / 128, st, edge, lde, x, uint32_t(ldx * 4), rowterm, ldr, unary,
                      slope, out, ldo, f, epilogue);
  };
  auto for_terms = [&](auto lanes_c) {
    constexpr int L = decltype(lanes_c)::value;
    if (x && edge) launch_es(edge_sum_kernel<L, true, true>);
    else if (x) launch_es(edge_sum_kernel<L, true, false>);
    else if (edge) launch_es(edge_sum_kernel<L, false, true>);
    else launch_es(edge_sum_kernel<L, false, false>);
  };
  switch (lanes) {
    case 4: for_terms(std::integral_constant<int, 4>()); break;
    case 8: for_terms(std::integral_constant<int, 8>()); break;
    case 16: for_terms(std::integral_constant<int, 16>()); break;
    default: for_terms(std::integral_constant<int, 32>()); break;
  }
  GTA_CHECK_LAUNCH("edge_sum_kernel");
  return GTA_OK;
}

int gta_gather_peak_probe(const float* table, int64_t rows, int64_t ld, int32_t f, int64_t gathers_per_group,
                          float* sink, void* stream_) {
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  if (!(table && sink && rows > 0 && rows < (int64_t(1) << 32) && f >= 4 && f <= 128 && f % 4 == 0 && ld >= f &&
        ld % 4 == 0 && gathers_per_group > 0)) {
    set_error("gta_gather_peak_probe: bad arguments");
    return -GTA_ERR_INVALID;
  }
  CachePolicies pol;
  if (cache_policies(&pol) != GTA_OK) return -GTA_ERR_CUDA;
  const int lanes = lanes_for(f);
  const int ctas = resident_ctas(gather_peak_kernel);
  gather_peak_kernel<<<ctas, kAggThreads, 0, st>>>(table, uint32_t(rows), uint32_t(ld) * 4u, lanes, gathers_per_group,
                                                  reinterpret_cast<float4*>(sink), pol.keep);
  count_launch();
  if (check_cuda(cudaGetLastError(), "gather_peak_kernel") != GTA_OK) return -GTA_ERR_CUDA;
  return ctas * kAggThreads / lanes;          // > 0: the number of groups that ran (each did gathers_per_group gathers)
}

}  // extern "C"
