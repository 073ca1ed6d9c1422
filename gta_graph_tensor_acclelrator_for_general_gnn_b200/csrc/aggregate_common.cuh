// Shared by aggregate.cu and gat_aggregate.cu: the work list and its persistent-launch cursor, the slot chain of
// multi-item rows, next-item staging, piece types of the gathered table, and the host-side launch helpers.
// (See aggregate.cu for the mapping and the determinism argument.)
#pragma once
#include <cuda_bf16.h>
#include <string.h>

#include <mutex>
#include <type_traits>
#include <unordered_map>

#include "common.cuh"
#include "exchange.cuh"

namespace gta {

#ifndef GTA_AGG_THREADS
#define GTA_AGG_THREADS 128
#endif
// Resident CTAs per SM (caps the registers) and row loads in flight per lane, per kernel family.  Measured on
// B200, Reddit shape, persistent launch (tools/agg_probe.py, gpurun_out/p2_probe.log):
//   weighted aggregate   6x8: 3.36 ms   8x8: 3.29   8x4: 3.29   10x4: 3.13   (48 registers, no spills)
//   GAT staged (H <= 4)  6x8: 3.89 ms   7x8: 3.88   8x8: 3.75   8x4: 3.49   10x4: 4.11 (spills)
// More resident warps beat a deeper unroll: the kernels wait on L2 latency (long scoreboard), not on issue.
// The GAT kernel as it now stands (bound cache, next-item staging, single-exp chain fold) reverses that: bench.py reddit-gat,
// NVIDIA B200 at 1000 W, kernel ms:  8x4: 3.87-3.92   7x4: 3.66   6x4: 3.77   7x8: 3.60   6x8: 3.73   8x8: 3.54-3.63
// (36 B of spill stores at 64 registers); 8x8 is also fastest on reddit-heavy-gat and the bf16 table, outputs bitwise equal.
#ifndef GTA_AGG_MINBLOCKS
#define GTA_AGG_MINBLOCKS 10
#endif
#ifndef GTA_AGG_UNROLL
#define GTA_AGG_UNROLL 4
#endif
#ifndef GTA_GAT_MINBLOCKS
#define GTA_GAT_MINBLOCKS 8
#endif
#ifndef GTA_GAT_UNROLL
#define GTA_GAT_UNROLL 8
#endif
#ifndef GTA_LLH_MINBLOCKS
#define GTA_LLH_MINBLOCKS 6
#endif
#ifndef GTA_LLH_UNROLL
#define GTA_LLH_UNROLL 8
#endif
constexpr int kAggThreads = GTA_AGG_THREADS;
constexpr int kAggWarps = kAggThreads / 32;

// floats per partial slot of the GAT kernel: acc[f] | per 128-feature window: max[H] | sum[H], padded to 16 bytes
__host__ __device__ inline int gat_stats_stride(int heads) { return (2 * heads + 3) & ~3; }
__host__ __device__ inline int gat_partial_stride(int f, int heads) { return f + ((f + 127) / 128) * gat_stats_stride(heads); }

// ---- slot chain of a multi-item row ----------------------------------------------------------
// flag[slot] becomes 1 once the state folded over slots [first, slot] is in partials[slot].
__device__ __forceinline__ void chain_wait(const int32_t* flag) {
  // Poll with a RELAXED load and fence once on success.  An acquire load in the loop costs an L1 invalidation per
  // iteration (ptxas emits CCTL.IVALL behind every acquire at gpu scope): with rows split into consecutive items,
  // thousands of polling warps kept every SM's L1 empty and the 8-GPU step went from 0.90 to 2.5 ms.
  int32_t v = 0;
#pragma unroll 1
  for (uint32_t spin = 0; spin < (1u << 27); ++spin) {
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    if (v != 0) {
      asm volatile("fence.acq_rel.gpu;" ::: "memory");
      return;
    }
    __nanosleep(100);
  }
  __trap();      // the predecessor never published: a protocol bug must not hang the GPU
}
// Called by ONE lane after a __syncwarp of its group: the barrier orders the other lanes' state stores before
// this lane, and its fence + release store make them visible, cumulatively, to whoever acquires the flag -- the
// idiom of a cooperative grid barrier (block barrier, then one thread fences and signals).  One fence per
// item instead of one per lane: a membar.gl is the most expensive instruction of a short item.
__device__ __forceinline__ void chain_publish(int32_t* flag) {
  // st.release is cumulative over what the barrier ordered before this lane (the idiom of CUTLASS's Semaphore::release:
  // barrier, then one thread's st.release.gpu); a __threadfence() in front of it is a second, sequentially consistent
  // fence (membar.gl) per item and buys nothing
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(flag), "r"(1) : "memory");
}
// predecessor state was written by another SM during this launch: read it at L2, never from L1
__device__ __forceinline__ float4 ld_state_f32x4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float ld_state_f32(const float* p) { return __ldcg(p); }
template <int LANES>
__device__ __forceinline__ uint32_t group_mask(int lane) {
  if constexpr (LANES == 32) return 0xffffffffu;
  else return ((1u << LANES) - 1u) << (lane & ~(LANES - 1));
}
// Run `body` once per group of the warp, groups in ascending order (one pass when the warp is a single
// group or no group of it sits in a chain): a predecessor that lives in the SAME warp has then
// published before its successor waits.
template <int LANES, typename F>
__device__ __forceinline__ void for_groups_in_order(int lane, bool chained, F&& body) {
  if (LANES == 32 || !__any_sync(0xffffffffu, chained)) {
    body();
  } else {
#pragma unroll 1
    for (int g = 0; g < 32 / LANES; ++g) {
      if (lane / LANES == g) body();
      __syncwarp();
    }
  }
}
// The end of item `it` (record {row, first edge, count, slot}; slot < 0: the row has no other item).  A chained item
// that is not the first of its row waits for its predecessor's flag and calls fold(it.w - 1) to merge that slot's
// state; then it either calls save(it.w) and publishes, or -- last item of the row, or not chained -- calls finish()
// to write the output.  slots() returns the row's slot range {first, end} and is only called for a chained item.
template <int LANES, typename Slots, typename Fold, typename Save, typename Finish>
__device__ __forceinline__ void chain_step(int32_t* flags, int lane, const int4& it, bool chained, Slots&& slots,
                                           Fold&& fold, Save&& save, Finish&& finish) {
  for_groups_in_order<LANES>(lane, chained, [&]() {
    const bool leader = (lane & (LANES - 1)) == 0;
    bool last = true;
    if (chained) {
      const int2 s = slots();
      last = it.w == s.y - 1;
      if (it.w != s.x) {
        if (leader) chain_wait(flags + it.w - 1);
        __syncwarp(group_mask<LANES>(lane));
        fold(it.w - 1);
      }
      if (!last) {
        save(it.w);
        __syncwarp(group_mask<LANES>(lane));          // the group's stores happen-before lane 0's release
        if (leader) chain_publish(flags + it.w);
      }
    }
    if (last) finish();
  });
}

template <int LANES>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
  for (int o = LANES / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
template <int LANES>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = LANES / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_max_i32(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// exp of a non-positive softmax exponent: the ex2.approx path (relative error about 2e-7 + |x| 1e-7; terms that matter
// have small |x|), two instructions instead of about ten
__device__ __forceinline__ float softmax_exp(float x) { return __expf(x); }
__device__ __forceinline__ float4 epilogue4(float4 a, float scale, int epi) {
  a.x = apply_epilogue(a.x * scale, epi);
  a.y = apply_epilogue(a.y * scale, epi);
  a.z = apply_epilogue(a.z * scale, epi);
  a.w = apply_epilogue(a.w * scale, epi);
  return a;
}

// ----------------------------------------------------------------------------------------
// the work list, its chain state and the dynamic item counter every aggregation launch takes
// ----------------------------------------------------------------------------------------
struct WorkList {
  const int4* items;
  int64_t num_items;
  const int32_t* row_slots;
  int64_t num_slots;
  const int32_t* indices;
  float* partials;
  int32_t* chain_flags;      // [windows][num_slots]
  int32_t* work_counter;     // [windows], zeroed before every launch
  int32_t take;              // 1: warps take items from the counter; 0: static striding (long lists of tiny items)
  uint64_t pol_stream;
  uint64_t pol_keep;
};

// Persistent launch: every warp takes the next 32/LANES items from a global counter until the list is
// empty.  (Round 1 launched one CTA per 4 items: a CTA slot stayed occupied until its longest item was
// done and only 18 of the 24 resident warps per SM were active.)  The grab for the NEXT items is issued
// before the current ones are processed and its result is only read afterwards, so the atomic's round
// trip hides under the gathers.  Items are still started in work-list order, which keeps the CTAs on one
// column block at a time and keeps the chain invariant: whoever holds a predecessor slot started earlier
// and is running, so a wait can never deadlock, whatever the grid size.
// Long lists of tiny items (RMAT: millions of items of a few edges) do not need the balancing and would
// hammer the counter: with wl.take == 0 the warps stride through the list statically (warp w takes groups
// w, w + W, ...; the host then sizes the grid so that all W warps are resident, which the chain argument now
// needs).  Consecutive items still go to different warps -- taking several consecutive items per grab
// instead was measured 3x slower on RMAT-20: a hub row's chain of 1024-edge items then serialises, every
// warp sitting on its predecessor's publish while that warp works through the rest of its batch.
struct ItemCursor {
  int32_t first;       // first item of the warp's current group-step
  int32_t pending;     // dynamic: the next grab (lane 0), in flight
  int32_t stride;      // static: items between two steps of this warp
};
template <int LANES>
__device__ __forceinline__ ItemCursor cursor_begin(const WorkList& wl, const Exchange& ex, int32_t* counter, int lane) {
  constexpr int kGroups = 32 / LANES;
  ItemCursor c;
  if (wl.take > 0) {
    int32_t v = 0;
    if (lane == 0) v = atomicAdd(counter, kGroups);
    c.first = __shfl_sync(0xffffffffu, v, 0);
    c.pending = 0;
    if (lane == 0) c.pending = atomicAdd(counter, kGroups);
    c.stride = 0;
  } else {
    // the copy CTAs of an exchange exist in feature window 0 only (they pull and return); in every other window
    // all of gridDim.x are work CTAs, so the warps of each window cover [0, num_items) exactly once
    const int copy = (ex.world > 1 && blockIdx.y == 0) ? ex.copy_ctas : 0;
    c.first = ((int32_t(blockIdx.x) - copy) * kAggWarps + int32_t(threadIdx.x >> 5)) * kGroups;
    c.stride = (int32_t(gridDim.x) - copy) * kAggWarps * kGroups;
    c.pending = 0;
  }
  return c;
}
template <int LANES>
__device__ __forceinline__ void cursor_next(ItemCursor& c, const WorkList& wl, int32_t* counter, int lane) {
  if (wl.take > 0) {
    c.first = __shfl_sync(0xffffffffu, c.pending, 0);
    if (c.first < wl.num_items && lane == 0) c.pending = atomicAdd(counter, 32 / LANES);
  } else {
    c.first = (c.first > 0x7fffffff - c.stride) ? 0x7fffffff : c.first + c.stride;
  }
}

// ---- the next item, staged while the current one runs ------------------------------------------
// An item costs a chain of dependent loads before its first gather can issue: the item record, then its first source
// ids (streamed from DRAM) and el row, then the er rows of those ids; and two row_slots reads in front of the chain fold.
// Measured on the Reddit shape (agg_probe, items of 20 edges against items of 164): about 5 us of warp time per item
// whatever its length, a quarter of the kernel.  The record of the NEXT item and the slot range of the CURRENT row are
// therefore copied into shared memory asynchronously at the top of an item (no registers held across the gather loop),
// and the next item's el row and first two id batches are requested right after the gather loop, so that they travel
// while the chain fold of the current item waits for its predecessor.
struct NextItem {
  int4 item;
  int32_t s0, s1, pad0, pad1;
};
__device__ __forceinline__ void cp_async_16(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(uint32_t(__cvta_generic_to_shared(smem))), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_4(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(uint32_t(__cvta_generic_to_shared(smem))), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// A warp group's walk of the work list with that staging, from the cursor of its first group-step (whose item is read
// directly).  Per item, in this order:
//   claim()        top of the item: take the next group-step, cp.async its record and this row's slot range
//   land()         after the gather loop: wait for the copies, return the next record and read `slots` (the
//                  staging entry is free again)
//   advance(next)  after the chain step: the next item becomes the current one
// The kernel requests its own inputs of `it` after construction and of the next item right after land().
template <int LANES>
struct ItemStage {
  ItemCursor cur, nxt;
  int4 it = make_int4(0, 0, 0, -1);
  bool have = false, next_have;
  int2 slots;                // this row's slot range, read in land() when the item is chained
  NextItem* nx;
  __device__ __forceinline__ ItemStage(const WorkList& wl, const ItemCursor& first, int lane, NextItem* entry)
      : cur(first), nx(entry) {
    const int64_t group = int64_t(cur.first) + lane / LANES;
    have = group < wl.num_items;
    if (have) it = __ldg(wl.items + group);
  }
  __device__ __forceinline__ void claim(const WorkList& wl, int32_t* counter, int lane) {
    nxt = cur;
    cursor_next<LANES>(nxt, wl, counter, lane);
    const int64_t ngroup = int64_t(nxt.first) + lane / LANES;
    next_have = nxt.first < wl.num_items && ngroup < wl.num_items;
    if ((lane & (LANES - 1)) == 0) {
      if (next_have) cp_async_16(&nx->item, wl.items + ngroup);
      if (have && it.w >= 0) {
        cp_async_4(&nx->s0, wl.row_slots + it.x);
        cp_async_4(&nx->s1, wl.row_slots + it.x + 1);
      }
    }
  }
  __device__ __forceinline__ int4 land(bool chained) {
    cp_async_wait_all();
    __syncwarp();
    const int4 next = next_have ? nx->item : make_int4(0, 0, 0, -1);
    slots = make_int2(chained ? nx->s0 : 0, chained ? nx->s1 : 0);
    __syncwarp();          // everybody has read the staging entry before lane 0 of the group overwrites it
    return next;
  }
  __device__ __forceinline__ void advance(const int4& next) {
    cur = nxt;
    it = next;
    have = next_have;
  }
};

// ----------------------------------------------------------------------------------------
// storage type of the gathered table: fp32, or bf16 with fp32 accumulation (SURVEY.md section 8d "bf16 mode";
// the reference's IR declares data_format FP16, template/IR_defination.yaml:10-27).  A lane always moves
// 16-byte pieces of a row: 4 fp32 or 8 bf16 features.
// ----------------------------------------------------------------------------------------
// A PIECE is what one lane moves of one gathered row: its storage type, how many features, how many bytes.
//   F32x4   4 fp32 in 16 bytes            (512-byte rows at 32 lanes: the fp32 mode)
//   Bf16x8  8 bf16 in 16 bytes            (rows wider than 128 features whose width, and per-head width, is a
//                                          multiple of 8; always 32 lanes)
//   Bf16x4  4 bf16 in  8 bytes            (rows of up to 128 features keep all 32 lanes on ONE item: the per-batch
//                                          work -- staging, softmax -- is then spread over 32 edges, not 16; measured
//                                          on the Reddit shape: Bf16x8 at 16 lanes per item was no faster than fp32.
//                                          Also wider rows of any other multiple of 4: two pieces per lane in the
//                                          aggregate, windows of 128 in the GAT kernel)
struct F32x4 {
  using T = float;
  using Raw = uint4;
  static constexpr int kPer = 4, kBytes = 16;
  static __device__ __forceinline__ Raw load(const char* p, uint64_t pol) {
    Raw v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
    return v;
  }
  static __device__ __forceinline__ Raw zero() { return make_uint4(0u, 0u, 0u, 0u); }
  static __device__ __forceinline__ void unpack(const Raw& r, float (&f)[4]) {
    f[0] = __uint_as_float(r.x); f[1] = __uint_as_float(r.y); f[2] = __uint_as_float(r.z); f[3] = __uint_as_float(r.w);
  }
  static __device__ __forceinline__ float4 unpack(const Raw& r) {
    return make_float4(__uint_as_float(r.x), __uint_as_float(r.y), __uint_as_float(r.z), __uint_as_float(r.w));
  }
};
struct Bf16x8 {
  using T = __nv_bfloat16;
  using Raw = uint4;
  static constexpr int kPer = 8, kBytes = 16;
  static __device__ __forceinline__ Raw load(const char* p, uint64_t pol) { return F32x4::load(p, pol); }
  static __device__ __forceinline__ Raw zero() { return make_uint4(0u, 0u, 0u, 0u); }
  static __device__ __forceinline__ void unpack(const Raw& r, float (&f)[8]) {      // bf16 -> fp32 is a shift
    f[0] = __uint_as_float(r.x << 16); f[1] = __uint_as_float(r.x & 0xffff0000u);
    f[2] = __uint_as_float(r.y << 16); f[3] = __uint_as_float(r.y & 0xffff0000u);
    f[4] = __uint_as_float(r.z << 16); f[5] = __uint_as_float(r.z & 0xffff0000u);
    f[6] = __uint_as_float(r.w << 16); f[7] = __uint_as_float(r.w & 0xffff0000u);
  }
};
struct Bf16x4 {
  using T = __nv_bfloat16;
  using Raw = uint2;
  static constexpr int kPer = 4, kBytes = 8;
  static __device__ __forceinline__ Raw load(const char* p, uint64_t pol) {
    Raw v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v2.u32 {%0,%1}, [%2], %3;"
                 : "=r"(v.x), "=r"(v.y) : "l"(p), "l"(pol));
    return v;
  }
  static __device__ __forceinline__ Raw zero() { return make_uint2(0u, 0u); }
  static __device__ __forceinline__ void unpack(const Raw& r, float (&f)[4]) {
    f[0] = __uint_as_float(r.x << 16); f[1] = __uint_as_float(r.x & 0xffff0000u);
    f[2] = __uint_as_float(r.y << 16); f[3] = __uint_as_float(r.y & 0xffff0000u);
  }
};
// address of a gathered row: base + id * row_bytes.  Written as a 64-bit multiply-add of two 32-bit
// values so ptxas emits ONE IMAD.WIDE.U32 with the lane's base pointer as the addend (an inline
// mad.wide.u32 was split into IMAD.WIDE + IADD3 + IADD3.X once the base pair was not register-aligned).
__device__ __forceinline__ const char* row_addr(const char* base, uint32_t id, uint32_t row_bytes) {
  return base + uint64_t(id) * row_bytes;
}
template <typename P>
__device__ __forceinline__ void fma_row(float (&acc)[P::kPer], float w, const typename P::Raw& raw) {
  float f[P::kPer];
  P::unpack(raw, f);
#pragma unroll
  for (int c = 0; c < P::kPer; ++c) acc[c] = fmaf(w, f[c], acc[c]);
}
// kPer consecutive fp32 of an output / partial row
template <int KP>
__device__ __forceinline__ void st_out(float* p, const float (&a)[KP], float scale, int epi) {
#pragma unroll
  for (int q = 0; q < KP / 4; ++q)
    st_stream_f32x4(p + 4 * q, make_float4(apply_epilogue(a[4 * q] * scale, epi), apply_epilogue(a[4 * q + 1] * scale, epi),
                                           apply_epilogue(a[4 * q + 2] * scale, epi), apply_epilogue(a[4 * q + 3] * scale, epi)));
}
template <int KP>
__device__ __forceinline__ void st_state(float* p, const float (&a)[KP]) {
#pragma unroll
  for (int q = 0; q < KP / 4; ++q)
    *reinterpret_cast<float4*>(p + 4 * q) = make_float4(a[4 * q], a[4 * q + 1], a[4 * q + 2], a[4 * q + 3]);
}
template <int KP>
__device__ __forceinline__ void ld_state(const float* p, float (&a)[KP]) {
#pragma unroll
  for (int q = 0; q < KP / 4; ++q) {
    const float4 t = ld_state_f32x4(p + 4 * q);
    a[4 * q] = t.x; a[4 * q + 1] = t.y; a[4 * q + 2] = t.z; a[4 * q + 3] = t.w;
  }
}

constexpr int kAggUnroll = GTA_AGG_UNROLL;
constexpr int kGatUnroll = GTA_GAT_UNROLL;
constexpr int kLlhUnroll = GTA_LLH_UNROLL;

// ----------------------------------------------------------------------------------------
// host side: lanes per item, persistent launch, exchange descriptor, work-list preparation
// ----------------------------------------------------------------------------------------
// lanes per item for rows of f features, kper features per 16-byte piece, v pieces per lane
static int lanes_for(int f, int kper = 4, int v = 1) {
  const int window = 32 * kper * v;
  int need = ((f < window ? f : window) + kper * v - 1) / (kper * v);
  int l = 1;
  while (l < need) l <<= 1;
  return l < 4 ? 4 : l;
}

// Cached per kernel, not per template argument K: K is the kernel's function-pointer type, which instances of one
// parameter list share (aggregate_kernel with one piece per lane at 48 registers, 10 CTAs per SM, and with two pieces
// at 64 registers, 8 per SM).  A count taken from another instance oversizes the grid, and static striding needs every
// CTA of a window resident: a chain then waits on a CTA that cannot start.
template <typename K>
static int resident_ctas(K kernel) {
  static std::mutex lock;
  static std::unordered_map<const void*, int> cached;
  std::lock_guard<std::mutex> hold(lock);
  const auto hit = cached.find(reinterpret_cast<const void*>(kernel));
  if (hit != cached.end()) return hit->second;
  int per_sm = 0, dev = 0, sms = kNumSMs;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kAggThreads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return cached[reinterpret_cast<const void*>(kernel)] = per_sm * sms;
}

// dynamic item fetch (take = 1) unless the caller asked for static striding (GTA_PHASE_STATIC: long lists of
// tiny items) and the list is long enough for every resident warp to get a few dozen group-steps
template <typename K>
static int32_t take_for(K kernel, const WorkList& wl, int lanes) {
  const int groups = 32 / lanes;
  const int64_t warps = int64_t(resident_ctas(kernel)) * (kAggThreads / 32);
  return (wl.take == 0 && wl.num_items / (warps * groups) >= 32) ? 0 : 1;      // wl.take == 0: the caller's hint
}

// Persistent launch of an aggregation kernel whose parameters are (WorkList, Exchange, args...): as many CTAs as the
// items need, at most as many as are resident, times grid_y feature windows, with the item fetch chosen for this list.
template <typename K, typename... Args>
static void launch_persistent(K kernel, WorkList wl, const Exchange& ex, int lanes, int grid_y, cudaStream_t st,
                              Args... args) {
  wl.take = take_for(kernel, wl, lanes);
  const int64_t need = (wl.num_items * lanes + kAggThreads - 1) / kAggThreads;
  int64_t cap = resident_ctas(kernel);
  // the copy CTAs of an exchange come first in the grid, so they are resident before any CTA can wait on them;
  // with static striding every work CTA must be resident too (a chain may wait on any of them)
  const int64_t copy = ex.world > 1 ? ex.copy_ctas : 0;
  if (wl.take == 0 && cap > copy + 1) cap -= copy;
  const dim3 grid((unsigned)((need < cap ? need : cap) + copy), (unsigned)grid_y);
  kernel<<<grid, kAggThreads, 0, st>>>(wl, ex, args...);
}

// gta_exchange_t (host) -> Exchange (kernel parameter); arrived[] lives behind the item counters
static int make_exchange(const char* who, const gta_exchange_t* h, int32_t* arrived, int64_t pitch_bytes, Exchange* ex) {
  memset(ex, 0, sizeof(*ex));
  if (h == nullptr || h->world <= 1) return GTA_OK;
  GTA_REQUIRE(h->world <= GTA_MAX_RANKS && h->rank >= 0 && h->rank < h->world && h->step >= 1,
              "%s: exchange world %d rank %d step %d", who, h->world, h->rank, h->step);
  GTA_REQUIRE(h->table && h->signals && h->slot_rows > 0, "%s: exchange table / signals / slot_rows missing", who);
  GTA_REQUIRE(h->row_bytes == pitch_bytes && h->row_bytes % 16 == 0,
              "%s: exchange row_bytes %lld does not match the table's row pitch %lld", who, (long long)h->row_bytes,
              (long long)pitch_bytes);
  GTA_REQUIRE((h->slot_rows * h->row_bytes) % 128 == 0,
              "%s: a slot (%lld rows of %lld bytes) must be a whole number of 128-byte lines", who,
              (long long)h->slot_rows, (long long)h->row_bytes);
  ex->world = h->world;
  ex->copy_ctas = h->copy_ctas > 0 ? h->copy_ctas : 96;
  ex->step = h->step;
  ex->row_bytes = uint32_t(h->row_bytes);
  ex->slot_rows = h->slot_rows;
  ex->table = static_cast<char*>(h->table);
  ex->signals = static_cast<const ExchangeSignals*>(h->signals);
  ex->arrived = arrived;
  for (int k = 0; k < h->world; ++k) {
    GTA_REQUIRE(k == 0 || h->peer_table[k], "%s: table of slot %d's owner is not mapped", who, k);
    GTA_REQUIRE(h->slot_valid_rows[k] >= 0 && h->slot_valid_rows[k] <= h->slot_rows, "%s: slot %d has %lld rows", who, k,
                (long long)h->slot_valid_rows[k]);
    ex->peer[k] = static_cast<const char*>(h->peer_table[k]);
    ex->valid_rows[k] = int32_t(h->slot_valid_rows[k]);
  }
  return GTA_OK;
}

// The work list of an entry point: the common argument checks, the RESET phase (clear the chain flags of every
// feature window) and the item counters (cleared before every launch).  chain_state = [windows][num_slots] flags,
// then [windows] item counters, then GTA_MAX_RANKS slot-arrival counters of an exchange.  *launch: the call has a
// MAIN phase with items to reduce.
static int prepare_worklist(const char* who, const int32_t* items, int64_t num_items, const int32_t* row_slots,
                            int64_t num_slots, const int32_t* indices, float* partials, int32_t* chain_state, int32_t f,
                            int32_t phases, cudaStream_t st, WorkList* wl, bool* launch) {
  *launch = false;
  GTA_REQUIRE(num_items >= 0 && num_items < (int64_t(1) << 31) - 64, "%s: bad item count", who);
  GTA_REQUIRE(chain_state, "%s: chain_state is required (chain flags and the item counters live there)", who);
  GTA_REQUIRE(num_slots == 0 || (partials && row_slots),
              "%s: partials and row_slots are required for %lld slots", who, (long long)num_slots);
  const size_t windows = size_t((f + 127) / 128);
  *wl = WorkList{};
  wl->items = reinterpret_cast<const int4*>(items);
  wl->num_items = num_items;
  wl->row_slots = row_slots;
  wl->num_slots = num_slots;
  wl->indices = indices;
  wl->partials = partials;
  wl->chain_flags = chain_state;
  wl->work_counter = chain_state + windows * size_t(num_slots);
  wl->take = (phases & GTA_PHASE_STATIC) ? 0 : 1;
  if ((phases & GTA_PHASE_RESET) && num_slots > 0) {
    GTA_CUDA(cudaMemsetAsync(wl->chain_flags, 0, windows * size_t(num_slots) * sizeof(int32_t), st));
    count_launch();
  }
  if (!(phases & GTA_PHASE_MAIN) || num_items == 0) return GTA_OK;
  GTA_CUDA(cudaMemsetAsync(wl->work_counter, 0, (windows + GTA_MAX_RANKS) * sizeof(int32_t), st));
  count_launch();
  CachePolicies pol;
  const int rc = cache_policies(&pol);
  if (rc != GTA_OK) return rc;
  wl->pol_stream = pol.stream;
  wl->pol_keep = pol.keep;
  *launch = true;
  return GTA_OK;
}

}  // namespace gta
