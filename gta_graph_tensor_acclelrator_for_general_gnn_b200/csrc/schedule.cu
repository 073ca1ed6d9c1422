// Work list of the aggregation kernels (gta_schedule_build).
//
// The reference walks the adjacency as TR x TC tiles, row tile major, source column ascending
// (interpreter.py:85-106 judge_comp_inst_tile; simulator.py:262-263,292).  On B200 the unit of
// work is an ITEM: at most `chunk` consecutive CSR edges of one destination row, all of whose
// sources fall into one COLUMN BLOCK of `col_block` source ids.  Items are ordered by
// (column block, row, position), so the CTAs resident at any moment gather from one slice of
// the source table -- sized by the caller to stay L2 resident (126 MB L2, two dies) -- while every
// row still sees its edges in ascending source order.  Rows that own more than one item reduce
// through numbered partial slots, merged in slot order by the combine kernels: a fixed-shape,
// deterministic reduction.
//
//   items     int32[4] per item: {row (relative to row_begin), edge_begin, edge_count, slot | -1}
//   row_slots int32[rows+1]: slots of row r are [row_slots[r], row_slots[r+1])  (empty if 1 item)
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace gta {

constexpr int kMaxColBlocks = 64;

// upper source-id bound of every column block (block cb holds sources below end[cb] that are not in an
// earlier block): uniform (cb + 1) * col_block, or the caller's cut points (an exchange walks its peers'
// slots in a few groups of growing size)
struct BlockEnds {
  int64_t end[kMaxColBlocks];
};

// first position in indices[b,e) whose source id is >= bound
__device__ __forceinline__ int64_t lower_bound_src(const int32_t* __restrict__ indices, int64_t b, int64_t e, int64_t bound) {
  while (b < e) {
    int64_t mid = (b + e) >> 1;
    if (int64_t(indices[mid]) < bound) b = mid + 1; else e = mid;
  }
  return b;
}

__device__ __forceinline__ int32_t items_of(int64_t len, int32_t chunk) { return int32_t((len + chunk - 1) / chunk); }

// counts[cb * rows + r] = items of (column block cb, row r); row_items[r] = total of the row
__global__ void sched_count_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                   int64_t row_begin, int64_t rows, int32_t chunk, const BlockEnds ends, int32_t n_cb,
                                   int32_t* __restrict__ counts, int32_t* __restrict__ row_slots_in) {
  int64_t r = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (; r < rows; r += stride) {
    const int64_t b = indptr[row_begin + r], e = indptr[row_begin + r + 1];
    int32_t total = 0;
    if (n_cb == 1) {
      total = b == e ? 1 : items_of(e - b, chunk);
      counts[r] = total;
    } else {
      int64_t lo = b;
      for (int32_t cb = 0; cb < n_cb; ++cb) {
        int64_t hi = (cb == n_cb - 1) ? e : lower_bound_src(indices, lo, e, ends.end[cb]);
        int32_t n = items_of(hi - lo, chunk);
        if (cb == 0 && b == e) n = 1;           // an empty row still writes its zero output
        counts[int64_t(cb) * rows + r] = n;
        total += n;
        lo = hi;
      }
    }
    row_slots_in[r] = total > 1 ? total : 0;
  }
}

__global__ void sched_fill_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                  int64_t row_begin, int64_t rows, int32_t chunk, const BlockEnds ends, int32_t n_cb,
                                  const int32_t* __restrict__ item_off, const int32_t* __restrict__ row_slots,
                                  int4* __restrict__ items) {
  int64_t r = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (; r < rows; r += stride) {
    const int64_t b = indptr[row_begin + r], e = indptr[row_begin + r + 1];
    const int32_t slot0 = row_slots[r];
    const bool multi = row_slots[r + 1] > slot0;
    int32_t slot = slot0;
    int64_t lo = b;
    for (int32_t cb = 0; cb < n_cb; ++cb) {
      int64_t hi = (cb == n_cb - 1) ? e : lower_bound_src(indices, lo, e, ends.end[cb]);
      int32_t n = items_of(hi - lo, chunk);
      if (cb == 0 && b == e) n = 1;
      int32_t o = item_off[int64_t(cb) * rows + r];
      // the segment's n items are cut EVENLY (a multiple of 32 edges each but the last), not chunk, chunk, ...,
      // remainder: the items of a row run concurrently on neighbouring warps and the later one waits for the
      // earlier one's state, so [128, 36] makes a warp idle for 92 edges' worth of time where [96, 68] costs 28
      int64_t per = n > 0 ? ((hi - lo + n - 1) / n + 31) / 32 * 32 : chunk;
      if (per > chunk) per = chunk;
      for (int32_t c = 0; c < n; ++c) {
        int64_t cbeg = lo + int64_t(c) * per;
        if (cbeg > hi) cbeg = hi;
        int64_t cend = (c == n - 1) ? hi : (cbeg + per < hi ? cbeg + per : hi);
        items[o + c] = make_int4(int32_t(r), int32_t(cbeg), int32_t(cend - cbeg), multi ? slot : -1);
        ++slot;
      }
      lo = hi;
    }
  }
}

static int sched_grid(int64_t n) {
  int64_t g = (n + 255) / 256;
  int64_t cap = int64_t(kNumSMs) * 16;
  return int(g > cap ? cap : (g < 1 ? 1 : g));
}

static int32_t col_blocks_for(int64_t num_sources, int64_t col_block) {
  if (col_block <= 0 || col_block >= num_sources) return 1;
  return int32_t((num_sources + col_block - 1) / col_block);
}

}  // namespace gta

using namespace gta;

extern "C" {

int32_t gta_schedule_col_blocks(int64_t num_sources, int64_t col_block) { return col_blocks_for(num_sources, col_block); }

size_t gta_schedule_workspace(int64_t num_rows, int64_t num_sources, int64_t col_block) {
  const int64_t n_cb = col_blocks_for(num_sources, col_block);
  const int64_t n = num_rows * n_cb + 1;
  size_t cub_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, (int32_t*)nullptr, (int32_t*)nullptr, n);
  return 2 * align_up(size_t(n) * 4, 256) + align_up(size_t(num_rows + 1) * 4, 256) + align_up(cub_bytes, 256);
}

int64_t gta_schedule_max_items(int64_t num_rows, int64_t num_edges, int32_t chunk, int64_t num_sources,
                               int64_t col_block) {
  if (chunk <= 0) return -1;
  return num_rows * col_blocks_for(num_sources, col_block) + num_edges / chunk + 1;
}

// shared body: n_cb column blocks whose upper bounds are ends.end[0 .. n_cb-2] (the last block takes the rest)
static int schedule_build_impl(const int64_t* indptr, const int32_t* indices, int64_t row_begin, int64_t row_end,
                               int32_t chunk, const BlockEnds& ends, int32_t n_cb, int64_t ws_col_block,
                               int64_t ws_sources, int32_t* items, int64_t items_capacity, int32_t* row_slots,
                               int64_t* h_counts, int64_t* h_block_begin, void* workspace, size_t workspace_bytes,
                               void* stream_);

int gta_schedule_build(const int64_t* indptr, const int32_t* indices, int64_t row_begin, int64_t row_end,
                       int64_t num_sources, int32_t chunk, int64_t col_block, int32_t* items,
                       int64_t items_capacity, int32_t* row_slots, int64_t* h_counts, int64_t* h_block_begin,
                       void* workspace, size_t workspace_bytes, void* stream_) {
  const int32_t n_cb = col_blocks_for(num_sources, col_block);
  GTA_REQUIRE(n_cb <= kMaxColBlocks, "gta_schedule_build: %d column blocks exceed the limit of %d", n_cb, kMaxColBlocks);
  BlockEnds ends{};
  for (int32_t cb = 0; cb < n_cb; ++cb) ends.end[cb] = int64_t(cb + 1) * col_block;
  return schedule_build_impl(indptr, indices, row_begin, row_end, chunk, ends, n_cb, col_block, num_sources, items,
                             items_capacity, row_slots, h_counts, h_block_begin, workspace, workspace_bytes, stream_);
}

int gta_schedule_build_cuts(const int64_t* indptr, const int32_t* indices, int64_t row_begin, int64_t row_end,
                            int32_t chunk, const int64_t* h_cuts, int32_t num_cuts, int32_t* items,
                            int64_t items_capacity, int32_t* row_slots, int64_t* h_counts, int64_t* h_block_begin,
                            void* workspace, size_t workspace_bytes, void* stream_) {
  GTA_REQUIRE(num_cuts >= 0 && num_cuts < kMaxColBlocks && (num_cuts == 0 || h_cuts), "gta_schedule_build_cuts: %d cuts", num_cuts);
  BlockEnds ends{};
  for (int32_t c = 0; c < num_cuts; ++c) {
    GTA_REQUIRE(h_cuts[c] > (c ? h_cuts[c - 1] : 0), "gta_schedule_build_cuts: cut points must be positive and ascending");
    ends.end[c] = h_cuts[c];
  }
  // workspace as for num_cuts + 1 uniform blocks: gta_schedule_workspace(rows, num_cuts + 1, 1)
  return schedule_build_impl(indptr, indices, row_begin, row_end, chunk, ends, num_cuts + 1, 1, num_cuts + 1, items,
                             items_capacity, row_slots, h_counts, h_block_begin, workspace, workspace_bytes, stream_);
}

static int schedule_build_impl(const int64_t* indptr, const int32_t* indices, int64_t row_begin, int64_t row_end,
                               int32_t chunk, const BlockEnds& ends, int32_t n_cb, int64_t ws_col_block,
                               int64_t ws_sources, int32_t* items, int64_t items_capacity, int32_t* row_slots,
                               int64_t* h_counts, int64_t* h_block_begin, void* workspace, size_t workspace_bytes,
                               void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  GTA_REQUIRE(indptr && items && row_slots && h_counts && workspace, "gta_schedule_build: null pointer");
  GTA_REQUIRE(chunk >= 32, "gta_schedule_build: chunk must be >= 32");
  GTA_REQUIRE(row_end >= row_begin, "gta_schedule_build: negative row range");
  const int64_t rows = row_end - row_begin;
  h_counts[0] = h_counts[1] = 0;
  if (h_block_begin)
    for (int32_t cb = 0; cb <= n_cb; ++cb) h_block_begin[cb] = 0;
  // no rows (a rank whose destination range is empty): no items, and the indices of its 0 edges may be NULL
  if (rows == 0) return GTA_OK;
  GTA_REQUIRE(n_cb == 1 || indices, "gta_schedule_build: column blocking needs the CSR indices");
  const size_t need = gta_schedule_workspace(rows, ws_sources, ws_col_block);
  if (workspace_bytes < need) {
    set_error("gta_schedule_build: workspace %zu < required %zu", workspace_bytes, need);
    return GTA_ERR_WORKSPACE;
  }
  const int64_t n = rows * n_cb + 1;
  const size_t nb = align_up(size_t(n) * 4, 256);
  const size_t rb = align_up(size_t(rows + 1) * 4, 256);
  char* base = static_cast<char*>(workspace);
  int32_t* counts = reinterpret_cast<int32_t*>(base);
  int32_t* item_off = reinterpret_cast<int32_t*>(base + nb);
  int32_t* slots_in = reinterpret_cast<int32_t*>(base + 2 * nb);
  void* cub_temp = base + 2 * nb + rb;
  size_t cub_bytes = workspace_bytes - (2 * nb + rb);
  // both scans run one entry past the end so the last output is the total
  GTA_CUDA(cudaMemsetAsync(counts + (n - 1), 0, 4, stream));
  GTA_CUDA(cudaMemsetAsync(slots_in + rows, 0, 4, stream));
  sched_count_kernel<<<sched_grid(rows), 256, 0, stream>>>(indptr, indices, row_begin, rows, chunk, ends, n_cb,
                                                          counts, slots_in);
  GTA_CHECK_LAUNCH("sched_count_kernel");
  GTA_CUDA(cub::DeviceScan::ExclusiveSum(cub_temp, cub_bytes, counts, item_off, n, stream));
  GTA_CUDA(cub::DeviceScan::ExclusiveSum(cub_temp, cub_bytes, slots_in, row_slots, rows + 1, stream));
  count_launch(4);
  int32_t totals[2];
  int32_t block_first[kMaxColBlocks];
  if (h_block_begin)
    for (int32_t cb = 0; cb < n_cb; ++cb)
      GTA_CUDA(cudaMemcpyAsync(&block_first[cb], item_off + int64_t(cb) * rows, 4, cudaMemcpyDeviceToHost, stream));
  GTA_CUDA(cudaMemcpyAsync(&totals[0], item_off + (n - 1), 4, cudaMemcpyDeviceToHost, stream));
  GTA_CUDA(cudaMemcpyAsync(&totals[1], row_slots + rows, 4, cudaMemcpyDeviceToHost, stream));
  GTA_CUDA(cudaStreamSynchronize(stream));
  if (int64_t(totals[0]) > items_capacity) {
    set_error("gta_schedule_build: %d items exceed capacity %lld", totals[0], (long long)items_capacity);
    return GTA_ERR_WORKSPACE;
  }
  sched_fill_kernel<<<sched_grid(rows), 256, 0, stream>>>(indptr, indices, row_begin, rows, chunk, ends, n_cb,
                                                         item_off, row_slots, reinterpret_cast<int4*>(items));
  GTA_CHECK_LAUNCH("sched_fill_kernel");
  h_counts[0] = totals[0];
  h_counts[1] = totals[1];
  if (h_block_begin) {
    for (int32_t cb = 0; cb < n_cb; ++cb) h_block_begin[cb] = block_first[cb];
    h_block_begin[n_cb] = totals[0];
  }
  return GTA_OK;
}

}  // extern "C"
