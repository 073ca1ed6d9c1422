// Device-side graph preprocessing: COO -> CSR, tile-nnz tables, partition bounds, degree
// reorder (the aggregation work list lives in schedule.cu).  Integer work, bit-exact against
// oracle/gta_oracle.py (csr_build / tile_nnz / partition_bounds / degree_reorder).
//
// The global radix sort and prefix sums call CUB (library code shipped with the CUDA
// toolkit); key packing, row-pointer extraction, histograms, searches and the work-list
// builder are kernels of this file.  All HBM-bound integer work: coalesced 8-byte
// streams, grids sized to cover the SMs several times over.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace gta {

static int bits_for(int64_t n) {
  int b = 1;
  while ((int64_t(1) << b) < n && b < 32) ++b;
  return b;
}

// ---- COO -> CSR ------------------------------------------------------------------------

// Ids outside the graph (dst not in [0, num_nodes), src < 0) would make unpack_rows_kernel write row pointers far
// out of bounds: they are counted in *bad and their key is clamped to row 0, and gta_csr_build reports
// GTA_ERR_INVALID instead of crashing on a damaged edge list.
__global__ void pack_keys_kernel(const int32_t* __restrict__ dst, const int32_t* __restrict__ src,
                                 int64_t n, int64_t num_nodes, uint64_t* __restrict__ keys, int64_t* __restrict__ vals,
                                 int32_t* __restrict__ bad) {
  int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) {
    int32_t d = dst[i], c = src[i];
    if (d < 0 || d >= num_nodes || c < 0) {
      atomicAdd(bad, 1);
      d = 0;
      c = 0;
    }
    keys[i] = (uint64_t(uint32_t(d)) << 32) | uint32_t(c);
    vals[i] = i;
  }
}

// sorted keys -> indices (low word) and row pointers (first position of every dst value)
__global__ void unpack_rows_kernel(const uint64_t* __restrict__ keys, int64_t n, int64_t num_nodes,
                                   int32_t* __restrict__ indices, int64_t* __restrict__ indptr) {
  int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  int64_t stride = int64_t(gridDim.x) * blockDim.x;
  if (i == 0 && n == 0) {
    for (int64_t r = 0; r <= num_nodes; ++r) indptr[r] = 0;
  }
  for (; i < n; i += stride) {
    uint64_t k = keys[i];
    int64_t d = int64_t(k >> 32);
    indices[i] = int32_t(uint32_t(k));
    int64_t prev = (i == 0) ? -1 : int64_t(keys[i - 1] >> 32);
    for (int64_t r = prev + 1; r <= d; ++r) indptr[r] = i;
    if (i == n - 1) {
      for (int64_t r = d + 1; r <= num_nodes; ++r) indptr[r] = n;
    }
  }
}

struct CsrWorkspace {
  uint64_t* keys_in;
  uint64_t* keys_out;
  int64_t* vals_in;
  int64_t* vals_out;
  void* cub_temp;
  size_t cub_bytes;
  int32_t* bad;       // count of edges whose ids are outside the graph
  size_t total;
};

static CsrWorkspace carve_csr(void* base, int64_t e, int64_t n) {
  CsrWorkspace w{};
  size_t cub_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (uint64_t*)nullptr, (uint64_t*)nullptr,
                                  (int64_t*)nullptr, (int64_t*)nullptr, e, 0, 32 + bits_for(n));
  size_t off = 0;
  char* b = static_cast<char*>(base);
  size_t ebytes = align_up(size_t(e > 0 ? e : 1) * 8, 256);
  w.keys_in = reinterpret_cast<uint64_t*>(b + off); off += ebytes;
  w.keys_out = reinterpret_cast<uint64_t*>(b + off); off += ebytes;
  w.vals_in = reinterpret_cast<int64_t*>(b + off); off += ebytes;
  w.vals_out = reinterpret_cast<int64_t*>(b + off); off += ebytes;
  w.cub_temp = b + off; off += align_up(cub_bytes, 256);
  w.cub_bytes = cub_bytes;
  w.bad = reinterpret_cast<int32_t*>(b + off); off += 256;
  w.total = off;
  return w;
}

// ---- tile nnz ----------------------------------------------------------------------------

// one warp per destination row of the requested tiles; counts[(tile - tile_begin)*N + src]++
__global__ void tile_nnz_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                int64_t num_nodes, int64_t tile_rows, int64_t tile_begin,
                                int64_t row_begin, int64_t row_end, int32_t* __restrict__ counts) {
  int64_t warp = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  int64_t nwarps = (int64_t(gridDim.x) * blockDim.x) >> 5;
  for (int64_t r = row_begin + warp; r < row_end; r += nwarps) {
    int64_t b = indptr[r], e = indptr[r + 1];
    int32_t* row_counts = counts + (r / tile_rows - tile_begin) * num_nodes;
    for (int64_t k = b + lane; k < e; k += 32) {
      int32_t c = indices[k];
      if (int64_t(c) != r) atomicAdd(row_counts + c, 1);   // self loops are zeroed (preprocessing.py:17)
    }
  }
}

__global__ void max_i32_kernel(const int32_t* __restrict__ v, int64_t n, int32_t* __restrict__ out) {
  int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  int64_t stride = int64_t(gridDim.x) * blockDim.x;
  int32_t m = 0;
  for (; i < n; i += stride) m = max(m, v[i]);
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(out, m);
}

// ---- partition ---------------------------------------------------------------------------

__global__ void partition_kernel(const int64_t* __restrict__ indptr, int64_t num_nodes, int32_t parts,
                                 int64_t* __restrict__ bounds) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > parts) return;
  if (k == 0) { bounds[0] = 0; return; }
  if (k == parts) { bounds[parts] = num_nodes; return; }
  int64_t e = indptr[num_nodes];
  int64_t target = (int64_t(k) * e) / parts;
  int64_t lo = 0, hi = num_nodes + 1;   // lower_bound over indptr[0..N]
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if (indptr[mid] < target) lo = mid + 1; else hi = mid;
  }
  bounds[k] = lo;
}

// ---- degree reorder ----------------------------------------------------------------------

__global__ void degree_keys_kernel(const int64_t* __restrict__ indptr, int64_t n, uint64_t* __restrict__ keys) {
  int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) {
    uint64_t deg = uint64_t(indptr[i + 1] - indptr[i]);
    keys[i] = ((0xFFFFFFFFull - deg) << 32) | uint64_t(uint32_t(i));   // descending degree, ascending id
  }
}

__global__ void low_word_kernel(const uint64_t* __restrict__ keys, int64_t n, int64_t* __restrict__ out) {
  int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) out[i] = int64_t(uint32_t(keys[i]));
}

// ---- source-id remap for destination-partitioned execution ---------------------------------
// The gathered source table of a rank is [parts, stride, F]: `parts` slots of `stride` rows (every
// rank's rows padded to `stride`).  Slot k of rank r holds the rows of rank (r + k) mod parts, so the
// rank's OWN rows are slot 0 and the work list -- ordered by column block = slot -- starts on data that
// needs no transfer, then walks the peers in ring order while their slots arrive (ipc.cu, aggregate.cu).
// Global source id j owned by rank p becomes ((p - rotate) mod parts)*stride + (j - bounds[p]).
// rotate = 0: p*stride + offset, monotonic in j (the layout of an NCCL all-gather).  rotate > 0 is a
// cyclic shift of every row's ascending source list: the caller re-sorts the rows by the new ids
// (a fixed, deterministic reduction order, but not the single-GPU one).
__global__ void remap_sources_kernel(const int32_t* __restrict__ in, int64_t n, const int64_t* __restrict__ bounds,
                                     int parts, int64_t stride, int rotate, int32_t* __restrict__ out) {
  int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  int64_t step = int64_t(gridDim.x) * blockDim.x;
  for (; i < n; i += step) {
    int64_t j = in[i];
    int lo = 0, hi = parts;            // largest p with bounds[p] <= j
    while (hi - lo > 1) {
      int mid = (lo + hi) >> 1;
      if (bounds[mid] <= j) lo = mid; else hi = mid;
    }
    const int slot = lo >= rotate ? lo - rotate : lo - rotate + parts;
    out[i] = int32_t(int64_t(slot) * stride + (j - bounds[lo]));
  }
}

static int grid_for(int64_t n, int block) {
  int64_t g = (n + block - 1) / block;
  int64_t cap = int64_t(kNumSMs) * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return int(g);
}

}  // namespace gta

using namespace gta;

extern "C" {

size_t gta_csr_build_workspace(int64_t num_edges, int64_t num_nodes) {
  return carve_csr(nullptr, num_edges, num_nodes).total;
}

int gta_csr_build(const int32_t* dst, const int32_t* src, int64_t num_edges, int64_t num_nodes,
                  int64_t* indptr, int32_t* indices, int64_t* perm, void* workspace,
                  size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  // num_nodes = 0 is the local graph of a rank whose destination range is empty: indptr = [0], and any edge names a
  // destination outside the graph, which the bad-id count below refuses
  GTA_REQUIRE(num_nodes >= 0 && num_nodes < (int64_t(1) << 31), "gta_csr_build: num_nodes out of range");
  GTA_REQUIRE(num_edges >= 0 && num_edges < (int64_t(1) << 31), "gta_csr_build: num_edges must be < 2^31");
  GTA_REQUIRE(indptr && (num_edges == 0 || (dst && src && indices)), "gta_csr_build: null pointer");
  CsrWorkspace w = carve_csr(workspace, num_edges, num_nodes);
  if (workspace == nullptr || workspace_bytes < w.total) {
    set_error("gta_csr_build: workspace %zu < required %zu", workspace_bytes, w.total);
    return GTA_ERR_WORKSPACE;
  }
  if (num_edges > 0) {
    GTA_CUDA(cudaMemsetAsync(w.bad, 0, sizeof(int32_t), stream));
    pack_keys_kernel<<<grid_for(num_edges, 256), 256, 0, stream>>>(dst, src, num_edges, num_nodes, w.keys_in, w.vals_in,
                                                                  w.bad);
    GTA_CHECK_LAUNCH("pack_keys_kernel");
    int64_t* vals_out = perm ? perm : w.vals_out;
    size_t cub_bytes = w.cub_bytes;
    GTA_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_temp, cub_bytes, w.keys_in, w.keys_out, w.vals_in, vals_out,
                                             num_edges, 0, 32 + bits_for(num_nodes), stream));
    count_launch(4);
  }
  unpack_rows_kernel<<<grid_for(num_edges, 256), 256, 0, stream>>>(w.keys_out, num_edges, num_nodes, indices, indptr);
  GTA_CHECK_LAUNCH("unpack_rows_kernel");
  if (num_edges > 0) {      // a set-up call: one small read-back so that a damaged edge list is an error, not a crash
    int32_t bad = 0;
    GTA_CUDA(cudaMemcpyAsync(&bad, w.bad, sizeof(bad), cudaMemcpyDeviceToHost, stream));
    GTA_CUDA(cudaStreamSynchronize(stream));
    GTA_REQUIRE(bad == 0, "gta_csr_build: %d edges name a destination outside [0, %lld) or a negative source", bad,
                (long long)num_nodes);
  }
  return GTA_OK;
}

int gta_tile_nnz(const int64_t* indptr, const int32_t* indices, int64_t num_nodes, int64_t tile_rows,
                 int64_t tile_begin, int64_t tile_end, int32_t* counts, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  GTA_REQUIRE(indptr && indices && counts, "gta_tile_nnz: null pointer");
  GTA_REQUIRE(tile_rows > 0 && num_nodes > 0, "gta_tile_nnz: tile_rows and num_nodes must be positive");
  int64_t tiles = ceil_div64(num_nodes, tile_rows);
  GTA_REQUIRE(0 <= tile_begin && tile_begin <= tile_end && tile_end <= tiles, "gta_tile_nnz: tile range outside [0,%lld]", (long long)tiles);
  if (tile_begin == tile_end) return GTA_OK;
  GTA_CUDA(cudaMemsetAsync(counts, 0, size_t(tile_end - tile_begin) * num_nodes * sizeof(int32_t), stream));
  int64_t row_begin = tile_begin * tile_rows;
  int64_t row_end = tile_end * tile_rows < num_nodes ? tile_end * tile_rows : num_nodes;
  int64_t rows = row_end - row_begin;
  tile_nnz_kernel<<<grid_for(rows * 32, 256), 256, 0, stream>>>(indptr, indices, num_nodes, tile_rows, tile_begin,
                                                                row_begin, row_end, counts);
  GTA_CHECK_LAUNCH("tile_nnz_kernel");
  return GTA_OK;
}

int gta_tile_nnz_max(const int64_t* indptr, const int32_t* indices, int64_t num_nodes, int64_t tile_rows,
                     void* workspace, size_t workspace_bytes, int32_t* h_max, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  GTA_REQUIRE(h_max && workspace, "gta_tile_nnz_max: null pointer");
  GTA_REQUIRE(tile_rows > 0 && num_nodes > 0, "gta_tile_nnz_max: tile_rows and num_nodes must be positive");
  if (workspace_bytes < 256 + size_t(num_nodes) * 4) {
    set_error("gta_tile_nnz_max: workspace %zu < %zu", workspace_bytes, 256 + size_t(num_nodes) * 4);
    return GTA_ERR_WORKSPACE;
  }
  int32_t* d_max = static_cast<int32_t*>(workspace);
  int32_t* table = reinterpret_cast<int32_t*>(static_cast<char*>(workspace) + 256);
  int64_t batch = int64_t((workspace_bytes - 256) / (size_t(num_nodes) * 4));
  int64_t tiles = ceil_div64(num_nodes, tile_rows);
  GTA_CUDA(cudaMemsetAsync(d_max, 0, sizeof(int32_t), stream));
  for (int64_t t = 0; t < tiles; t += batch) {
    int64_t te = t + batch < tiles ? t + batch : tiles;
    int rc = gta_tile_nnz(indptr, indices, num_nodes, tile_rows, t, te, table, stream_);
    if (rc != GTA_OK) return rc;
    int64_t n = (te - t) * num_nodes;
    max_i32_kernel<<<grid_for(n, 256), 256, 0, stream>>>(table, n, d_max);
    GTA_CHECK_LAUNCH("max_i32_kernel");
  }
  GTA_CUDA(cudaMemcpyAsync(h_max, d_max, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
  GTA_CUDA(cudaStreamSynchronize(stream));
  return GTA_OK;
}

int gta_partition(const int64_t* indptr, int64_t num_nodes, int32_t parts, int64_t* bounds, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  GTA_REQUIRE(indptr && bounds, "gta_partition: null pointer");
  GTA_REQUIRE(parts >= 1 && parts <= 65536, "gta_partition: parts must be in [1,65536]");
  partition_kernel<<<(parts + 1 + 127) / 128, 128, 0, stream>>>(indptr, num_nodes, parts, bounds);
  GTA_CHECK_LAUNCH("partition_kernel");
  return GTA_OK;
}

size_t gta_reorder_workspace(int64_t num_nodes) {
  size_t cub_bytes = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, cub_bytes, (uint64_t*)nullptr, (uint64_t*)nullptr, num_nodes, 0, 64);
  return 2 * align_up(size_t(num_nodes) * 8, 256) + align_up(cub_bytes, 256);
}

int gta_reorder(const int64_t* indptr, int64_t num_nodes, int64_t* perm, void* workspace,
                size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  GTA_REQUIRE(indptr && perm && workspace, "gta_reorder: null pointer");
  GTA_REQUIRE(num_nodes > 0 && num_nodes < (int64_t(1) << 31), "gta_reorder: num_nodes out of range");
  size_t need = gta_reorder_workspace(num_nodes);
  if (workspace_bytes < need) {
    set_error("gta_reorder: workspace %zu < required %zu", workspace_bytes, need);
    return GTA_ERR_WORKSPACE;
  }
  size_t nb = align_up(size_t(num_nodes) * 8, 256);
  uint64_t* keys_in = static_cast<uint64_t*>(workspace);
  uint64_t* keys_out = reinterpret_cast<uint64_t*>(static_cast<char*>(workspace) + nb);
  void* cub_temp = static_cast<char*>(workspace) + 2 * nb;
  size_t cub_bytes = workspace_bytes - 2 * nb;
  degree_keys_kernel<<<grid_for(num_nodes, 256), 256, 0, stream>>>(indptr, num_nodes, keys_in);
  GTA_CHECK_LAUNCH("degree_keys_kernel");
  GTA_CUDA(cub::DeviceRadixSort::SortKeys(cub_temp, cub_bytes, keys_in, keys_out, num_nodes, 0, 64, stream));
  count_launch(4);
  low_word_kernel<<<grid_for(num_nodes, 256), 256, 0, stream>>>(keys_out, num_nodes, perm);
  GTA_CHECK_LAUNCH("low_word_kernel");
  return GTA_OK;
}

int gta_remap_sources(const int32_t* indices, int64_t num_edges, const int64_t* bounds, int32_t parts,
                      int64_t stride, int32_t rotate, int32_t* out, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (num_edges == 0) return GTA_OK;
  GTA_REQUIRE(indices && bounds && out, "gta_remap_sources: null pointer");
  GTA_REQUIRE(parts >= 1 && stride >= 1 && int64_t(parts) * stride < (int64_t(1) << 31),
              "gta_remap_sources: parts*stride must fit int32");
  GTA_REQUIRE(rotate >= 0 && rotate < parts, "gta_remap_sources: rotate=%d outside [0, %d)", rotate, parts);
  remap_sources_kernel<<<grid_for(num_edges, 256), 256, 0, stream>>>(indices, num_edges, bounds, parts, stride, rotate, out);
  GTA_CHECK_LAUNCH("remap_sources_kernel");
  return GTA_OK;
}


}  // extern "C"
