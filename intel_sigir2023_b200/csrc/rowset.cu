// Row sets of the sparse embedding-table gradients (IntEL(sparse_grad=1), DESIGN.md section 6): the ascending unique
// in-range ids that one step's index tensors name, and a row -> slot map that the backward scatters write through
// (embed.cu, scatter_add_rows with a slot map), so a table's gradient is a compact [U, d] block instead of the table.
//
// The map is a caller-owned int32 array over the whole table that also serves as the mark array:
//   mark:    row_slot[id] = -1 for every in-range id of the step (plain stores, duplicates are harmless)
//   count:   per chunk of CHUNK rows, the number of marked rows
//   scan:    exclusive scan of the chunk counts (one CTA), total -> *count_out
//   write:   each marked row gets its rank among the marked rows: row_slot[r] = slot, rows_out[slot] = r
// After the write pass every entry is >= 0 again, so the next call starts from a valid state without a reset pass.
// The output order depends only on the set of ids, never on the order of the atomics-free passes: deterministic.
// Traffic: the ids once, the map twice (8 B per table row per step).
#include "kernels.h"
#include "../../include/intel_b200.h"

namespace intel {

static const int RS_THREADS = 256;
static const int RS_PER_THREAD = 16;
static const int64_t RS_CHUNK = (int64_t)RS_THREADS * RS_PER_THREAD;

__global__ void __launch_bounds__(256) rowset_mark_kernel(const int64_t* __restrict__ a, int64_t na,
                                                          const int64_t* __restrict__ b, int64_t nb, int64_t table_rows,
                                                          int32_t* row_slot) {
    const int64_t n = na + nb;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t id = e < na ? a[e] : b[e - na];
        if (id >= 0 && id < table_rows) row_slot[id] = -1;      // out-of-range ids: the dense scatter skips them too
    }
}

// number of marked rows among the RS_PER_THREAD consecutive rows of this thread
__device__ __forceinline__ int rowset_thread_count(const int32_t* row_slot, int64_t r0, int64_t table_rows) {
    int c = 0;
    for (int i = 0; i < RS_PER_THREAD; ++i) {
        const int64_t r = r0 + i;
        if (r < table_rows && row_slot[r] < 0) ++c;
    }
    return c;
}

// inclusive scan over the CTA's RS_THREADS values (Hillis-Steele in shared memory)
__device__ __forceinline__ int rowset_block_scan(int v, int* sh) {
    const int t = threadIdx.x;
    sh[t] = v;
    __syncthreads();
    for (int o = 1; o < RS_THREADS; o <<= 1) {
        const int add = t >= o ? sh[t - o] : 0;
        __syncthreads();
        sh[t] += add;
        __syncthreads();
    }
    const int r = sh[t];
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(256) rowset_count_kernel(const int32_t* __restrict__ row_slot, int64_t table_rows,
                                                           int32_t* chunk_count) {
    __shared__ int sh[RS_THREADS];
    const int64_t r0 = (int64_t)blockIdx.x * RS_CHUNK + (int64_t)threadIdx.x * RS_PER_THREAD;
    const int incl = rowset_block_scan(rowset_thread_count(row_slot, r0, table_rows), sh);
    if (threadIdx.x == RS_THREADS - 1) chunk_count[blockIdx.x] = incl;
}

// one CTA: chunk_count[0..n) -> exclusive prefix sums in place, the total to *count_out
__global__ void __launch_bounds__(1024) rowset_scan_kernel(int32_t* chunk_count, int64_t n, int64_t* count_out) {
    __shared__ int64_t sh[1024];
    const int t = threadIdx.x, T = blockDim.x;
    const int64_t per = (n + T - 1) / T, lo = t * per, hi = lo + per < n ? lo + per : n;
    int64_t own = 0;
    for (int64_t i = lo; i < hi; ++i) own += chunk_count[i];
    sh[t] = own;
    __syncthreads();
    for (int o = 1; o < T; o <<= 1) {
        const int64_t add = t >= o ? sh[t - o] : 0;
        __syncthreads();
        sh[t] += add;
        __syncthreads();
    }
    int64_t run = sh[t] - own;
    for (int64_t i = lo; i < hi; ++i) {
        const int64_t c = chunk_count[i];
        chunk_count[i] = (int32_t)run;
        run += c;
    }
    if (t == T - 1) *count_out = sh[t];
}

__global__ void __launch_bounds__(256) rowset_write_kernel(int32_t* row_slot, int64_t table_rows,
                                                           const int32_t* __restrict__ chunk_base, int64_t* rows_out) {
    __shared__ int sh[RS_THREADS];
    const int64_t r0 = (int64_t)blockIdx.x * RS_CHUNK + (int64_t)threadIdx.x * RS_PER_THREAD;
    const int own = rowset_thread_count(row_slot, r0, table_rows);
    int slot = chunk_base[blockIdx.x] + rowset_block_scan(own, sh) - own;
    for (int i = 0; i < RS_PER_THREAD; ++i) {
        const int64_t r = r0 + i;
        if (r < table_rows && row_slot[r] < 0) {
            row_slot[r] = slot;
            rows_out[slot] = r;
            ++slot;
        }
    }
}

size_t rowset_workspace_bytes(int64_t table_rows) {
    return (size_t)(table_rows > 0 ? ceil_div(table_rows, RS_CHUNK) : 1) * sizeof(int32_t) + 256;
}

int rowset_build(int64_t table_rows, const int64_t* a, int64_t na, const int64_t* b, int64_t nb, int32_t* row_slot,
                 int64_t* rows_out, int64_t* count_out, void* ws, size_t ws_bytes, cudaStream_t s) {
    INTEL_REQUIRE(table_rows > 0 && table_rows < ((int64_t)1 << 31), INTEL_ERR_ARG, "rowset: table rows must be in [1, 2^31)");
    INTEL_REQUIRE(na >= 0 && nb >= 0 && (a || na == 0) && (b || nb == 0), INTEL_ERR_ARG, "rowset: bad id arrays");
    INTEL_REQUIRE(row_slot && rows_out && count_out, INTEL_ERR_ARG, "rowset: null output");
    const int64_t chunks = ceil_div(table_rows, RS_CHUNK);
    INTEL_REQUIRE(ws && ws_bytes >= rowset_workspace_bytes(table_rows), INTEL_ERR_WORKSPACE, "rowset workspace too small: need %zu",
                  rowset_workspace_bytes(table_rows));
    int32_t* chunk = reinterpret_cast<int32_t*>(ws);
    if (na + nb > 0) {
        LAUNCH(rowset_mark_kernel, dim3(stream_grid(ceil_div(na + nb, 256), 8)), dim3(256), 0, s, a, na, b, nb, table_rows, row_slot);
        INTEL_TRY(check_launch("rowset_mark", 12.0 * (double)(na + nb), 0.0));
    }
    LAUNCH(rowset_count_kernel, dim3((unsigned)chunks), dim3(RS_THREADS), 0, s, row_slot, table_rows, chunk);
    INTEL_TRY(check_launch("rowset_count", 4.0 * (double)table_rows, 0.0));
    LAUNCH(rowset_scan_kernel, dim3(1), dim3(1024), 0, s, chunk, chunks, count_out);
    INTEL_TRY(check_launch("rowset_scan", 8.0 * (double)chunks, 0.0));
    LAUNCH(rowset_write_kernel, dim3((unsigned)chunks), dim3(RS_THREADS), 0, s, row_slot, table_rows, chunk, rows_out);
    return check_launch("rowset_write", 4.0 * (double)table_rows, 0.0);
}

}  // namespace intel

using namespace intel;

size_t intel_rowset_workspace_bytes(int64_t table_rows) { return rowset_workspace_bytes(table_rows); }

int intel_rowset_build(int64_t table_rows, const int64_t* ids_a, int64_t n_a, const int64_t* ids_b, int64_t n_b,
                       int32_t* row_slot, int64_t* rows_out, int64_t* count_out, void* workspace, size_t workspace_bytes,
                       intel_stream_t stream) {
    return rowset_build(table_rows, ids_a, n_a, ids_b, n_b, row_slot, rows_out, count_out, workspace, workspace_bytes,
                        (cudaStream_t)stream);
}
