// Host-side solver for centroid-linkage agglomerative clustering on one B200 (see ahc_kernels.cu).
#pragma once

#include "ahc_core.cuh"
#include <cuda_runtime.h>
#include <vector>

namespace fa {
namespace ahc {

// Master -> workers: ONE 64-bit word, written with st.release and polled with ld.acquire (8-byte accesses are
// single-copy atomic, so sequence tag and payload can never tear):
//   [63:62] type (1 MERGE a,b | 2 RESCAN for node a | 3 EXIT)   [61:48] command counter mod 2^14
//   [47:24] node id a                                           [23:0]  node id b
// The id of a freshly merged node is implicit (N + number of MERGE commands so far).  Workers find the slots of
// a and b themselves (every thread knows which node its slot holds) and read member counts from node_weight[].
// Workers -> master: two self-validating 64-bit words per worker CTA (no atomic counter, no second round trip):
//   w0 = [63:32] high half of the distance bits | [31:8] node id (0xFFFFFE = NaN seen, 0xFFFFFF = none) | [7:0] counter
//   w1 = [63:32] low half of the distance bits  | [31:0] counter                       (written with st.release)
// The master polls both words of all its slots with relaxed loads until every word carries the current command
// counter; the fence inside its next st.release completes the acquire side of the workers' releases.
struct ResultSlot {
    unsigned long long w0;
    unsigned long long w1;
};

// Everything the persistent kernel needs, resident in HBM.
struct Problem {
    int N, D, Ns;            // points, dimension, slot stride (N rounded up to 32)
    double *rows;            // [(2N-1) x D] node store, row-major: rows 0..N-1 = input, N.. = merged centroids
    double *cols;            // [D x Ns]     scan copy, k-major: cols[k*Ns + slot]
    int *node_weight;        // [2N-1] member count per node id (written by the CTA that creates the node)
    // master state, slot-indexed; staged into shared memory when it fits (idx16 != 0)
    double *key;             // [N]   nearest-neighbour squared distance of the node in each slot (heap keys)
    int *nn;                 // [N]   nearest neighbour (node id) of the node in each slot
    void *heap_at;           // [N-1] heap position -> slot   (uint16_t if idx16 else int)
    void *heap_where;        // [N]   slot -> heap position
    int *node_of;            // [N]   node id held by each slot (-1 when empty)
    int *slot_of;            // [2N-1] slot of each node id
    unsigned *live_bits;     // [(2N-1+31)/32]
    int *merge_a, *merge_b;  // [N-1] merge log
    double *merge_d;         // [N-1] squared distance of each merge
    // synchronisation
    unsigned long long *cmd;        // explicit command word (master -> workers)
    unsigned long long *threshold;  // [2 parities][2 words] per-round self-issue threshold (master -> workers)
    ResultSlot *results;     // [2][result_stride]: per-CTA candidates, double-buffered by scan-round parity
    int result_stride;       // slots between the two parities
    int slot_shift;          // log2 of the distance (in slots) between two CTAs' candidates
    int *error;              // 0 ok, 1 NaN distance (host-visible copy)
    int heap_size;           // after host heapify
    int idx16;               // heap index arrays are uint16_t and the master state lives in shared memory
    int smem_level;          // how much master state fits in smem: 1 = heap, 2 = + nn, 3 = + node_of
    unsigned long long *trace;   // [kTraceSteps x 8] globaltimer stamps (flags bit 2), diagnostics only
    int flags;               // bit 2: globaltimer trace; bit 3: never self-issue (every merge waits for the master)
    int resident;            // 1: every worker keeps its nodes' vectors in shared memory; 0: streamed from `cols`
    int slots_per_cta;       // resident mode: slots [w*slots_per_cta, (w+1)*slots_per_cta) belong to worker w
};

constexpr int kTraceSteps = 256;

struct Solver {
    int num_sms = 0;
    int max_workers = 0;      // worker CTAs available for one problem (grid = workers + 1)
    long long launches = 0;
    cudaStream_t stream = nullptr;
    // device storage (grown on demand, reused across calls)
    void *d_pool = nullptr;
    size_t pool_bytes = 0;
    Problem *d_problem = nullptr;
    double *d_input = nullptr;   // staging of the caller's [N x D] rows when they come from the host
    size_t input_cap = 0;
    // pinned host mirrors
    void *h_pool = nullptr;
    size_t h_pool_bytes = 0;
    float last_ms[4] = {0, 0, 0, 0};
    double trace_avg_ns[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // mean offsets from "command published" (flags bit 2)   // init-nn, host heapify + copies, merge loop, total

    ~Solver();
    void release();
    int init(cudaStream_t s, int worker_limit);
    // rows: device pointer to N x D row-major doubles (already normalised by the caller, as the reference requires).
    // Z: host buffer of (N-1) x 4 doubles.  Status codes follow FastClusterWrapper.h.
    int linkage_device(const double *d_rows, int N, int D, double *Z_host);
    int linkage_host(const double *rows_host, size_t N, size_t D, double *Z_host, size_t z_len);
    int ensure_pool(int N, int D);
};

// [0] initial nearest-neighbour kernels, [1] heapify + copies, [2] merge kernel, [3] total (ms) of the calling
// thread's most recent linkage
const float *last_stage_ms();
// placement of the calling thread's most recent linkage (layout: fa_ahc_last_placement in fluidaudio_b200.h)
enum { kInitExact = 0, kInitFilterRows = 1, kInitFilterTiles = 2, kInitFilterFellBack = 3 };
const int *last_placement();

// Standalone kernels used by the clustering pipeline
int launch_normalize_rows(const double *d_in, double *d_out, int rows, int dim, cudaStream_t s);
int resident_workers_needed(int N, int D);   // worker CTAs for the shared-memory-resident placement (0: impossible)
int launch_normalize_rows_keep(const double *d_in, double *d_out, int rows, int dim, cudaStream_t s);   // zero rows kept
int launch_widen_rows(const float *d_in, double *d_out, long long count, cudaStream_t s);

// Swift-side dendrogram cut + first-appearance relabel (AHCClustering.swift:112-121,124-210), host, O(N).
void dendrogram_cut(const double *Z, long long count, double threshold, int32_t *labels);

} // namespace ahc
} // namespace fa
