// sketch_core.cuh -- internal interface between sketch.cu and screen.cu
#pragma once
#include "common.cuh"

namespace mashgpu {

// A device-resident byte stream split into sketch units.
struct SketchStream {
    const void *d_stream = nullptr;         // ASCII source, or
    const uint64_t *d_codes = nullptr;      // packed source: 2-bit codes (32 positions per word) ...
    const uint32_t *d_inval = nullptr;      // ... and the invalid-position bit mask (see pack.cpp)
    const uint64_t *unit_start = nullptr;   // host, n_units + 1
    uint64_t n_units = 0;
    cudaEvent_t data_ready = nullptr;       // when set: the scan kernel waits for this event (an upload on another stream); the parameter
                                            // copies of the pass are enqueued before the wait -- they come from pageable memory and would
                                            // otherwise hold the calling thread until the upload has finished
    bool t_cap = false;                     // clamp every unit threshold to t_cap_value (screen: running s-th smallest)
    uint64_t t_cap_value = 0;
};

// Reference hash table of a screen job (distinct keys + hit counters)
struct ScreenProbe {
    const uint64_t *keys;
    const uint32_t *idx;
    uint32_t *cnt;
    uint32_t log2cap;
    uint64_t hmax;
    const uint32_t *bitmap;     // value-indexed presence bitmap over the reference hashes (NULL: none), see scan.cuh
    uint32_t bitmap_shift;
};

// One sketch_stream pass in flight: the kernels are enqueued by sketch_stream_enqueue and the per-unit status flags come back
// into pinned memory; sketch_stream_finalize waits for them and re-runs flagged units exactly.  The stream data, the output
// buffers and the context's scratch must stay untouched between the two calls (one ticket in flight per context).
struct SketchTicket {
    bool active = false;
    mashgpu_sketch_params params{};
    SketchStream S;
    std::vector<uint64_t> unit_start;       // own copy of S.unit_start
    uint64_t *d_out_hashes = nullptr; uint32_t *d_out_counts = nullptr, *d_out_n = nullptr;
    cudaStream_t st = nullptr;
    uint32_t min_copies = 1;                // `-m` of the tables (1 for the screen mixture), the same in the re-runs
    uint64_t *d_qtarget = nullptr, *d_qtstar = nullptr;
};

int validate_sketch_params(mashgpu_ctx *ctx, const mashgpu_sketch_params *p);
bool is_dna_alphabet(const mashgpu_sketch_params *p);
int sketch_stream_core(mashgpu_ctx *ctx, const mashgpu_sketch_params *p, const SketchStream &S,
                       uint64_t *d_out_hashes, uint32_t *d_out_counts, uint32_t *d_out_n, cudaStream_t st,
                       const ScreenProbe *probe);
int sketch_stream_enqueue(mashgpu_ctx *ctx, const mashgpu_sketch_params *p, const SketchStream &S,
                          uint64_t *d_out_hashes, uint32_t *d_out_counts, uint32_t *d_out_n, cudaStream_t st,
                          const ScreenProbe *probe, SketchTicket &t);
int sketch_stream_finalize(mashgpu_ctx *ctx, SketchTicket &t);

}  // namespace mashgpu
