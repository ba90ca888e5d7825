// sketch.cu -- hot path 1: batched bottom-s sketching on the GPU (C-ABI: mashgpu_sketch_*, mashgpu_hash_windows).
//
// Pipeline per batch (see DESIGN.md):
//   flat byte stream in HBM  ->  scan_kernel (scan.cuh): hash every valid canonical k-mer, keep hash <= T_unit
//   in the unit's open-addressing table (distinct keys + multiplicities)  ->  select_kernel: compact the table,
//   sort, emit the s smallest.  This replaces MinHashHeap::tryInsert / HashSet::toHashList
//   (reference MinHashHeap.cpp:68-146, HashSet.cpp:78-118): bottom-s of a set does not depend on insertion order.
//   T_unit is chosen so that ~SURVIVOR_FACTOR*s distinct hashes are expected; a unit that ends with fewer than s
//   distinct survivors (while k-mers were dropped) or overflows its table is re-run exactly with a larger T.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_segmented_radix_sort.cuh>

#include "common.cuh"
#include "scan.cuh"
#include "sketch_core.cuh"
#include "pack.h"
#include <chrono>
#include <condition_variable>
#include <future>
#include <mutex>
#include <thread>
#include <cstdlib>

namespace mashgpu {

scan_launch_fn get_scan_launcher_part0(int, bool, bool);
scan_launch_fn get_scan_launcher_part1(int, bool, bool);
scan_launch_fn get_scan_launcher_part2(int, bool, bool);
scan_launch_fn get_scan_launcher_part3(int, bool, bool);

scan_launch_fn get_bytes_launcher_part0(int);
scan_launch_fn get_bytes_launcher_part1(int);
scan_launch_fn get_bytes_launcher_part2(int);
scan_launch_fn get_bytes_launcher_part3(int);

scan_launch_fn get_bytes_launcher(int k)
{
    if (auto f = get_bytes_launcher_part0(k)) return f;
    if (auto f = get_bytes_launcher_part1(k)) return f;
    if (auto f = get_bytes_launcher_part2(k)) return f;
    return get_bytes_launcher_part3(k);
}

scan_launch_fn get_scan_launcher(int k, bool canonical, bool packed)
{
    if (auto f = get_scan_launcher_part0(k, canonical, packed)) return f;
    if (auto f = get_scan_launcher_part1(k, canonical, packed)) return f;
    if (auto f = get_scan_launcher_part2(k, canonical, packed)) return f;
    return get_scan_launcher_part3(k, canonical, packed);
}

constexpr double SURVIVOR_FACTOR = 3.0;   // expected distinct survivors = 3 s
constexpr double TABLE_SLACK = 2.7;       // table slots per expected survivor
constexpr uint32_t SEL_MAX_LOG2 = 14;     // select_kernel sorts up to 2^14 keys in shared memory (128 KB)
constexpr int SEL_THREADS = 256;

// ---------------------------------------------------------------------------------------------------------
// per-tile coarse threshold: max T over the units a tile touches
// ---------------------------------------------------------------------------------------------------------
__global__ void tile_tmax_kernel(const uint64_t *unit_start, uint32_t n_units, const uint64_t *unit_t,
                                 uint64_t stream_len, uint64_t tile_begin, uint64_t tile_end, uint64_t *tile_tmax)
{
    uint64_t tile = tile_begin + blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (tile >= tile_end) return;
    uint64_t first = tile * (uint64_t)SCAN_TILE;
    uint64_t last = first + SCAN_TILE - 1;
    if (last >= stream_len) last = stream_len ? stream_len - 1 : 0;
    uint32_t lo = 0, hi = n_units;
    while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (unit_start[mid] <= first) lo = mid; else hi = mid; }
    uint64_t t = 0;
    for (uint32_t u = lo; u < n_units && unit_start[u] <= last; u++) t = max(t, unit_t[u]);
    tile_tmax[tile] = t;
}

// ---------------------------------------------------------------------------------------------------------
// select: table -> ascending bottom-s (+ counts)
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t table_count(const uint64_t *keys, const uint32_t *cnt, uint32_t log2cap, uint64_t key)
{
    const uint32_t mask = (1u << log2cap) - 1;
    uint32_t slot = slot_hash(key, log2cap);
    for (;;) {
        uint64_t k = keys[slot];
        if (k == key) return cnt[slot];
        if (k == EMPTY_KEY) return 0;
        slot = (slot + 1) & mask;
    }
}

// One CTA per unit; tables up to 2^SEL_MAX_LOG2 slots.  flags bit1 = fewer than s distinct survivors although
// k-mers were filtered (unit_t != max); units whose table is too large for shared memory are left to the batched
// segmented sort below (large sketch sizes: `-s 10000` needs ~2^17 candidate slots per unit).
__global__ void __launch_bounds__(SEL_THREADS) select_kernel(
    uint32_t unit_begin, uint32_t n_units, const uint64_t *unit_t, const uint64_t *tab_off, const uint32_t *tab_log2,
    const uint64_t *tab_keys, const uint32_t *tab_cnt, const uint32_t *unit_maxhash, uint32_t *unit_flags,
    uint32_t s, uint64_t capped_t, uint64_t *out_hashes, uint32_t *out_counts, uint32_t *out_n, uint32_t min_copies)
{
    extern __shared__ uint64_t sk[];
    __shared__ uint32_t n_s;
    const uint32_t u = unit_begin + blockIdx.x;
    if (u >= unit_begin + n_units) return;
    const uint32_t log2cap = tab_log2[u];
    if (unit_flags[u] & 1u) return;                    // overflowed: will be re-run
    if (log2cap > SEL_MAX_LOG2) return;              // tables beyond the shared-memory sort: batched segmented sort (select_big_*)
    const uint32_t cap = 1u << log2cap;
    const uint64_t *keys = tab_keys + tab_off[u];
    const uint32_t *cnt = tab_cnt + tab_off[u];
    if (threadIdx.x == 0) n_s = 0;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < cap; i += SEL_THREADS) {
        uint64_t k = keys[i];
        if (k != EMPTY_KEY && cnt[i] >= min_copies) sk[atomicAdd(&n_s, 1u)] = k;      // `-m`: only hashes seen at least m times qualify
    }
    __syncthreads();
    const uint32_t n = n_s;
    uint32_t N = 2;
    while (N < n) N <<= 1;
    for (uint32_t i = n + threadIdx.x; i < N; i += SEL_THREADS) sk[i] = EMPTY_KEY;
    __syncthreads();
    for (uint32_t size = 2; size <= N; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t t = threadIdx.x; t < N / 2; t += SEL_THREADS) {
                uint32_t lo = 2 * t - (t & (stride - 1));
                uint32_t hi = lo + stride;
                bool up = (lo & size) == 0;
                uint64_t a = sk[lo], b = sk[hi];
                if ((a > b) == up) { sk[lo] = b; sk[hi] = a; }
            }
            __syncthreads();
        }
    }
    const uint32_t n_max = (unit_maxhash[u] && unit_maxhash[u] >= min_copies) ? 1u : 0u;          // the value 2^64-1 itself, largest possible
    const uint32_t total = n + n_max;
    const uint32_t m = total < s ? total : s;
    if (threadIdx.x == 0) {
        out_n[u] = m;
        // too few survivors although k-mers were dropped -- unless the threshold is the caller's cap (screen: the
        // running s-th smallest of the mixture; nothing above it can enter the bottom-s)
        if (total < s && unit_t[u] != EMPTY_KEY && unit_t[u] != capped_t) atomicOr(&unit_flags[u], 2u);
    }
    for (uint32_t i = threadIdx.x; i < m; i += SEL_THREADS) {
        uint64_t key = i < n ? sk[i] : EMPTY_KEY;
        out_hashes[(uint64_t)u * s + i] = key;
        if (out_counts) out_counts[(uint64_t)u * s + i] = i < n ? table_count(keys, cnt, log2cap, key) : unit_maxhash[u];
    }
}

// ---- big tables: compact the qualifying keys of every big unit into one buffer (segment b = unit big_units[b]), sort all
// segments with one segmented radix sort, emit the first s of each.  Same outputs and flags as select_kernel.
__global__ void select_big_compact_kernel(const uint32_t *big_units, uint32_t n_big, const uint64_t *seg_off, const uint64_t *tab_off, const uint32_t *tab_log2,
                                          const uint64_t *tab_keys, const uint32_t *tab_cnt, const uint32_t *unit_flags, uint32_t min_copies,
                                          uint64_t *comp, uint32_t *seg_n)
{
    const uint32_t b = blockIdx.y;
    if (b >= n_big) return;
    const uint32_t u = big_units[b];
    if (unit_flags[u] & 1u) return;                    // overflowed: will be re-run
    const uint64_t cap = 1ull << tab_log2[u];
    const uint64_t *keys = tab_keys + tab_off[u];
    const uint32_t *cnt = tab_cnt + tab_off[u];
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < cap; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[i];
        if (k != EMPTY_KEY && cnt[i] >= min_copies) comp[seg_off[b] + atomicAdd(&seg_n[b], 1u)] = k;
    }
}

__global__ void select_big_bounds_kernel(const uint64_t *seg_off, const uint32_t *seg_n, uint32_t n_big, long long *seg_begin, long long *seg_end)
{
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_big) return;
    seg_begin[b] = (long long)seg_off[b];
    seg_end[b] = (long long)(seg_off[b] + seg_n[b]);
}

__global__ void __launch_bounds__(SEL_THREADS) select_big_emit_kernel(
    const uint32_t *big_units, uint32_t n_big, const uint64_t *seg_off, const uint32_t *seg_n, const uint64_t *sorted,
    const uint64_t *unit_t, const uint64_t *tab_off, const uint32_t *tab_log2, const uint64_t *tab_keys, const uint32_t *tab_cnt,
    const uint32_t *unit_maxhash, uint32_t *unit_flags, uint32_t s, uint64_t capped_t, uint64_t *out_hashes, uint32_t *out_counts, uint32_t *out_n,
    uint32_t min_copies)
{
    const uint32_t b = blockIdx.x;
    if (b >= n_big) return;
    const uint32_t u = big_units[b];
    if (unit_flags[u] & 1u) return;
    const uint32_t n = seg_n[b];
    const uint32_t n_max = (unit_maxhash[u] && unit_maxhash[u] >= min_copies) ? 1u : 0u;
    const uint64_t total = (uint64_t)n + n_max;
    const uint32_t m = (uint32_t)(total < s ? total : s);
    if (threadIdx.x == 0) {
        out_n[u] = m;
        if (total < s && unit_t[u] != EMPTY_KEY && unit_t[u] != capped_t) atomicOr(&unit_flags[u], 2u);
    }
    const uint64_t *keys = tab_keys + tab_off[u];
    const uint32_t *cnt = tab_cnt + tab_off[u];
    for (uint32_t i = threadIdx.x; i < m; i += SEL_THREADS) {
        const uint64_t key = i < n ? sorted[seg_off[b] + i] : EMPTY_KEY;
        out_hashes[(uint64_t)u * s + i] = key;
        if (out_counts) out_counts[(uint64_t)u * s + i] = i < n ? table_count(keys, cnt, tab_log2[u], key) : unit_maxhash[u];
    }
}

__device__ __forceinline__ int64_t table_find(const uint64_t *keys, uint32_t log2cap, uint64_t key)
{
    const uint32_t mask = (1u << log2cap) - 1;
    uint32_t slot = slot_hash(key, log2cap);
    for (;;) {
        uint64_t k = keys[slot];
        if (k == key) return slot;
        if (k == EMPTY_KEY) return -1;
        slot = (slot + 1) & mask;
    }
}

// Multiplicity counts, the reference's way.  MinHashHeap::tryInsert (MinHashHeap.cpp:68-74) only accepts a hash when
// the heap is not full or the hash is strictly below the current top, so once all s final hashes have been seen
// (stream position t* = the latest first occurrence among them) further occurrences of the largest final hash are
// neither inserted nor counted; every other count is the true multiplicity (SURVEY.md 8 a5).
// One CTA per full sketch: t* by max-reduction, then count[last] = occurrences of the largest hash at positions <= t*:
// equal to the table count if its last occurrence is <= t*, 1 if it was the last hash to arrive, otherwise the unit
// is flagged (bit 3) for a targeted recount over [unit start, t*].
__global__ void __launch_bounds__(SEL_THREADS) quirk_kernel(
    uint32_t unit_begin, uint32_t n_units, uint32_t s, const uint64_t *out_hashes, uint32_t *out_counts, const uint32_t *out_n,
    const uint64_t *tab_off, const uint32_t *tab_log2, const uint64_t *tab_keys, const uint32_t *tab_cnt,
    const uint64_t *tab_first, const uint64_t *tab_last, uint32_t *unit_flags, uint64_t *quirk_target, uint64_t *quirk_tstar, uint32_t m)
{
    // m = multiplicityMinimum: a hash is promoted into the heap at its m-th occurrence (tab_first level m-1) holding count m
    __shared__ unsigned long long tstar_s;
    const uint32_t u = unit_begin + blockIdx.x;
    if (u >= unit_begin + n_units) return;
    if (unit_flags[u] & 7u) return;                 // will be re-run
    if (out_n[u] < s) return;                       // heap never full: every count is exact
    const uint64_t *keys = tab_keys + tab_off[u];
    const uint32_t lg = tab_log2[u];
    if (threadIdx.x == 0) tstar_s = 0;
    __syncthreads();
    unsigned long long local = 0;
    for (uint32_t i = threadIdx.x; i < s; i += SEL_THREADS) {
        int64_t slot = table_find(keys, lg, out_hashes[(uint64_t)u * s + i]);
        if (slot >= 0) local = max(local, (unsigned long long)tab_first[(tab_off[u] + slot) * m + (m - 1)]);
    }
    atomicMax(&tstar_s, local);
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint64_t tstar = tstar_s;
        const uint64_t key = out_hashes[(uint64_t)u * s + s - 1];
        int64_t slot = table_find(keys, lg, key);
        if (slot >= 0) {
            const uint32_t c = tab_cnt[tab_off[u] + slot];
            const uint64_t f = tab_first[(tab_off[u] + slot) * m + (m - 1)], l = tab_last[tab_off[u] + slot];
            if (c > m && l > tstar) {
                if (f == tstar) out_counts[(uint64_t)u * s + s - 1] = m;
                else { quirk_target[u] = key; quirk_tstar[u] = tstar; atomicOr(&unit_flags[u], 8u); }
            }
        }
    }
}

// Packed source: expand the host's list of invalid runs into the 1-bit-per-position mask.  One warp per run; runs
// are disjoint, so interior words are plain stores and only the two edge words need atomics.
// record separators of the directly copied records of a wave (one launch instead of one 1-byte memset per record)
__global__ void write_separators_kernel(uint8_t *stream, const uint64_t *offsets, uint32_t n)
{
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) stream[offsets[t]] = 0;
}

__global__ void apply_runs_kernel(const PackRun *runs, uint64_t n_runs, uint32_t *mask)
{
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5, n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (uint64_t r = warp; r < n_runs; r += n_warps) {
        const uint64_t start = runs[r].start, end = start + runs[r].len;      // [start, end)
        if (end == start) continue;
        const uint64_t w0 = start >> 5, w1 = (end - 1) >> 5;
        const uint32_t first = 0xFFFFFFFFu << (start & 31), last = 0xFFFFFFFFu >> (31 - ((end - 1) & 31));
        if (w0 == w1) { if (lane == 0) atomicOr(&mask[w0], first & last); continue; }
        if (lane == 0) atomicOr(&mask[w0], first);
        if (lane == 1) atomicOr(&mask[w1], last);
        for (uint64_t w = w0 + 1 + lane; w < w1; w += 32) mask[w] = 0xFFFFFFFFu;
    }
}

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
static int alphabet_size(const mashgpu_sketch_params *p)
{
    int n = 0;
    for (int i = 0; i < 256; i++) n += p->alphabet[i] != 0;
    return n;
}

bool is_dna_alphabet(const mashgpu_sketch_params *p)
{
    return alphabet_size(p) == 4 && p->alphabet['A'] && p->alphabet['C'] && p->alphabet['G'] && p->alphabet['T'];
}

static double kmer_space_of(const mashgpu_sketch_params *p)
{
    return std::pow((double)alphabet_size(p), (double)p->kmer_size);
}

int validate_sketch_params(mashgpu_ctx *ctx, const mashgpu_sketch_params *p)
{
    if (!p) return fail(ctx, MASHGPU_ERR_INVALID, "params is NULL");
    if (p->kmer_size < 1 || p->kmer_size > 32) return fail(ctx, MASHGPU_ERR_INVALID, "kmer_size %d outside 1..32", p->kmer_size);
    if (p->sketch_size < 1) return fail(ctx, MASHGPU_ERR_INVALID, "sketch_size must be >= 1");
    const int n = alphabet_size(p);
    if (n == 0) return fail(ctx, MASHGPU_ERR_INVALID, "empty alphabet");
    if ((p->use64 != 0) != (kmer_space_of(p) > std::pow(2.0, 32.0)))
        return fail(ctx, MASHGPU_ERR_INVALID, "use64=%d contradicts the reference rule alphabetSize^k > 2^32 for k=%d, %d letters (Sketch.cpp:1136)", p->use64, p->kmer_size, n);
    if (p->alphabet[0]) return fail(ctx, MASHGPU_ERR_INVALID, "byte 0 cannot be an alphabet letter");
    if (p->min_copies > 255) return fail(ctx, MASHGPU_ERR_UNSUPPORTED, "min_copies (-m) above 255");
    if (!is_dna_alphabet(p) && !p->noncanonical)
        return fail(ctx, MASHGPU_ERR_UNSUPPORTED,
                    "canonical k-mers are only defined for the alphabet {A,C,G,T}; other alphabets must be non-canonical "
                    "(the reference forces -n for -a / -z, sketchParameterSetup.cpp:79-95)");
    return MASHGPU_OK;
}

// Threshold / table geometry of one unit. factor = expected-survivor multiple of s.
void plan_unit(const mashgpu_sketch_params *p, uint64_t span, double factor, uint64_t *t_out, uint32_t *log2_out)
{
    const double hash_space = p->use64 ? 18446744073709551616.0 : 4294967296.0;
    double kspace = kmer_space_of(p);
    double distinct_max = std::min((double)span, kspace);          // upper bound on distinct hashes
    double expect = factor * (double)p->sketch_size;
    if (expect >= (double)span * 0.5 || expect >= kspace * 0.25) {
        *t_out = EMPTY_KEY;                                            // keep all
        *log2_out = std::max(4u, ceil_log2((uint64_t)(2.0 * distinct_max) + 2));
        return;
    }
    double frac = expect / (double)span;
    double t = frac * hash_space;
    *t_out = t >= 18446744073709549568.0 ? (EMPTY_KEY - 1) : (uint64_t)t;
    *log2_out = std::max(4u, ceil_log2((uint64_t)(TABLE_SLACK * expect) + 2));
}

// Scan arguments of a pass over a stream (ASCII, or packed codes + invalid mask): the source and the hash parameters
static ScanArgs scan_args(const mashgpu_sketch_params *p, const void *stream, const uint64_t *codes, const uint32_t *inval, uint64_t stream_len)
{
    ScanArgs a;
    memset(&a, 0, sizeof a);
    a.stream = (const uint8_t *)stream;
    a.codes = codes;
    a.inval = inval;
    a.stream_len = stream_len;
    a.seed = p->seed;
    a.use64 = p->use64;
    a.preserve_case = p->preserve_case;
    for (int b = 0; b < 256; b++) {
        int u = (!p->preserve_case && b > 96 && b < 123) ? b - 32 : b;     // reference Sketch.cpp:524-530
        a.byte_lut[b] = p->alphabet[u] ? (uint8_t)u : 0;
    }
    a.only_unit = -1;
    return a;
}

static int launch_scan(mashgpu_ctx *ctx, const mashgpu_sketch_params *p, const ScanArgs &a, cudaStream_t st)
{
    const bool dna = is_dna_alphabet(p);
    if (!dna && !a.stream) return fail(ctx, MASHGPU_ERR_UNSUPPORTED, "the packed source only carries the alphabet {A,C,G,T}");
    scan_launch_fn fn = dna ? get_scan_launcher(p->kmer_size, !p->noncanonical, a.codes != nullptr) : get_bytes_launcher(p->kmer_size);
    if (!fn) return fail(ctx, MASHGPU_ERR_INVALID, "no scan kernel for k=%d", p->kmer_size);
    uint64_t ntiles = a.tile_end - a.tile_begin;
    if (ntiles == 0) return MASHGPU_OK;
    time_begin(ctx, ctx->scan_events, st);
    fn(a, 0, st);     // grid = resident CTAs (persistent warps striding over warp tiles)
    time_end(ctx, ctx->scan_events, st);
    ctx->kernel_launches++;
    ctx->scan_launches++;
    MG_CUDA(ctx, cudaGetLastError());
    return MASHGPU_OK;
}

// Occurrences of `target` at stream positions [unit start, tstar] -> the count of unit u's last hash
static int recount_hash(mashgpu_ctx *ctx, const SketchTicket &t, uint32_t u, uint64_t tstar, uint64_t target)
{
    const uint32_t s = t.params.sketch_size;
    uint32_t *d_count_slot = t.d_out_counts + (uint64_t)u * s + s - 1;
    ScanArgs c = scan_args(&t.params, t.S.d_stream, t.S.d_codes, t.S.d_inval, t.S.unit_start[t.S.n_units]);
    c.mode = SCAN_COUNT;
    c.tile_begin = t.S.unit_start[u] / SCAN_TILE;
    c.tile_end = tstar / SCAN_TILE + 1;
    c.coarse_t = target;
    c.count_target = target; c.count_lo = t.S.unit_start[u]; c.count_hi = tstar; c.count_out = d_count_slot;
    MG_CUDA(ctx, cudaMemsetAsync(d_count_slot, 0, 4, t.st));
    return launch_scan(ctx, &t.params, c, t.st);
}

// One pass over units of the ticket's stream: plan thresholds and tables, scan, select the bottom-s, apply the counting quirk and
// copy the units' flags into ctx->flags_pinned at their unit numbers.  No sync.
//   only_unit < 0: the first pass, over every unit, with the caller's threshold cap and the screen probe.
//   only_unit = u: the exact re-run of unit u with a larger survivor factor.  Per-unit device arrays keep their absolute index.
static int sketch_pass(mashgpu_ctx *ctx, SketchTicket &t, const ScreenProbe *probe, int64_t only_unit, double factor)
{
    const mashgpu_sketch_params *p = &t.params;
    const SketchStream &S = t.S;
    cudaStream_t st = t.st;
    const bool first = only_unit < 0;
    const uint32_t n_units = (uint32_t)S.n_units;
    const uint32_t u0 = first ? 0 : (uint32_t)only_unit, nu = first ? n_units : 1;
    const uint32_t s = p->sketch_size, mc = t.min_copies;
    const bool capped = first && S.t_cap;
    const uint64_t capped_t = capped ? S.t_cap_value : EMPTY_KEY;
    const uint64_t tile_begin = S.unit_start[u0] / SCAN_TILE, tile_end = (S.unit_start[u0 + nu] + SCAN_TILE - 1) / SCAN_TILE;

    // plan: entry i is unit u0 + i; the pass's tables start at slot 0
    std::vector<uint64_t> h_t(nu), h_off(nu);
    std::vector<uint32_t> h_log2(nu);
    uint64_t slots = 0;
    for (uint32_t i = 0; i < nu; i++) {
        uint64_t span = S.unit_start[u0 + i + 1] - S.unit_start[u0 + i];
        plan_unit(p, span, factor, &h_t[i], &h_log2[i]);
        // screen, mixture already holds s hashes: exactly the hashes <= its s-th smallest can still matter -- use that
        // value as the threshold whether the planned one is larger (fewer candidates) or smaller (it would miss some and
        // force an exact re-run when the chunk is full of repeats, e.g. reads at 5x coverage)
        if (capped) h_t[i] = S.t_cap_value;
        h_off[i] = slots;
        slots += 1ull << h_log2[i];
    }
    uint64_t *d_start = ctx->sc_start.get<uint64_t>(n_units + 1), *d_t = ctx->sc_t.get<uint64_t>(n_units), *d_off = ctx->sc_off.get<uint64_t>(n_units);
    uint32_t *d_log2 = ctx->sc_log2.get<uint32_t>(n_units), *d_flags = ctx->sc_flags.get<uint32_t>(n_units), *d_maxhash = ctx->sc_maxhash.get<uint32_t>(n_units);
    uint64_t *d_keys = ctx->sc_keys.get<uint64_t>(slots), *d_tmax = ctx->sc_tmax.get<uint64_t>(tile_end);
    uint32_t *d_cnt = ctx->sc_cnt.get<uint32_t>(slots);
    if (!d_start || !d_t || !d_off || !d_log2 || !d_flags || !d_maxhash || !d_keys || !d_cnt || !d_tmax)
        return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (%llu candidate slots for %u units)", (unsigned long long)slots, nu);
    const bool want_counts = t.d_out_counts != nullptr;
    uint64_t *d_first = nullptr, *d_last = nullptr;
    if (want_counts) {
        d_first = ctx->sc_first.get<uint64_t>(slots * mc); d_last = ctx->sc_last.get<uint64_t>(slots);
        t.d_qtarget = ctx->sc_qtarget.get<uint64_t>(n_units); t.d_qtstar = ctx->sc_qtstar.get<uint64_t>(n_units);
        if (!d_first || !d_last || !t.d_qtarget || !t.d_qtstar) return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (first/last occurrence tables)");
        MG_CUDA(ctx, cudaMemsetAsync(d_first, 0xFF, slots * mc * 8ull, st));
        MG_CUDA(ctx, cudaMemsetAsync(d_last, 0, slots * 8ull, st));
    }
    if (first) MG_CUDA(ctx, cudaMemcpyAsync(d_start, S.unit_start, (n_units + 1) * 8ull, cudaMemcpyHostToDevice, st));
    MG_CUDA(ctx, cudaMemcpyAsync(d_t + u0, h_t.data(), nu * 8ull, cudaMemcpyHostToDevice, st));
    MG_CUDA(ctx, cudaMemcpyAsync(d_off + u0, h_off.data(), nu * 8ull, cudaMemcpyHostToDevice, st));
    MG_CUDA(ctx, cudaMemcpyAsync(d_log2 + u0, h_log2.data(), nu * 4ull, cudaMemcpyHostToDevice, st));
    MG_CUDA(ctx, cudaMemsetAsync(d_flags + u0, 0, nu * 4ull, st));
    MG_CUDA(ctx, cudaMemsetAsync(d_maxhash + u0, 0, nu * 4ull, st));
    MG_CUDA(ctx, cudaMemsetAsync(d_keys, 0xFF, slots * 8ull, st));
    MG_CUDA(ctx, cudaMemsetAsync(d_cnt, 0, slots * 4ull, st));

    ScanArgs a = scan_args(p, S.d_stream, S.d_codes, S.d_inval, S.unit_start[n_units]);
    a.tile_begin = tile_begin;
    a.tile_end = tile_end;
    a.mode = probe ? SCAN_SCREEN : SCAN_SKETCH;      // a re-run has no probe: reference-table hits were counted in the first pass
    a.unit_start = d_start;
    a.n_units = n_units;
    a.unit_t = d_t;
    a.tab_off = d_off;
    a.tab_log2 = d_log2;
    a.tab_keys = d_keys;
    a.tab_cnt = d_cnt;
    a.unit_flags = d_flags;
    a.unit_maxhash = d_maxhash;
    a.tab_first = d_first;
    a.tab_last = d_last;
    a.only_unit = only_unit;
    a.min_copies = mc;
    uint64_t tm = 0;
    for (uint32_t i = 0; i < nu; i++) tm = std::max(tm, h_t[i]);
    a.coarse_t = tm;                                   // used without per-tile thresholds: a re-run (one unit)
    if (first) {
        if (tile_end > tile_begin) {
            tile_tmax_kernel<<<(unsigned)((tile_end - tile_begin + 255) / 256), 256, 0, st>>>(d_start, n_units, d_t, a.stream_len, tile_begin, tile_end, d_tmax);
            ctx->kernel_launches++;
        }
        a.tile_tmax = d_tmax;
    }
    if (probe) {
        a.ref_keys = probe->keys; a.ref_idx = probe->idx; a.ref_cnt = probe->cnt; a.ref_log2 = probe->log2cap; a.ref_hmax = probe->hmax;
        a.ref_bitmap = probe->bitmap; a.ref_bitmap_shift = probe->bitmap_shift;
        // coarse filter must also let reference-hash candidates through
        a.tile_tmax = nullptr;
        a.coarse_t = std::max(tm, probe->hmax);
        a.screen_mix_t = tm;
    }
    if (first && S.data_ready) MG_CUDA(ctx, cudaStreamWaitEvent(st, S.data_ready, 0));
    MG_TRY(launch_scan(ctx, p, a, st));

    const size_t sel_smem = (size_t)8 << SEL_MAX_LOG2;
    if (!ctx->attr_select) {   // per context: function attributes are per device
        MG_CUDA(ctx, cudaFuncSetAttribute(select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sel_smem));
        ctx->attr_select = true;
    }
    uint32_t max_log2 = 4;
    for (uint32_t i = 0; i < nu; i++) max_log2 = std::max(max_log2, std::min(h_log2[i], SEL_MAX_LOG2));
    select_kernel<<<nu, SEL_THREADS, (size_t)8 << max_log2, st>>>(u0, nu, d_t, d_off, d_log2, d_keys, d_cnt, d_maxhash, d_flags, s, capped_t,
                                                                t.d_out_hashes, t.d_out_counts, t.d_out_n, mc);
    ctx->kernel_launches++;
    MG_CUDA(ctx, cudaGetLastError());
    {   // units whose candidate table exceeds the shared-memory sort (large sketch sizes): one segmented sort for all of them
        std::vector<uint32_t> big;
        std::vector<uint64_t> seg_off;
        uint64_t comp_total = 0, max_cap = 0;
        for (uint32_t i = 0; i < nu; i++)
            if (h_log2[i] > SEL_MAX_LOG2) { big.push_back(u0 + i); seg_off.push_back(comp_total); comp_total += 1ull << h_log2[i]; max_cap = std::max<uint64_t>(max_cap, 1ull << h_log2[i]); }
        if (!big.empty()) {
            if (comp_total >= 0x7FFFFFFFull) return fail(ctx, MASHGPU_ERR_UNSUPPORTED, "candidate tables of one wave exceed 2^31 slots (sketch_size %u x %zu units): feed fewer units per call", s, big.size());
            const uint32_t n_big = (uint32_t)big.size();
            uint32_t *d_big = ctx->sc_big_units.get<uint32_t>(n_big), *d_seg_n = ctx->sc_big_n.get<uint32_t>(n_big);
            uint64_t *d_seg_off = ctx->sc_big_off.get<uint64_t>(n_big);
            long long *d_bounds = ctx->sc_big_bounds.get<long long>(2ull * n_big);
            uint64_t *d_comp = ctx->sc_big_comp.get<uint64_t>(comp_total), *d_sorted = ctx->sc_big_sorted.get<uint64_t>(comp_total);
            if (!d_big || !d_seg_n || !d_seg_off || !d_bounds || !d_comp || !d_sorted) return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (sort buffers of %llu candidate slots)", (unsigned long long)comp_total);
            MG_CUDA(ctx, cudaMemcpyAsync(d_big, big.data(), n_big * 4ull, cudaMemcpyHostToDevice, st));
            MG_CUDA(ctx, cudaMemcpyAsync(d_seg_off, seg_off.data(), n_big * 8ull, cudaMemcpyHostToDevice, st));
            MG_CUDA(ctx, cudaMemsetAsync(d_seg_n, 0, n_big * 4ull, st));
            const unsigned bx = (unsigned)std::min<uint64_t>((max_cap + 255) / 256, 256);
            select_big_compact_kernel<<<dim3(bx, n_big), 256, 0, st>>>(d_big, n_big, d_seg_off, d_off, d_log2, d_keys, d_cnt, d_flags, mc, d_comp, d_seg_n);
            select_big_bounds_kernel<<<(n_big + 255) / 256, 256, 0, st>>>(d_seg_off, d_seg_n, n_big, d_bounds, d_bounds + n_big);
            size_t tmp_bytes = 0;
            cub::DeviceSegmentedRadixSort::SortKeys(nullptr, tmp_bytes, d_comp, d_sorted, (int)comp_total, (int)n_big, d_bounds, d_bounds + n_big, 0, 64, st);
            uint8_t *d_tmp = ctx->sc_big_tmp.get<uint8_t>(tmp_bytes);
            if (!d_tmp) return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (segmented sort scratch)");
            MG_CUDA(ctx, cub::DeviceSegmentedRadixSort::SortKeys(d_tmp, tmp_bytes, d_comp, d_sorted, (int)comp_total, (int)n_big, d_bounds, d_bounds + n_big, 0, 64, st));
            select_big_emit_kernel<<<n_big, SEL_THREADS, 0, st>>>(d_big, n_big, d_seg_off, d_seg_n, d_sorted, d_t, d_off, d_log2, d_keys, d_cnt, d_maxhash, d_flags,
                                                                s, capped_t, t.d_out_hashes, t.d_out_counts, t.d_out_n, mc);
            ctx->kernel_launches += 4;
            MG_CUDA(ctx, cudaGetLastError());
        }
    }
    if (want_counts) {
        quirk_kernel<<<nu, SEL_THREADS, 0, st>>>(u0, nu, s, t.d_out_hashes, t.d_out_counts, t.d_out_n, d_off, d_log2, d_keys, d_cnt,
                                                 d_first, d_last, d_flags, t.d_qtarget, t.d_qtstar, mc);
        ctx->kernel_launches++;
        MG_CUDA(ctx, cudaGetLastError());
    }

    if (ctx->flags_pinned_n < n_units) {          // one ticket in flight per context: its flags land in the context's pinned buffer
        if (ctx->flags_pinned) cudaFreeHost(ctx->flags_pinned);
        ctx->flags_pinned = nullptr; ctx->flags_pinned_n = 0;
        const size_t want = (size_t)n_units + n_units / 4 + 64;
        if (cudaMallocHost(&ctx->flags_pinned, want * 4) != cudaSuccess) return fail(ctx, MASHGPU_ERR_NOMEM, "out of pinned host memory (unit flags)");
        ctx->flags_pinned_n = want;
    }
    MG_CUDA(ctx, cudaMemcpyAsync((uint32_t *)ctx->flags_pinned + u0, d_flags + u0, nu * 4ull, cudaMemcpyDeviceToHost, st));
    return MASHGPU_OK;
}

// Core: sketch every unit of a device-resident stream.
int sketch_stream_core(mashgpu_ctx *ctx, const mashgpu_sketch_params *p, const SketchStream &S,
                       uint64_t *d_out_hashes, uint32_t *d_out_counts, uint32_t *d_out_n, cudaStream_t st,
                       const ScreenProbe *probe)
{
    SketchTicket t;
    MG_TRY(sketch_stream_enqueue(ctx, p, S, d_out_hashes, d_out_counts, d_out_n, st, probe, t));
    return sketch_stream_finalize(ctx, t);
}

int sketch_stream_enqueue(mashgpu_ctx *ctx, const mashgpu_sketch_params *p, const SketchStream &S,
                          uint64_t *d_out_hashes, uint32_t *d_out_counts, uint32_t *d_out_n, cudaStream_t st,
                          const ScreenProbe *probe, SketchTicket &t)
{
    t.active = false;
    const uint32_t n_units = (uint32_t)S.n_units;
    if (n_units == 0) return MASHGPU_OK;
    t.params = *p;
    t.S = S;
    t.unit_start.assign(S.unit_start, S.unit_start + n_units + 1);
    t.S.unit_start = t.unit_start.data();
    t.d_out_hashes = d_out_hashes; t.d_out_counts = d_out_counts; t.d_out_n = d_out_n; t.st = st;
    t.min_copies = probe ? 1u : std::max(1u, p->min_copies);      // the screen mixture is a plain MinHashHeap (CommandScreen.cpp:114-119)
    MG_TRY(sketch_pass(ctx, t, probe, -1, SURVIVOR_FACTOR));
    t.active = true;
    return MASHGPU_OK;
}

int sketch_stream_finalize(mashgpu_ctx *ctx, SketchTicket &t)
{
    if (!t.active) return MASHGPU_OK;
    t.active = false;
    const uint32_t n_units = (uint32_t)t.S.n_units;
    const uint32_t *flags = (const uint32_t *)ctx->flags_pinned;      // a re-run of unit u rewrites entry u only
    MG_CUDA(ctx, cudaStreamSynchronize(t.st));
    bool any_recount = false;
    for (uint32_t u = 0; u < n_units; u++) {
        if (flags[u] & 7u) {
            // overflow or too few survivors: re-run the unit alone with 8x the expected survivors until it passes (keep-all always does)
            ctx->exact_reruns++;
            double factor = SURVIVOR_FACTOR;
            for (int attempt = 0; flags[u] & 7u; attempt++) {
                if (attempt == 64) return fail(ctx, MASHGPU_ERR_CUDA, "exact re-run of unit %u did not converge", u);
                factor *= 8.0;
                MG_TRY(sketch_pass(ctx, t, nullptr, u, factor));
                MG_CUDA(ctx, cudaStreamSynchronize(t.st));
            }
        }
        any_recount |= (flags[u] & 8u) != 0;
    }
    if (!any_recount) return MASHGPU_OK;
    std::vector<uint64_t> qtarget(n_units), qtstar(n_units);
    MG_CUDA(ctx, cudaMemcpyAsync(qtarget.data(), t.d_qtarget, n_units * 8ull, cudaMemcpyDeviceToHost, t.st));
    MG_CUDA(ctx, cudaMemcpyAsync(qtstar.data(), t.d_qtstar, n_units * 8ull, cudaMemcpyDeviceToHost, t.st));
    MG_CUDA(ctx, cudaStreamSynchronize(t.st));
    for (uint32_t u = 0; u < n_units; u++)
        if (flags[u] & 8u) MG_TRY(recount_hash(ctx, t, u, qtstar[u], qtarget[u]));
    MG_CUDA(ctx, cudaStreamSynchronize(t.st));
    return MASHGPU_OK;
}

}  // namespace mashgpu

using namespace mashgpu;

extern "C" uint32_t mashgpu_set_alphabet(mashgpu_sketch_params *p, const char *characters)
{
    // setAlphabetFromString, reference Sketch.cpp:1108-1137
    memset(p->alphabet, 0, 256);
    for (const char *c = characters; *c; c++) {
        unsigned char u = (unsigned char)*c;
        if (!p->preserve_case && u > 96 && u < 123) u -= 32;
        p->alphabet[u] = 1;
    }
    p->use64 = kmer_space_of(p) > std::pow(2.0, 32.0);
    return alphabet_size(p);
}

extern "C" int mashgpu_sketch_stream_dev(mashgpu_ctx *ctx, const mashgpu_sketch_params *params,
                                         const void *d_stream, const uint64_t *unit_start, uint64_t n_units,
                                         uint64_t *d_out_hashes, uint32_t *d_out_counts, uint32_t *d_out_n, void *stream)
{
    if (!ctx) return MASHGPU_ERR_INVALID;
    MG_TRY(validate_sketch_params(ctx, params));
    if (n_units > 0xFFFFFFF0ull) return fail(ctx, MASHGPU_ERR_INVALID, "too many units");
    if (n_units && (!d_stream || !unit_start || !d_out_hashes || !d_out_n)) return fail(ctx, MASHGPU_ERR_INVALID, "NULL argument");
    MG_CUDA(ctx, cudaSetDevice(ctx->device));
    SketchStream S;
    S.d_stream = d_stream; S.unit_start = unit_start; S.n_units = n_units;
    return sketch_stream_core(ctx, params, S, d_out_hashes, d_out_counts, d_out_n, stream ? (cudaStream_t)stream : ctx->stream, nullptr);
}

namespace {

struct Wave { uint64_t unit_begin, unit_end, rec_begin, rec_end, bytes; };

constexpr uint64_t WAVE_BYTES = 1ull << 30;        // stream bytes per wave (the two feed paths share the waves of a batch: finer than 2 GiB balances better)
constexpr uint32_t SEP_LIST_MAX = 1u << 15;        // directly copied records per wave whose separators go through the list
constexpr uint64_t DIRECT_COPY_MIN = 1ull << 18;   // records at least this long are copied straight from the caller's buffer

// Waves are cut by stream bytes and by unit count (outputs and candidate tables grow with the number of units, not with their
// length -- a multi-FASTA of millions of short records must not allocate units x s outputs at once).
struct WaveLimits { uint64_t bytes, units; };

WaveLimits wave_limits(uint32_t s)
{
    WaveLimits w{WAVE_BYTES, std::max<uint64_t>(64, (1ull << 28) / ((uint64_t)s * 8))};
    if (const char *env = getenv("MASHGPU_WAVE_BYTES")) w.bytes = std::max<uint64_t>(1024, strtoull(env, nullptr, 10));      // tests: many waves from little data
    if (const char *env = getenv("MASHGPU_WAVE_UNITS")) w.units = std::max<uint64_t>(1, strtoull(env, nullptr, 10));
    return w;
}

// The sketches of a call's waves: computed into the context's output scratch (sized for the largest wave), then copied to the
// caller's arrays at the wave's first unit.
struct WaveOutputs {
    uint64_t *d_hashes; uint32_t *d_counts, *d_n;
    uint64_t *hashes; uint32_t *counts, *n;       // the caller's (counts may be NULL)
};

int wave_outputs(mashgpu_ctx *ctx, uint32_t s, uint64_t max_units, uint64_t *hashes, uint32_t *counts, uint32_t *n, WaveOutputs &o)
{
    o.d_hashes = ctx->sc_out_hashes.get<uint64_t>(max_units * s);
    o.d_n = ctx->sc_out_n.get<uint32_t>(max_units);
    o.d_counts = counts ? ctx->sc_out_counts.get<uint32_t>(max_units * s) : nullptr;
    o.hashes = hashes; o.counts = counts; o.n = n;
    if (!o.d_hashes || !o.d_n || (counts && !o.d_counts)) return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (outputs)");
    return MASHGPU_OK;
}

int sketch_wave(mashgpu_ctx *ctx, const mashgpu_sketch_params *p, const SketchStream &S, uint64_t unit_begin, const WaveOutputs &o)
{
    const uint64_t s = p->sketch_size, nu = S.n_units;
    MG_TRY(sketch_stream_core(ctx, p, S, o.d_hashes, o.d_counts, o.d_n, ctx->stream, nullptr));
    MG_CUDA(ctx, cudaMemcpyAsync(o.hashes + unit_begin * s, o.d_hashes, nu * s * 8ull, cudaMemcpyDeviceToHost, ctx->stream));
    MG_CUDA(ctx, cudaMemcpyAsync(o.n + unit_begin, o.d_n, nu * 4ull, cudaMemcpyDeviceToHost, ctx->stream));
    if (o.counts) MG_CUDA(ctx, cudaMemcpyAsync(o.counts + unit_begin * s, o.d_counts, nu * s * 4ull, cudaMemcpyDeviceToHost, ctx->stream));
    MG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MASHGPU_OK;
}

}  // namespace

extern "C" int mashgpu_sketch_batch(mashgpu_ctx *ctx, const mashgpu_sketch_params *params,
                                    uint64_t n_records, const char *const *seq, const uint64_t *len,
                                    const uint32_t *unit_of_record, uint64_t n_units,
                                    uint64_t *out_hashes, uint32_t *out_counts, uint32_t *out_n, uint64_t *out_length)
{
    if (!ctx) return MASHGPU_ERR_INVALID;
    MG_TRY(validate_sketch_params(ctx, params));
    if (n_units == 0) return MASHGPU_OK;
    if (!out_hashes || !out_n) return fail(ctx, MASHGPU_ERR_INVALID, "out_hashes/out_n is NULL");
    if (n_records && (!seq || !len)) return fail(ctx, MASHGPU_ERR_INVALID, "seq/len is NULL");
    if (n_units > 0xFFFFFFF0ull) return fail(ctx, MASHGPU_ERR_INVALID, "too many units");
    MG_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t s = params->sketch_size;
    const uint64_t k = (uint64_t)params->kmer_size;

    // unit spans in the flat stream: kept records back to back, one separator byte after each
    std::vector<uint64_t> unit_bytes(n_units, 0), unit_rec_begin(n_units + 1, 0);
    {
        uint64_t r = 0;
        for (uint64_t u = 0; u < n_units; u++) {
            unit_rec_begin[u] = r;
            while (r < n_records && (unit_of_record ? unit_of_record[r] : r) == u) {
                if (len[r] >= k) unit_bytes[u] += len[r] + 1;
                r++;
            }
            if (r < n_records && unit_of_record && unit_of_record[r] < u)
                return fail(ctx, MASHGPU_ERR_INVALID, "unit_of_record must be non-decreasing");
        }
        unit_rec_begin[n_units] = r;
        if (r != n_records) return fail(ctx, MASHGPU_ERR_INVALID, "unit_of_record refers to units >= n_units or is not sorted");
    }
    if (out_length)
        for (uint64_t u = 0; u < n_units; u++) {
            uint64_t L = 0;
            for (uint64_t r = unit_rec_begin[u]; r < unit_rec_begin[u + 1]; r++)
                if (len[r] >= k) L += len[r];
            out_length[u] = L;
        }

    const WaveLimits lim = wave_limits(s);
    std::vector<Wave> waves;
    {
        Wave w{0, 0, 0, 0, 0};
        for (uint64_t u = 0; u < n_units; u++) {
            if (w.unit_end > w.unit_begin && (w.bytes + unit_bytes[u] > lim.bytes || w.unit_end - w.unit_begin >= lim.units)) {
                w.rec_end = unit_rec_begin[u];
                waves.push_back(w);
                w = Wave{u, u, unit_rec_begin[u], 0, 0};
            }
            w.unit_end = u + 1;
            w.bytes += unit_bytes[u];
        }
        w.rec_end = n_records;
        waves.push_back(w);
    }
    const size_t n_waves = waves.size();
    uint64_t max_bytes = 32, max_units = 1;
    for (auto &w : waves) { max_bytes = std::max(max_bytes, w.bytes); max_units = std::max(max_units, w.unit_end - w.unit_begin); }

    // ---- feed paths.  A wave reaches the GPU either as ASCII (DMA straight from the caller's buffers: no host CPU work, 1 byte
    // per base over PCIe) or 2-bit packed by host threads (pack.cpp: a quarter of the bytes, but ~6 GB/s per host core).  The two
    // producers run side by side and claim waves from one list, so the split follows their real speeds: PCIe carries
    // ~52 GB/s of ASCII, 15 packer threads add ~60 GB/s of bases at 15 GB/s of PCIe (hybrid: ~2x the ASCII-only rate, measured
    // in profiles/r02_feed_path.md).  Packing is the only producer for waves with small records or pageable buffers (a
    // cudaMemcpyAsync from pageable memory is staged by the driver at a fraction of the PCIe rate and blocks this thread).
    // MASHGPU_HOST_PACK=0: ASCII only; =1: packed only; unset: both.  Non-DNA alphabets are ASCII only.
    enum { FEED_ASCII = 1, FEED_PACK = 2 };
    int feed = FEED_ASCII | FEED_PACK;
    if (const char *env = getenv("MASHGPU_HOST_PACK")) feed = env[0] == '0' ? FEED_ASCII : (env[0] == '1' ? FEED_PACK : feed);
    if (!is_dna_alphabet(params)) feed = FEED_ASCII;
    // ASCII-eligible waves: every kept record is long enough for a direct copy and lies in pinned (page-locked) memory
    std::vector<uint8_t> ascii_ok(n_waves, 1);
    if (feed == (FEED_ASCII | FEED_PACK)) {
        for (size_t wi = 0; wi < n_waves; wi++) {
            const Wave &w = waves[wi];
            bool ok = true;
            bool probed = false;
            for (uint64_t r = w.rec_begin; r < w.rec_end && ok; r++) {
                if (len[r] < k) continue;
                if (len[r] < DIRECT_COPY_MIN) ok = false;
                else if (!probed) {          // one probe per wave: callers allocate their records the same way
                    cudaPointerAttributes at;
                    if (cudaPointerGetAttributes(&at, seq[r]) != cudaSuccess) { cudaGetLastError(); ok = false; }
                    else if (at.type != cudaMemoryTypeHost && at.type != cudaMemoryTypeManaged) ok = false;
                    probed = true;
                }
            }
            ascii_ok[wi] = ok;
        }
    }
    // packer threads: as many as the process may actually run (pack.cpp: hardware threads, the container's CPU quota,
    // MASHGPU_PACK_THREADS) -- minus one for this thread when it also drives the ASCII copies
    int threads = host_pack_threads();
    if ((feed & FEED_ASCII) && !getenv("MASHGPU_PACK_THREADS")) threads = std::max(1, threads - 1);

    WaveOutputs outs;
    MG_TRY(wave_outputs(ctx, s, max_units, out_hashes, out_counts, out_n, outs));

    // ---- ASCII producer: two device wave buffers, copies on copy_stream
    struct AsciiSlot { int64_t wave = -1; uint8_t *d = nullptr; std::vector<uint64_t> unit_start; };
    AsciiSlot aslot[2];
    const uint64_t buf_bytes = ((max_bytes + 15) / 16) * 16 + 16;
    const int n_aslots = (feed & FEED_ASCII) ? (n_waves > 1 ? 2 : 1) : 0;
    cudaEvent_t *copied = ctx->wave_copied;
    for (int b = 0; b < n_aslots; b++) {
        aslot[b].d = ctx->sc_wave[b].get<uint8_t>(buf_bytes);
        if (!aslot[b].d) return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (stream buffer %llu B)", (unsigned long long)buf_bytes);
        if (!copied[b]) MG_CUDA(ctx, cudaEventCreateWithFlags(&copied[b], cudaEventDisableTiming));
    }
    auto issue_copy = [&](size_t wi, int b) -> int {
        const Wave &w = waves[wi];
        uint8_t *dst = aslot[b].d;
        // staging size: all small records of the wave
        uint64_t small_bytes = 0;
        for (uint64_t r = w.rec_begin; r < w.rec_end; r++)
            if (len[r] >= k && len[r] < DIRECT_COPY_MIN) small_bytes += len[r] + 1;
        if (ctx->pinned_bytes[b] < small_bytes) {
            if (ctx->pinned[b]) cudaFreeHost(ctx->pinned[b]);
            ctx->pinned[b] = nullptr; ctx->pinned_bytes[b] = 0;
            if (cudaMallocHost(&ctx->pinned[b], small_bytes + small_bytes / 8) != cudaSuccess)
                return fail(ctx, MASHGPU_ERR_NOMEM, "out of pinned host memory (%llu B)", (unsigned long long)small_bytes);
            ctx->pinned_bytes[b] = small_bytes + small_bytes / 8;
        }
        uint8_t *stage = (uint8_t *)ctx->pinned[b];
        std::vector<uint64_t> &us = aslot[b].unit_start;
        us.assign(w.unit_end - w.unit_begin + 1, 0);
        // separator offsets of the directly copied records (pinned list -> device -> one kernel); list full: 1-byte memsets
        if (!ctx->pinned_sep[b]) {
            if (cudaMallocHost(&ctx->pinned_sep[b], SEP_LIST_MAX * 8) != cudaSuccess) return fail(ctx, MASHGPU_ERR_NOMEM, "out of pinned host memory (separator list)");
        }
        uint64_t *h_sep = (uint64_t *)ctx->pinned_sep[b];
        uint64_t *d_sep = ctx->sc_sep[b].get<uint64_t>(SEP_LIST_MAX);
        if (!d_sep) return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (separator list)");
        uint32_t n_sep = 0;
        uint64_t off = 0, st_off = 0;
        uint64_t run_dst = 0, run_src = 0, run_len = 0;   // pending staged run
        auto flush_run = [&]() -> cudaError_t {
            if (!run_len) return cudaSuccess;
            cudaError_t e = cudaMemcpyAsync(dst + run_dst, stage + run_src, run_len, cudaMemcpyHostToDevice, ctx->copy_stream);
            run_len = 0;
            return e;
        };
        for (uint64_t u = w.unit_begin; u < w.unit_end; u++) {
            us[u - w.unit_begin] = off;
            for (uint64_t r = unit_rec_begin[u]; r < unit_rec_begin[u + 1]; r++) {
                if (len[r] < k) continue;
                if (len[r] >= DIRECT_COPY_MIN) {
                    MG_CUDA(ctx, flush_run());
                    MG_CUDA(ctx, cudaMemcpyAsync(dst + off, seq[r], len[r], cudaMemcpyHostToDevice, ctx->copy_stream));
                    if (n_sep < SEP_LIST_MAX) h_sep[n_sep++] = off + len[r];
                    else MG_CUDA(ctx, cudaMemsetAsync(dst + off + len[r], 0, 1, ctx->copy_stream));
                } else {
                    if (!run_len) { run_dst = off; run_src = st_off; }
                    memcpy(stage + st_off, seq[r], len[r]);
                    stage[st_off + len[r]] = 0;
                    st_off += len[r] + 1;
                    run_len += len[r] + 1;
                }
                off += len[r] + 1;
            }
        }
        MG_CUDA(ctx, flush_run());
        if (n_sep) {
            MG_CUDA(ctx, cudaMemcpyAsync(d_sep, h_sep, n_sep * 8ull, cudaMemcpyHostToDevice, ctx->copy_stream));
            write_separators_kernel<<<(n_sep + 255) / 256, 256, 0, ctx->copy_stream>>>(dst, d_sep, n_sep);
            MG_CUDA(ctx, cudaGetLastError());
            ctx->kernel_launches++;
        }
        us[w.unit_end - w.unit_begin] = off;
        MG_CUDA(ctx, cudaEventRecord(copied[b], ctx->copy_stream));
        aslot[b].wave = (int64_t)wi;
        return MASHGPU_OK;
    };

    // ---- packed producer: two pinned code buffers, one packing job at a time on `threads` host threads; the job itself enqueues
    // its upload (codes, invalid runs -> mask) on pack_stream, so a finished future means "event recorded"
    struct PackSlot {
        int64_t wave = -1;
        uint64_t *h_codes = nullptr, *d_codes = nullptr; uint32_t *d_inval = nullptr;
        std::vector<uint64_t> unit_start; std::vector<PackRun> runs; uint64_t len = 0;
    };
    PackSlot pslot[2];
    const int n_pslots = (feed & FEED_PACK) ? (n_waves > 1 ? 2 : 1) : 0;
    const uint64_t max_tiles = (max_bytes + SCAN_TILE - 1) / SCAN_TILE;
    const uint64_t groups_alloc = max_tiles * (SCAN_TILE / 32) + 64;       // tile-padded + halo
    for (int b = 0; b < n_pslots; b++) {
        pslot[b].d_codes = ctx->sc_codes[b].get<uint64_t>(groups_alloc);
        pslot[b].d_inval = ctx->sc_inval[b].get<uint32_t>(groups_alloc);
        if (!pslot[b].d_codes || !pslot[b].d_inval) return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (packed stream of %llu groups)", (unsigned long long)groups_alloc);
        if (ctx->pinned_codes_bytes[b] < groups_alloc * 8) {
            if (ctx->pinned_codes[b]) cudaFreeHost(ctx->pinned_codes[b]);
            ctx->pinned_codes[b] = nullptr; ctx->pinned_codes_bytes[b] = 0;
            if (cudaMallocHost(&ctx->pinned_codes[b], groups_alloc * 8) != cudaSuccess)
                return fail(ctx, MASHGPU_ERR_NOMEM, "out of pinned host memory (%llu B)", (unsigned long long)(groups_alloc * 8));
            ctx->pinned_codes_bytes[b] = groups_alloc * 8;
        }
        pslot[b].h_codes = (uint64_t *)ctx->pinned_codes[b];
        if (!ctx->pack_copied[b]) MG_CUDA(ctx, cudaEventCreateWithFlags(&ctx->pack_copied[b], cudaEventDisableTiming));
    }
    if (n_pslots && !ctx->pack_stream) MG_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->pack_stream, cudaStreamNonBlocking));
    auto pack_job = [&](size_t wi, int b) -> int {
        cudaSetDevice(ctx->device);
        const Wave &w = waves[wi];
        PackSlot &P = pslot[b];
        std::vector<PackSegment> segs;
        segs.reserve(w.rec_end - w.rec_begin);
        P.unit_start.assign(w.unit_end - w.unit_begin + 1, 0);
        uint64_t off = 0;
        for (uint64_t u = w.unit_begin; u < w.unit_end; u++) {
            P.unit_start[u - w.unit_begin] = off;
            for (uint64_t r = unit_rec_begin[u]; r < unit_rec_begin[u + 1]; r++) {
                if (len[r] < k) continue;
                segs.push_back(PackSegment{(const uint8_t *)seq[r], off, len[r]});
                off += len[r] + 1;                     // one separator position after every record
            }
        }
        P.unit_start[w.unit_end - w.unit_begin] = off;
        P.len = off;
        pack_stream(segs.data(), segs.size(), off, params->preserve_case, threads, P.h_codes, P.runs);
        P.runs.push_back(PackRun{off, groups_alloc * 32 - off});      // everything from the end of the stream to the end of the allocation is invalid
        // upload: codes, zeroed mask, runs -> mask
        const uint64_t groups = (P.len + 31) / 32;
        cudaStream_t cs = ctx->pack_stream;
        if (groups && cudaMemcpyAsync(P.d_codes, P.h_codes, groups * 8, cudaMemcpyHostToDevice, cs) != cudaSuccess) return MASHGPU_ERR_CUDA;
        if (cudaMemsetAsync(P.d_inval, 0, groups_alloc * 4, cs) != cudaSuccess) return MASHGPU_ERR_CUDA;
        PackRun *d_runs = ctx->sc_runs[b].get<PackRun>(P.runs.size());
        if (!d_runs) return MASHGPU_ERR_NOMEM;
        if (cudaMemcpyAsync(d_runs, P.runs.data(), P.runs.size() * sizeof(PackRun), cudaMemcpyHostToDevice, cs) != cudaSuccess) return MASHGPU_ERR_CUDA;
        const uint64_t nr = P.runs.size();
        const unsigned blocks = (unsigned)std::min<uint64_t>((nr * 32 + 255) / 256, 148 * 16);
        apply_runs_kernel<<<std::max(1u, blocks), 256, 0, cs>>>(d_runs, nr, P.d_inval);
        if (cudaGetLastError() != cudaSuccess) return MASHGPU_ERR_CUDA;
        if (cudaEventRecord(ctx->pack_copied[b], cs) != cudaSuccess) return MASHGPU_ERR_CUDA;
        return MASHGPU_OK;          // the upload is in flight: the slot is ready once the event has fired (its buffers are reused only after that)
    };

    // ---- scheduler: both producers claim the next unclaimed wave they may take; this thread runs the kernels of whichever
    // wave is ready first and hands its sketches back
    std::vector<uint8_t> claimed(n_waves, 0);
    size_t a_cursor = 0, p_cursor = 0, done = 0;
    std::mutex mu;                      // guards `claimed` and the packed slots' states (this thread and the packer thread)
    std::condition_variable cv;
    auto claim = [&](size_t &cursor, bool need_ascii) -> int64_t {
        std::lock_guard<std::mutex> lock(mu);
        for (size_t wi = cursor; wi < n_waves; wi++) {
            if (claimed[wi]) { if (wi == cursor) cursor++; continue; }
            if (need_ascii && !ascii_ok[wi] && (feed & FEED_PACK)) continue;      // left to the packer
            claimed[wi] = 1;
            return (int64_t)wi;
        }
        return -1;
    };
    int rc = MASHGPU_OK;
    enum { P_EMPTY, P_PACKING, P_UPLOADING };
    int pstate[2] = {P_EMPTY, P_EMPTY};         // under `mu`
    int pack_rc = MASHGPU_OK;                   // under `mu`: first failure of the packer thread
    bool stop = false, packer_done = n_pslots == 0;
    // the packer thread: claims a wave whenever one of its two slots is empty, packs it on `threads` host threads, enqueues the
    // upload and moves on -- it never waits for this thread's kernels
    std::thread packer;
    if (n_pslots)
        packer = std::thread([&]() {
            cudaSetDevice(ctx->device);
            for (;;) {
                int b = -1;
                {
                    std::unique_lock<std::mutex> lock(mu);
                    cv.wait(lock, [&] { return stop || pstate[0] == P_EMPTY || (n_pslots > 1 && pstate[1] == P_EMPTY); });
                    if (stop) break;
                    b = pstate[0] == P_EMPTY ? 0 : 1;
                }
                const int64_t wi = claim(p_cursor, false);
                if (wi < 0) break;
                { std::lock_guard<std::mutex> lock(mu); pslot[b].wave = wi; pstate[b] = P_PACKING; }
                const int r = pack_job((size_t)wi, b);
                std::lock_guard<std::mutex> lock(mu);
                if (r != MASHGPU_OK) { pack_rc = r; break; }
                pstate[b] = P_UPLOADING;
            }
            std::lock_guard<std::mutex> lock(mu);
            packer_done = true;
        });
    while (done < n_waves && rc == MASHGPU_OK) {
        // 1. keep the ASCII producer busy
        for (int b = 0; b < n_aslots && rc == MASHGPU_OK; b++)
            if (aslot[b].wave < 0) {
                const int64_t wi = claim(a_cursor, true);
                if (wi >= 0) rc = issue_copy((size_t)wi, b);
            }
        if (rc != MASHGPU_OK) break;
        // 2. a finished wave?  packed first, then ASCII copies in issue order
        int ready_p = -1, ready_a = -1, uploading = -1;
        bool packing = false, p_done = false;
        {
            std::lock_guard<std::mutex> lock(mu);
            if (pack_rc != MASHGPU_OK) { rc = fail(ctx, pack_rc, "host packing / packed upload failed"); break; }
            p_done = packer_done;
            for (int b = 0; b < n_pslots; b++) {
                if (pstate[b] == P_PACKING) packing = true;
                if (pstate[b] == P_UPLOADING) {
                    const cudaError_t q = cudaEventQuery(ctx->pack_copied[b]);
                    if (q == cudaSuccess) { if (ready_p < 0 || pslot[b].wave < pslot[ready_p].wave) ready_p = b; }
                    else if (q != cudaErrorNotReady) { rc = fail(ctx, MASHGPU_ERR_CUDA, "packed upload failed: %s", cudaGetErrorString(q)); break; }
                    else { cudaGetLastError(); uploading = b; }
                }
            }
        }
        if (rc != MASHGPU_OK) break;
        if (ready_p < 0) {
            int64_t best = -1;
            for (int b = 0; b < n_aslots; b++)
                if (aslot[b].wave >= 0 && (best < 0 || aslot[b].wave < best)) {
                    const cudaError_t q = cudaEventQuery(copied[b]);
                    if (q == cudaSuccess) { ready_a = b; best = aslot[b].wave; }
                    else if (q != cudaErrorNotReady) { rc = fail(ctx, MASHGPU_ERR_CUDA, "H2D copy failed: %s", cudaGetErrorString(q)); break; }
                    else cudaGetLastError();
                }
        }
        if (rc != MASHGPU_OK) break;
        if (ready_p >= 0) {
            PackSlot &P = pslot[ready_p];
            ctx->kernel_launches++;             // apply_runs_kernel of the upload
            SketchStream S;
            S.d_codes = P.d_codes; S.d_inval = P.d_inval; S.unit_start = P.unit_start.data(); S.n_units = waves[P.wave].unit_end - waves[P.wave].unit_begin;
            rc = sketch_wave(ctx, params, S, waves[P.wave].unit_begin, outs);
            { std::lock_guard<std::mutex> lock(mu); P.wave = -1; pstate[ready_p] = P_EMPTY; }
            cv.notify_all();
            done++;
        } else if (ready_a >= 0) {
            AsciiSlot &A = aslot[ready_a];
            SketchStream S;
            S.d_stream = A.d; S.unit_start = A.unit_start.data(); S.n_units = waves[A.wave].unit_end - waves[A.wave].unit_begin;
            rc = sketch_wave(ctx, params, S, waves[A.wave].unit_begin, outs);
            A.wave = -1;
            done++;
        } else {
            // nothing ready: wait for whichever producer is in flight
            int64_t best = -1; int bb = -1;
            for (int b = 0; b < n_aslots; b++)
                if (aslot[b].wave >= 0 && (best < 0 || aslot[b].wave < best)) { best = aslot[b].wave; bb = b; }
            if (uploading >= 0) cudaEventSynchronize(ctx->pack_copied[uploading]);
            else if (packing || (!p_done && bb < 0)) std::this_thread::sleep_for(std::chrono::microseconds(50));
            else if (bb >= 0) MG_CUDA(ctx, cudaEventSynchronize(copied[bb]));
            else { rc = fail(ctx, MASHGPU_ERR_INVALID, "feed scheduler stalled (%zu of %zu waves done)", done, n_waves); break; }
        }
    }
    if (packer.joinable()) {
        { std::lock_guard<std::mutex> lock(mu); stop = true; }
        cv.notify_all();
        packer.join();                           // never leave the packer thread behind (it references this frame)
    }
    cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->pack_stream) cudaStreamSynchronize(ctx->pack_stream);
    return rc;
}

extern "C" int mashgpu_sketch_batch_packed(mashgpu_ctx *ctx, const mashgpu_sketch_params *params,
                                           const uint64_t *codes, uint64_t stream_len, const uint64_t *runs, uint64_t n_runs,
                                           const uint64_t *unit_start, uint64_t n_units,
                                           uint64_t *out_hashes, uint32_t *out_counts, uint32_t *out_n)
{
    if (!ctx) return MASHGPU_ERR_INVALID;
    MG_TRY(validate_sketch_params(ctx, params));
    if (n_units == 0) return MASHGPU_OK;
    if (!is_dna_alphabet(params)) return fail(ctx, MASHGPU_ERR_UNSUPPORTED, "the packed source only carries the alphabet {A,C,G,T}");
    if (!codes || !unit_start || !out_hashes || !out_n || (n_runs && !runs)) return fail(ctx, MASHGPU_ERR_INVALID, "NULL argument");
    if (n_units > 0xFFFFFFF0ull) return fail(ctx, MASHGPU_ERR_INVALID, "too many units");
    for (uint64_t u = 0; u < n_units; u++)
        if (unit_start[u + 1] < unit_start[u]) return fail(ctx, MASHGPU_ERR_INVALID, "unit_start must be ascending");
    if (unit_start[n_units] > stream_len) return fail(ctx, MASHGPU_ERR_INVALID, "unit_start exceeds stream_len");
    MG_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint32_t s = params->sketch_size;
    // waves of whole units, each starting at the 32-position group that holds its first unit's first position
    struct PWave { uint64_t u0, u1, g0, g1; };      // units [u0, u1), groups [g0, g1)
    const WaveLimits lim = wave_limits(s);
    std::vector<PWave> waves;
    for (uint64_t u = 0; u < n_units;) {
        uint64_t v = u + 1;
        while (v < n_units && v - u < lim.units && unit_start[v + 1] - unit_start[u] <= lim.bytes) v++;
        waves.push_back(PWave{u, v, unit_start[u] / 32, (unit_start[v] + 31) / 32});
        u = v;
    }
    uint64_t max_groups = 1, max_units = 1;
    for (auto &w : waves) { max_groups = std::max(max_groups, w.g1 - w.g0); max_units = std::max(max_units, w.u1 - w.u0); }
    const uint64_t max_tiles = (max_groups * 32 + SCAN_TILE - 1) / SCAN_TILE;
    const uint64_t groups_alloc = max_tiles * (SCAN_TILE / 32) + 64;       // tile-padded + halo
    const int nbuf = waves.size() > 1 ? 2 : 1;
    uint64_t *d_codes[2] = {nullptr, nullptr}; uint32_t *d_inval[2] = {nullptr, nullptr};
    for (int b = 0; b < nbuf; b++) {
        d_codes[b] = ctx->sc_codes[b].get<uint64_t>(groups_alloc);
        d_inval[b] = ctx->sc_inval[b].get<uint32_t>(groups_alloc);
        if (!d_codes[b] || !d_inval[b]) return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (packed stream of %llu groups)", (unsigned long long)groups_alloc);
        if (!ctx->pack_copied[b]) MG_CUDA(ctx, cudaEventCreateWithFlags(&ctx->pack_copied[b], cudaEventDisableTiming));
    }
    if (!ctx->pack_stream) MG_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->pack_stream, cudaStreamNonBlocking));
    WaveOutputs outs;
    MG_TRY(wave_outputs(ctx, s, max_units, out_hashes, out_counts, out_n, outs));

    std::vector<PackRun> wruns[2];
    std::vector<uint64_t> wstart[2];
    uint64_t run_cursor = 0;        // first run that may still reach into the current wave (runs ascending)
    auto upload = [&](size_t wi) -> int {
        const PWave &w = waves[wi];
        const int b = (int)(wi % nbuf);
        cudaStream_t cs = ctx->pack_stream;
        const uint64_t p0 = w.g0 * 32, p1 = unit_start[w.u1];           // wave-local position = position - p0
        MG_CUDA(ctx, cudaMemcpyAsync(d_codes[b], codes + w.g0, (w.g1 - w.g0) * 8, cudaMemcpyHostToDevice, cs));
        MG_CUDA(ctx, cudaMemsetAsync(d_inval[b], 0, groups_alloc * 4, cs));
        std::vector<PackRun> &R = wruns[b];
        R.clear();
        if (unit_start[w.u0] > p0) R.push_back(PackRun{0, unit_start[w.u0] - p0});       // the tail of the previous unit in the first group
        while (run_cursor < n_runs && runs[2 * run_cursor] + runs[2 * run_cursor + 1] <= unit_start[w.u0]) run_cursor++;
        for (uint64_t r = run_cursor; r < n_runs && runs[2 * r] < p1; r++) {
            const uint64_t a = std::max(runs[2 * r], unit_start[w.u0]), e = std::min(runs[2 * r] + runs[2 * r + 1], p1);
            if (e > a) R.push_back(PackRun{a - p0, e - a});
        }
        R.push_back(PackRun{p1 - p0, groups_alloc * 32 - (p1 - p0)});                   // everything past the wave's last unit
        PackRun *d_runs = ctx->sc_runs[b].get<PackRun>(R.size());
        if (!d_runs) return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (invalid runs)");
        MG_CUDA(ctx, cudaMemcpyAsync(d_runs, R.data(), R.size() * sizeof(PackRun), cudaMemcpyHostToDevice, cs));
        const unsigned blocks = (unsigned)std::min<uint64_t>((R.size() * 32 + 255) / 256, 148 * 16);
        apply_runs_kernel<<<std::max(1u, blocks), 256, 0, cs>>>(d_runs, R.size(), d_inval[b]);
        ctx->kernel_launches++;
        MG_CUDA(ctx, cudaGetLastError());
        MG_CUDA(ctx, cudaEventRecord(ctx->pack_copied[b], cs));
        wstart[b].resize(w.u1 - w.u0 + 1);
        for (uint64_t u = w.u0; u <= w.u1; u++) wstart[b][u - w.u0] = unit_start[u] - p0;
        return MASHGPU_OK;
    };
    MG_TRY(upload(0));
    int rc = MASHGPU_OK;
    for (size_t wi = 0; wi < waves.size() && rc == MASHGPU_OK; wi++) {
        const PWave &w = waves[wi];
        const int b = (int)(wi % nbuf);
        if (wi + 1 < waves.size()) {
            // buffer (wi+1)%2 was last read by the kernels of wave wi-1 (synchronised below); its run list by upload(wi-1)
            if (wi >= 1) MG_CUDA(ctx, cudaEventSynchronize(ctx->pack_copied[(wi + 1) % nbuf]));
            rc = upload(wi + 1);
            if (rc != MASHGPU_OK) break;
        }
        MG_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->pack_copied[b], 0));
        SketchStream S;
        S.d_codes = d_codes[b]; S.d_inval = d_inval[b]; S.unit_start = wstart[b].data(); S.n_units = w.u1 - w.u0;
        rc = sketch_wave(ctx, params, S, w.u0, outs);
    }
    cudaStreamSynchronize(ctx->pack_stream);
    return rc;
}

// ---------------------------------------------------------------------------------------------------------
// `mash sketch -r -m -c`: the order-dependent stop at a target coverage, found exactly.
//
// MinHashHeap::tryInsert only looks at a k-mer when the heap is not full or its hash is below the heap's top (MinHashHeap.cpp:70-74),
// and once the heap is full the top never rises.  So the exact top at a stream position P (the largest hash of the ordinary
// bottom-s(-m) sketch of the prefix [0, P), computed by the normal kernels) bounds every k-mer after P that can still change the
// heap.  Prefixes at record boundaries near total / 2^j give position bands with a threshold each (the first band, and any
// band that starts before the heap is full, keeps everything); one more scan collects the k-mers at or below their band's
// threshold as events {position, hash}; sorted by position they are replayed through the reference's heap logic by
// reads_replay_kernel -- a faithful, sequential restatement of MinHashHeap::tryInsert (MinHashHeap.cpp:68-146) with the stop
// test of Sketch.cpp:1258-1262 at every read boundary.  A few 10^5 events for a read set of any size.
// ---------------------------------------------------------------------------------------------------------
namespace mashgpu {

struct ReplayMap { uint64_t *key; uint32_t *cnt; uint64_t mask; };     // open addressing, cnt == 0 marks a free slot

__device__ __forceinline__ uint64_t rm_slot(const ReplayMap &m, uint64_t key) { return ((key * 0x9E3779B97F4A7C15ULL) >> 11) & m.mask; }
__device__ uint32_t *rm_find(const ReplayMap &m, uint64_t key)
{
    uint64_t i = rm_slot(m, key);
    while (m.cnt[i]) {
        if (m.key[i] == key) return &m.cnt[i];
        i = (i + 1) & m.mask;
    }
    return nullptr;
}
__device__ void rm_insert_new(const ReplayMap &m, uint64_t key, uint32_t cnt)
{
    uint64_t i = rm_slot(m, key);
    while (m.cnt[i]) i = (i + 1) & m.mask;
    m.key[i] = key; m.cnt[i] = cnt;
}
__device__ void rm_erase(const ReplayMap &m, uint64_t key)      // backward-shift deletion
{
    uint64_t i = rm_slot(m, key);
    while (m.cnt[i] && m.key[i] != key) i = (i + 1) & m.mask;
    if (!m.cnt[i]) return;
    uint64_t j = i;
    for (;;) {
        j = (j + 1) & m.mask;
        if (!m.cnt[j]) break;
        const uint64_t k = rm_slot(m, m.key[j]);
        const bool between = (i <= j) ? (i < k && k <= j) : (i < k || k <= j);
        if (!between) { m.key[i] = m.key[j]; m.cnt[i] = m.cnt[j]; i = j; }
    }
    m.cnt[i] = 0;
}
__device__ void rh_push(uint64_t *heap, uint64_t &n, uint64_t v)     // binary max-heap
{
    uint64_t i = n++;
    while (i > 0) {
        const uint64_t p = (i - 1) / 2;
        if (heap[p] >= v) break;
        heap[i] = heap[p]; i = p;
    }
    heap[i] = v;
}
__device__ void rh_pop(uint64_t *heap, uint64_t &n)
{
    const uint64_t v = heap[--n];
    uint64_t i = 0;
    for (;;) {
        uint64_t c = 2 * i + 1;
        if (c >= n) break;
        if (c + 1 < n && heap[c + 1] > heap[c]) c++;
        if (heap[c] <= v) break;
        heap[i] = heap[c]; i = c;
    }
    if (n) heap[i] = v;
}

// One thread replays the events.  acc = hashes + hashesQueue, pend = hashesPending + hashesQueuePending of MinHashHeap.
__global__ void reads_replay_kernel(const uint64_t *ev_pos, const uint64_t *ev_hash, uint64_t n_ev, const uint64_t *rec_end, uint64_t n_rec,
                                    uint32_t s, uint32_t m, double target_cov,
                                    ReplayMap acc, uint64_t *acc_heap, ReplayMap pend, uint64_t *pend_heap,
                                    uint64_t *out_hashes, uint32_t *out_counts, uint32_t *out_n, uint64_t *out_used)
{
    if (blockIdx.x || threadIdx.x) return;
    uint64_t size = 0, heap_n = 0, pend_n = 0, msum = 0;
    uint64_t rec = 0, cur = ~0ull, used = n_rec;
    bool stopped = false;
    for (uint64_t e = 0; e <= n_ev && !stopped; e++) {
        uint64_t r = ~0ull;
        if (e < n_ev) {
            const uint64_t pos = ev_pos[e];
            while (rec < n_rec && rec_end[rec] <= pos) rec++;
            r = rec;
        }
        if (cur != ~0ull && r != cur) {                     // record `cur` is complete: Sketch.cpp:1258-1262
            if (size && (double)msum / (double)size >= target_cov) { used = cur + 1; stopped = true; break; }
        }
        if (e == n_ev) break;
        cur = r;
        const uint64_t hash = ev_hash[e];
        if (!(size < s || hash < acc_heap[0])) continue;    // MinHashHeap.cpp:70-74
        uint32_t *c = rm_find(acc, hash);
        if (!c) {
            uint32_t *pc = m > 1 ? rm_find(pend, hash) : nullptr;
            const uint64_t pending = pc ? *pc : 0;
            if (m == 1 || pending == m - 1) {               // :96-108
                rm_insert_new(acc, hash, m);
                rh_push(acc_heap, heap_n, hash);
                size++; msum += m;
                if (m > 1 && pc) rm_erase(pend, hash);
            } else if (!pc) {                               // :110-118
                rh_push(pend_heap, pend_n, hash);
                rm_insert_new(pend, hash, 1);
            } else (*pc)++;
        } else { (*c)++; msum++; }                          // :120-124
        if (size > s) {                                     // :126-144
            const uint64_t top = acc_heap[0];
            uint32_t *tc = rm_find(acc, top);
            msum -= tc ? *tc : 0;
            rm_erase(acc, top);
            while (pend_n > 0 && top < pend_heap[0]) {
                if (rm_find(pend, pend_heap[0])) rm_erase(pend, pend_heap[0]);
                rh_pop(pend_heap, pend_n);
            }
            rh_pop(acc_heap, heap_n);
            size--;
        }
    }
    // toHashList: ascending hashes + counts (HashSet.cpp:78-118); popping the max-heap yields them in descending order
    *out_n = (uint32_t)size;
    *out_used = used;
    for (uint64_t i = size; i-- > 0;) {
        const uint64_t v = acc_heap[0];
        out_hashes[i] = v;
        if (out_counts) { const uint32_t *c = rm_find(acc, v); out_counts[i] = c ? *c : 0; }
        rh_pop(acc_heap, heap_n);
    }
}

}  // namespace mashgpu

extern "C" int mashgpu_sketch_reads(mashgpu_ctx *ctx, const mashgpu_sketch_params *params,
                                    uint64_t n_records, const char *const *seq, const uint64_t *len,
                                    uint64_t *out_hashes, uint32_t *out_counts, uint32_t *out_n, uint64_t *out_records_used)
{
    if (!ctx) return MASHGPU_ERR_INVALID;
    MG_TRY(validate_sketch_params(ctx, params));
    if (!out_hashes || !out_n || !out_records_used) return fail(ctx, MASHGPU_ERR_INVALID, "NULL output");
    if (n_records && (!seq || !len)) return fail(ctx, MASHGPU_ERR_INVALID, "seq/len is NULL");
    if (!is_dna_alphabet(params)) return fail(ctx, MASHGPU_ERR_UNSUPPORTED, "reads mode with a target coverage is only provided for the alphabet {A,C,G,T}");
    MG_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const uint32_t s = params->sketch_size;
    const uint64_t k = (uint64_t)params->kmer_size;
    const uint32_t mc = std::max(1u, params->min_copies);
    *out_n = 0; *out_records_used = 0;
    // kept records -> one flat device stream (record, separator, record, ...) + the end offset of every kept record
    std::vector<uint64_t> rec_end;
    uint64_t total = 0;
    for (uint64_t r = 0; r < n_records; r++)
        if (len[r] >= k) { total += len[r] + 1; rec_end.push_back(total - 1); }
    const uint64_t n_rec = rec_end.size();
    if (n_rec == 0) return MASHGPU_OK;
    DevBuf<uint8_t> d_stream; DevBuf<uint64_t> d_hashes, d_rec_end; DevBuf<uint32_t> d_n, d_counts;
    if (d_stream.alloc(((total + 15) / 16) * 16 + 64) != cudaSuccess || d_hashes.alloc(s) != cudaSuccess || d_n.alloc(1) != cudaSuccess ||
        d_counts.alloc(s) != cudaSuccess || d_rec_end.alloc(n_rec) != cudaSuccess)
        return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (read set of %llu B)", (unsigned long long)total);
    {
        const size_t chunk = 64ull << 20;
        PinnedBuf<uint8_t> stage[2];
        if (stage[0].alloc(chunk) != cudaSuccess || stage[1].alloc(chunk) != cudaSuccess) return fail(ctx, MASHGPU_ERR_NOMEM, "out of pinned host memory");
        cudaEvent_t done[2];
        MG_CUDA(ctx, cudaEventCreateWithFlags(&done[0], cudaEventDisableTiming));
        MG_CUDA(ctx, cudaEventCreateWithFlags(&done[1], cudaEventDisableTiming));
        uint64_t off = 0, fill = 0, base = 0;
        int b = 0;
        bool used_ev[2] = {false, false};
        auto flush = [&]() -> cudaError_t {
            if (!fill) return cudaSuccess;
            cudaError_t e = cudaMemcpyAsync(d_stream.p + base, stage[b].p, fill, cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) return e;
            e = cudaEventRecord(done[b], st);
            used_ev[b] = true;
            b ^= 1;
            if (used_ev[b]) cudaEventSynchronize(done[b]);
            base += fill; fill = 0;
            return e;
        };
        cudaError_t e = cudaSuccess;
        for (uint64_t r = 0; r < n_records && e == cudaSuccess; r++) {
            if (len[r] < k) continue;
            uint64_t done_r = 0;
            while (done_r < len[r] + 1 && e == cudaSuccess) {            // the record's bytes, then its separator
                const uint64_t room = chunk - fill, want = len[r] + 1 - done_r;
                const uint64_t take = std::min(room, want);
                const uint64_t from_seq = done_r < len[r] ? std::min(take, len[r] - done_r) : 0;
                if (from_seq) memcpy(stage[b].p + fill, seq[r] + done_r, from_seq);
                if (take > from_seq) stage[b].p[fill + from_seq] = 0;
                fill += take; done_r += take; off += take;
                if (fill == chunk) e = flush();
            }
        }
        if (e == cudaSuccess) e = flush();
        cudaStreamSynchronize(st);
        cudaEventDestroy(done[0]); cudaEventDestroy(done[1]);
        if (e != cudaSuccess) return fail(ctx, MASHGPU_ERR_CUDA, "upload of the read set failed: %s", cudaGetErrorString(e));
        (void)off;
    }
    MG_CUDA(ctx, cudaMemcpyAsync(d_rec_end.p, rec_end.data(), n_rec * 8, cudaMemcpyHostToDevice, st));
    auto prefix_sketch = [&](uint64_t end, bool want_counts) -> int {        // ordinary sketch of the stream prefix [0, end)
        uint64_t us[2] = {0, end};
        SketchStream S;
        S.d_stream = d_stream.p; S.unit_start = us; S.n_units = 1;
        return sketch_stream_core(ctx, params, S, d_hashes.p, want_counts ? d_counts.p : nullptr, d_n.p, st, nullptr);
    };
    auto emit_result = [&](uint64_t used) -> int {
        uint32_t n = 0;
        MG_CUDA(ctx, cudaMemcpyAsync(&n, d_n.p, 4, cudaMemcpyDeviceToHost, st));
        MG_CUDA(ctx, cudaStreamSynchronize(st));
        if (n) MG_CUDA(ctx, cudaMemcpyAsync(out_hashes, d_hashes.p, n * 8ull, cudaMemcpyDeviceToHost, st));
        if (n && out_counts) MG_CUDA(ctx, cudaMemcpyAsync(out_counts, d_counts.p, n * 4ull, cudaMemcpyDeviceToHost, st));
        MG_CUDA(ctx, cudaStreamSynchronize(st));
        *out_n = n; *out_records_used = used;
        return MASHGPU_OK;
    };
    if (!(params->target_cov > 0)) {
        MG_TRY(prefix_sketch(total, out_counts != nullptr));
        return emit_result(n_rec);
    }
    // ---- position bands: record boundaries near total / 2^j, down to ~2^20 positions; threshold = exact top of the heap at the band's start
    std::vector<uint64_t> band_start(1, 0), band_t(1, EMPTY_KEY);
    {
        std::vector<uint64_t> cuts;
        for (uint64_t target = total / 2; target >= (1ull << 20); target /= 2) {
            auto it = std::upper_bound(rec_end.begin(), rec_end.end(), target);     // first record that ends after the target
            if (it == rec_end.begin()) break;
            const uint64_t cut = *(it - 1) + 1;                                     // the position after that record's separator
            if (cuts.empty() || cut < cuts.back()) cuts.push_back(cut);
        }
        std::reverse(cuts.begin(), cuts.end());
        for (uint64_t cut : cuts) {
            if (cut <= band_start.back()) continue;
            MG_TRY(prefix_sketch(cut, false));
            uint32_t n = 0; uint64_t top = EMPTY_KEY;
            MG_CUDA(ctx, cudaMemcpyAsync(&n, d_n.p, 4, cudaMemcpyDeviceToHost, st));
            MG_CUDA(ctx, cudaStreamSynchronize(st));
            if (n == s) {
                MG_CUDA(ctx, cudaMemcpyAsync(&top, d_hashes.p + (s - 1), 8, cudaMemcpyDeviceToHost, st));
                MG_CUDA(ctx, cudaStreamSynchronize(st));
            }
            band_start.push_back(cut);
            band_t.push_back(n == s ? top : EMPTY_KEY);                             // heap not full yet: its gate is open
        }
    }
    // ---- events
    const uint32_t n_bands = (uint32_t)band_start.size();
    const uint64_t ev_cap = 1ull << 24;
    DevBuf<uint64_t> d_bstart, d_bt, ev_pos, ev_hash, ev_pos2, ev_hash2, d_tmax; DevBuf<unsigned long long> ev_count; DevBuf<uint8_t> tmp;
    const uint64_t ntiles = (total + SCAN_TILE - 1) / SCAN_TILE;
    if (d_bstart.alloc(n_bands + 1) != cudaSuccess || d_bt.alloc(n_bands) != cudaSuccess || ev_pos.alloc(ev_cap) != cudaSuccess || ev_hash.alloc(ev_cap) != cudaSuccess ||
        ev_pos2.alloc(ev_cap) != cudaSuccess || ev_hash2.alloc(ev_cap) != cudaSuccess || ev_count.alloc(1) != cudaSuccess || d_tmax.alloc(ntiles) != cudaSuccess)
        return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (event buffers)");
    band_start.push_back(total);
    MG_CUDA(ctx, cudaMemcpyAsync(d_bstart.p, band_start.data(), (n_bands + 1) * 8ull, cudaMemcpyHostToDevice, st));
    MG_CUDA(ctx, cudaMemcpyAsync(d_bt.p, band_t.data(), n_bands * 8ull, cudaMemcpyHostToDevice, st));
    MG_CUDA(ctx, cudaMemsetAsync(ev_count.p, 0, 8, st));
    tile_tmax_kernel<<<(unsigned)((ntiles + 255) / 256), 256, 0, st>>>(d_bstart.p, n_bands, d_bt.p, total, 0, ntiles, d_tmax.p);
    ScanArgs a = scan_args(params, d_stream.p, nullptr, nullptr, total);
    a.tile_begin = 0; a.tile_end = ntiles; a.tile_tmax = d_tmax.p;
    a.mode = SCAN_EVENTS; a.min_copies = 1;
    a.unit_start = d_bstart.p; a.n_units = n_bands; a.unit_t = d_bt.p;
    a.ev_pos = ev_pos.p; a.ev_hash = ev_hash.p; a.ev_count = ev_count.p; a.ev_capacity = ev_cap;
    MG_TRY(launch_scan(ctx, params, a, st));
    unsigned long long n_ev = 0;
    MG_CUDA(ctx, cudaMemcpyAsync(&n_ev, ev_count.p, 8, cudaMemcpyDeviceToHost, st));
    MG_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->kernel_launches++;
    if (n_ev > ev_cap)
        return fail(ctx, MASHGPU_ERR_UNSUPPORTED, "-c: %llu k-mers could pass the heap's gate (more than %llu): the heap fills too slowly on this read set "
                                                  "(very low coverage or a high -m)", n_ev, (unsigned long long)ev_cap);
    if (n_ev) {
        size_t tb = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tb, ev_pos.p, ev_pos2.p, ev_hash.p, ev_hash2.p, (int)n_ev, 0, 64, st);
        if (tmp.alloc(tb) != cudaSuccess) return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (sort scratch)");
        MG_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp.p, tb, ev_pos.p, ev_pos2.p, ev_hash.p, ev_hash2.p, (int)n_ev, 0, 64, st));
        ctx->kernel_launches += 8;
    }
    // ---- replay
    uint64_t cap_a = 16, cap_p = 16;
    while (cap_a < 4ull * (s + 2)) cap_a <<= 1;
    while (cap_p < 2 * n_ev + 16) cap_p <<= 1;
    DevBuf<uint64_t> a_key, a_heap, p_key, p_heap, d_used; DevBuf<uint32_t> a_cnt, p_cnt;
    if (a_key.alloc(cap_a) != cudaSuccess || a_cnt.alloc(cap_a) != cudaSuccess || a_heap.alloc(s + 2) != cudaSuccess || p_key.alloc(cap_p) != cudaSuccess ||
        p_cnt.alloc(cap_p) != cudaSuccess || p_heap.alloc(n_ev + 2) != cudaSuccess || d_used.alloc(1) != cudaSuccess)
        return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory (replay tables)");
    MG_CUDA(ctx, cudaMemsetAsync(a_cnt.p, 0, cap_a * 4, st));
    MG_CUDA(ctx, cudaMemsetAsync(p_cnt.p, 0, cap_p * 4, st));
    ReplayMap acc{a_key.p, a_cnt.p, cap_a - 1}, pend{p_key.p, p_cnt.p, cap_p - 1};
    reads_replay_kernel<<<1, 32, 0, st>>>(ev_pos2.p, ev_hash2.p, n_ev, d_rec_end.p, n_rec, s, mc, params->target_cov, acc, a_heap.p, pend, p_heap.p,
                                          d_hashes.p, d_counts.p, d_n.p, d_used.p);
    ctx->kernel_launches++;
    MG_CUDA(ctx, cudaGetLastError());
    uint64_t used = 0;
    MG_CUDA(ctx, cudaMemcpyAsync(&used, d_used.p, 8, cudaMemcpyDeviceToHost, st));
    MG_CUDA(ctx, cudaStreamSynchronize(st));
    return emit_result(used);
}

extern "C" int mashgpu_host_pack(const mashgpu_sketch_params *params, uint64_t n_records, const char *const *seq, const uint64_t *len,
                                 int threads, uint64_t *codes, uint64_t *runs, uint64_t runs_capacity, uint64_t *n_runs)
{
    if (!params || !codes || !n_runs || (n_records && (!seq || !len))) return MASHGPU_ERR_INVALID;
    std::vector<PackSegment> segs;
    uint64_t off = 0;
    for (uint64_t r = 0; r < n_records; r++) {
        segs.push_back(PackSegment{(const uint8_t *)seq[r], off, len[r]});
        off += len[r] + 1;
    }
    std::vector<PackRun> found;
    pack_stream(segs.data(), segs.size(), off, params->preserve_case, threads, codes, found);
    *n_runs = found.size();
    for (uint64_t i = 0; i < found.size() && i < runs_capacity; i++) { runs[2 * i] = found[i].start; runs[2 * i + 1] = found[i].len; }
    return MASHGPU_OK;
}

extern "C" int mashgpu_hash_windows(mashgpu_ctx *ctx, const mashgpu_sketch_params *params,
                                    const char *seq, uint64_t len, uint64_t *out_hash, uint8_t *out_valid)
{
    if (!ctx) return MASHGPU_ERR_INVALID;
    MG_TRY(validate_sketch_params(ctx, params));
    const uint64_t k = (uint64_t)params->kmer_size;
    if (len < k) return MASHGPU_OK;
    if (!seq || !out_hash || !out_valid) return fail(ctx, MASHGPU_ERR_INVALID, "NULL argument");
    MG_CUDA(ctx, cudaSetDevice(ctx->device));
    const uint64_t nwin = len - k + 1;
    DevBuf<uint8_t> d_seq, d_valid; DevBuf<uint64_t> d_hash;
    const uint64_t padded = ((len + 15) / 16) * 16;
    if (d_seq.alloc(padded) != cudaSuccess || d_valid.alloc(len) != cudaSuccess || d_hash.alloc(len) != cudaSuccess)
        return fail(ctx, MASHGPU_ERR_NOMEM, "out of device memory");
    cudaStream_t st = ctx->stream;
    MG_CUDA(ctx, cudaMemcpyAsync(d_seq.p, seq, len, cudaMemcpyHostToDevice, st));
    MG_CUDA(ctx, cudaMemsetAsync(d_valid.p, 0, len, st));
    MG_CUDA(ctx, cudaMemsetAsync(d_hash.p, 0, len * 8, st));
    ScanArgs a = scan_args(params, d_seq.p, nullptr, nullptr, len);
    a.tile_begin = 0; a.tile_end = (len + SCAN_TILE - 1) / SCAN_TILE;
    a.coarse_t = EMPTY_KEY;
    a.mode = SCAN_DUMP;
    a.out_hash = d_hash.p; a.out_valid = d_valid.p;
    MG_TRY(launch_scan(ctx, params, a, st));
    MG_CUDA(ctx, cudaMemcpyAsync(out_hash, d_hash.p, nwin * 8, cudaMemcpyDeviceToHost, st));
    MG_CUDA(ctx, cudaMemcpyAsync(out_valid, d_valid.p, nwin, cudaMemcpyDeviceToHost, st));
    MG_CUDA(ctx, cudaStreamSynchronize(st));
    return MASHGPU_OK;
}
