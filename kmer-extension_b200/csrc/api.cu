// api.cu -- the C ABI of libkmer_cuda.so (include/kmer_cuda.h): context, workspaces, error mapping,
// host-buffer batch submit and the device-resident entry points.  No CPU compute path exists here:
// every operation is a sequence of CUDA kernels; without a device the calls fail.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "kernels.cuh"

using namespace kmer;

namespace {

struct Buf {
    void* p = nullptr;
    size_t cap = 0;
};

struct PinnedBuf {
    void* p;
    size_t cap;
    bool in_use;
};

enum PendingOp { OP_NONE = 0, OP_EXTRACT, OP_COUNT, OP_MATCH, OP_DECODE, OP_ENCODE, OP_SHARD_PART, OP_SHARD_COUNT, OP_DENSE_TABLE, OP_MERGE,
                 OP_PAIRS_SPECTRUM };

}  // namespace

struct kmer_cuda_ctx {
    DeviceInfo di{};
    cudaStream_t stream = nullptr;
    kmer_cuda_error err{};
    uint64_t launches = 0;
    DevStatus* d_status = nullptr;
    DevStatus* h_status = nullptr;  // pinned
    // host-buffer submit: copies run on their own streams beside the kernels (kmer_cuda_submit_count*)
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[8] = {}, ev_leaf[16] = {}, ev_off = nullptr;
    DevStatus* h_ring = nullptr;    // pinned: status snapshots behind every group of buckets
    // device workspaces, grown on demand and kept between calls
    Buf seq, off, mask, tile_row, table, consts, ops, codes, pairs, bits, hits, lens, text, fill, recs, spill, failed, seg, segfill, hist;
    uint64_t merge_slots = 0;     // table slots of the merge in progress (kmer_cuda_dev_merge_*)
    uint64_t last_tier2 = 0;      // k-mers counted by the tier-2 kernel in the last count
    uint64_t last_overflow = 0;   // k-mers the partition counter could not place (batch was recounted)
    std::vector<PinnedBuf> pinned;
    // the operation kmer_cuda_dev_finish() has to report on
    PendingOp pending = OP_NONE;
    uint64_t p_n_bases = 0, p_n_rows = 0;
    int p_k = 0;
    uint64_t p_expected_kmers = 0;
    // a partition count whose tiers overflowed is recounted by kmer_cuda_dev_finish through the global hash table
    bool p_recountable = false;
    bool p_chained = false;       // shard count chained to its partition: finish() also reports the partition's input errors
    const char* p_seq = nullptr;
    const uint64_t* p_off = nullptr;
    kmer_count_pair* p_pairs = nullptr;
    uint64_t p_pairs_cap = 0;
    // ... or, in the spectrum result format, re-zeroes the histogram and rebins into it (the tail cursor is DevStatus::n_distinct)
    bool p_spectrum = false;
    bool p_canonical = false;     // ... and counts canonical k-mers (kmer_cuda_*_count_canonical*)
    uint64_t* p_hist = nullptr;
    uint64_t p_hist_len = 0;
    kmer_count_pair* p_tail = nullptr;
    uint64_t p_tail_cap = 0;
    // optional phase timing (bench.py's per-kernel roofline): events recorded after each phase
    bool profiling = false;
    std::vector<cudaEvent_t> ev_pool;
    std::vector<const char*> ev_names;   // ev_names[i] = phase that ENDS at event i ("" for the start mark)
    size_t ev_used = 0;
    std::vector<float> phase_ms;
    std::vector<const char*> phase_names;
};

static void mark(kmer_cuda_ctx* c, cudaStream_t st, const char* name) {
    if (!c->profiling) return;
    if (c->ev_used == c->ev_pool.size()) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return;
        c->ev_pool.push_back(e);
        c->ev_names.push_back("");
    }
    c->ev_names[c->ev_used] = name;
    cudaEventRecord(c->ev_pool[c->ev_used++], st);
}

static kmer_cuda_error g_init_error;  // error of a failed kmer_cuda_init (no ctx to hold it)

// ------------------------------------------------------------------------------------------------
// errors

static int set_error(kmer_cuda_error* e, int status, const char* sqlstate, const char* msg, const char* detail,
                     int64_t row) {
    e->status = status;
    snprintf(e->sqlstate, sizeof(e->sqlstate), "%s", sqlstate);
    snprintf(e->message, sizeof(e->message), "%s", msg);
    snprintf(e->detail, sizeof(e->detail), "%s", detail ? detail : "");
    e->row = row;
    return status;
}

// the reference's own errors: same SQLSTATE, same text (kmer.c:33-36,117-119,151-153,179-181,311-313)
static int ref_error(kmer_cuda_error* e, int status, int64_t row) {
    switch (status) {
        case KMER_ERR_INVALID_DNA:
            return set_error(e, status, "22P02", "Invalid DNA Sequence",
                             "Valid characters are A, C, G, T (case-insensitive).", row);
        case KMER_ERR_KMER_TOO_LONG:
            return set_error(e, status, "22001", "KMer Sequence larger than length 32", "", row);
        case KMER_ERR_INVALID_QKMER:
            return set_error(e, status, "22P02", "Invalid QKMer Sequence", "", row);
        case KMER_ERR_INVALID_K:
            return set_error(e, status, "22023", "Invalid KMER Length", "", row);
        case KMER_ERR_QKMER_TOO_LONG:
            return set_error(e, status, "22001", "QKMer Sequence larger than length 32", "", row);
    }
    return set_error(e, status, "XX000", "kmer_cuda: internal error", "", row);
}

static int cuda_error(kmer_cuda_ctx* c, cudaError_t ce, const char* what) {
    char msg[160];
    snprintf(msg, sizeof(msg), "kmer_cuda: %s failed: %s", what, cudaGetErrorString(ce));
    bool oom = ce == cudaErrorMemoryAllocation;
    return set_error(c ? &c->err : &g_init_error, oom ? KMER_ERR_OOM : KMER_ERR_CUDA, oom ? "53200" : "XX000", msg, "", -1);
}

static int bad_arg(kmer_cuda_ctx* c, const char* what) {
    char msg[160];
    snprintf(msg, sizeof(msg), "kmer_cuda: bad argument: %s", what);
    return set_error(&c->err, KMER_ERR_BAD_ARGUMENT, "XX000", msg, "", -1);
}

#define CU(call, what)                                      \
    do {                                                    \
        cudaError_t ce__ = (call);                          \
        if (ce__ != cudaSuccess) return cuda_error(c, ce__, what); \
    } while (0)

// ------------------------------------------------------------------------------------------------
// memory

static int ws(kmer_cuda_ctx* c, Buf& b, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (b.cap >= bytes) return KMER_OK;
    if (b.p) {
        cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
    }
    size_t want = (bytes + 255) & ~(size_t)255;
    cudaError_t ce = cudaMalloc(&b.p, want);
    if (ce != cudaSuccess) {
        b.p = nullptr;
        cudaGetLastError();
        return cuda_error(c, ce, "cudaMalloc");
    }
    b.cap = want;
    return KMER_OK;
}

static void* pinned_get(kmer_cuda_ctx* c, size_t bytes) {
    if (bytes == 0) bytes = 16;
    int best = -1;
    for (size_t i = 0; i < c->pinned.size(); i++)
        if (!c->pinned[i].in_use && c->pinned[i].cap >= bytes && (best < 0 || c->pinned[i].cap < c->pinned[best].cap))
            best = (int)i;
    if (best >= 0) {
        c->pinned[best].in_use = true;
        return c->pinned[best].p;
    }
    // drop idle buffers that are too small before growing (keeps the pinned footprint bounded)
    for (size_t i = 0; i < c->pinned.size();) {
        if (!c->pinned[i].in_use) {
            cudaFreeHost(c->pinned[i].p);
            c->pinned.erase(c->pinned.begin() + i);
        } else
            i++;
    }
    void* p = nullptr;
    cudaError_t ce = cudaHostAlloc(&p, bytes, cudaHostAllocDefault);
    if (ce != cudaSuccess) {
        cudaGetLastError();
        cuda_error(c, ce, "cudaHostAlloc");
        return nullptr;
    }
    c->pinned.push_back({p, bytes, true});
    return p;
}

static bool is_device_accessible_host(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

// ------------------------------------------------------------------------------------------------
// small kernels of the API layer

__global__ void status_reset_kernel(DevStatus* s) {
    s->bad_char_pos = kNoError;
    s->short_row = kNoError;
    s->n_kmers = 0;
    s->n_distinct = 0;
    s->n_overflow = 0;
    s->special_count = 0;
    s->out_overflow = 0;
    s->pad = kNoError;
    s->n_spill = 0;
    s->n_failed = 0;
    s->failed_kmers = 0;
    s->n_unique = 0;
    s->t2_mode = 0;
    s->t2_slots = 0;
}

// sharded counting: the count that follows a partition on the same stream WITHOUT a finish in between keeps what the partition
// found in the input (first bad character / short row / overflowed segments); one finish at the end reports everything
__global__ void status_reset_keep_input_kernel(DevStatus* s) {
    s->n_kmers = 0;
    s->n_distinct = 0;
    s->special_count = 0;
    s->out_overflow = 0;
    s->n_spill = 0;
    s->n_failed = 0;
    s->failed_kmers = 0;
    s->n_unique = 0;
    s->t2_mode = 0;
    s->t2_slots = 0;
}

// pad := row containing bad_char_pos (so the host never needs the offsets)
__global__ void resolve_bad_row_kernel(DevStatus* s, const uint64_t* off, uint64_t n_rows) {
    unsigned long long pos = s->bad_char_pos;
    if (pos == kNoError) return;
    uint64_t lo = 0, hi = n_rows;
    while (lo < hi) {
        uint64_t mid = (lo + hi) >> 1;
        if (off[mid] <= pos) lo = mid + 1; else hi = mid;
    }
    s->pad = lo - 1;
}

// ------------------------------------------------------------------------------------------------
// constants: kmer / qkmer literals -> MatchConst   (kmer_in kmer.c:109-129, qkmer_in kmer.c:141-190, match() kmer.h:21-53)

static int base_of(int ch) {
    switch (ch | 0x20) {
        case 'a': return 0;
        case 'c': return 1;
        case 'g': return 2;
        case 't': return 3;
    }
    return -1;
}

static int iupac_set(int ch) {  // bit b set <=> base b admitted ; -1 invalid letter
    if (!((ch >= 'A' && ch <= 'Z') || (ch >= 'a' && ch <= 'z'))) return -1;
    switch (ch | 0x20) {
        case 'a': return 1;
        case 'c': return 2;
        case 'g': return 4;
        case 't': return 8;
        case 'u': return 0;  // accepted by qkmer_in (kmer.c:165) but matches nothing (kmer.h:50-51)
        case 'r': return 1 | 4;
        case 'y': return 2 | 8;
        case 'k': return 4 | 8;
        case 'm': return 1 | 2;
        case 's': return 4 | 2;
        case 'w': return 1 | 8;
        case 'b': return 2 | 4 | 8;
        case 'd': return 1 | 4 | 8;
        case 'h': return 1 | 2 | 8;
        case 'v': return 1 | 2 | 4;
        case 'n': return 15;
    }
    return -1;
}

static int compile_const(kmer_cuda_ctx* c, int op, const char* text, int64_t idx, MatchConst* out) {
    memset(out, 0, sizeof(*out));
    if (!text) return bad_arg(c, "NULL constant (the SQL functions are STRICT: filter NULLs in the caller)");
    size_t len = strlen(text);
    if (op == KMER_OP_CONTAINS) {
        if (len > KMER_CUDA_MAX_K) return ref_error(&c->err, KMER_ERR_QKMER_TOO_LONG, idx);
        uint64_t pl[4] = {0, 0, 0, 0};
        for (size_t i = 0; i < len; i++) {
            int s = iupac_set((unsigned char)text[i]);
            if (s < 0) return ref_error(&c->err, KMER_ERR_INVALID_QKMER, idx);
            size_t j = len - 1 - i;
            for (int b = 0; b < 4; b++)
                if (s & (1 << b)) pl[b] |= 1ull << j;
        }
        out->m0 = pl[0]; out->m1 = pl[1]; out->m2 = pl[2]; out->m3 = pl[3];
    } else if (op == KMER_OP_EQUALS || op == KMER_OP_STARTS_WITH) {
        if (len > KMER_CUDA_MAX_K) return ref_error(&c->err, KMER_ERR_KMER_TOO_LONG, idx);
        uint64_t v = 0;
        for (size_t i = 0; i < len; i++) {
            int b = base_of((unsigned char)text[i]);
            if (b < 0) return ref_error(&c->err, KMER_ERR_INVALID_DNA, idx);
            v = (v << 2) | (uint64_t)b;
        }
        out->code = v;
    } else
        return bad_arg(c, "unknown match op");
    out->len = (uint32_t)len;
    return KMER_OK;
}

// ------------------------------------------------------------------------------------------------
// lifecycle

extern "C" int kmer_cuda_abi_version(void) { return KMER_CUDA_ABI_VERSION; }

extern "C" int kmer_cuda_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int kmer_cuda_init(kmer_cuda_ctx** out, int device) {
    kmer_cuda_ctx* c = nullptr;
    if (!out) return set_error(&g_init_error, KMER_ERR_BAD_ARGUMENT, "XX000", "kmer_cuda: bad argument: ctx", "", -1);
    *out = nullptr;
    int n = kmer_cuda_device_count();
    if (n <= 0)
        return set_error(&g_init_error, KMER_ERR_NO_DEVICE, "XX000",
                         "kmer_cuda: no CUDA device available (this library has no CPU path)", "", -1);
    if (device < 0 || device >= n)
        return set_error(&g_init_error, KMER_ERR_BAD_ARGUMENT, "XX000", "kmer_cuda: bad argument: device index", "", -1);
    CU(cudaSetDevice(device), "cudaSetDevice");
    c = new (std::nothrow) kmer_cuda_ctx();
    if (!c) return set_error(&g_init_error, KMER_ERR_OOM, "53200", "kmer_cuda: out of host memory", "", -1);
    cudaDeviceProp prop;
    cudaError_t ce = cudaGetDeviceProperties(&prop, device);
    if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaMalloc((void**)&c->d_status, sizeof(DevStatus));
    if (ce == cudaSuccess) ce = cudaHostAlloc((void**)&c->h_status, sizeof(DevStatus), cudaHostAllocDefault);
    if (ce != cudaSuccess) {
        int rc = cuda_error(nullptr, ce, "context setup");
        delete c;
        return rc;
    }
    c->di.device = device;
    c->di.sm_count = prop.multiProcessorCount;
    c->di.total_mem = prop.totalGlobalMem;
    if (prop.major < 10) {
        delete c;
        return set_error(&g_init_error, KMER_ERR_NO_DEVICE, "XX000", "kmer_cuda: built for sm_100a (B200) only", "", -1);
    }
    c->err.status = KMER_OK;
    c->err.row = -1;
    *out = c;
    return KMER_OK;
}

static void buf_free(Buf& b) {
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

extern "C" void kmer_cuda_shutdown(kmer_cuda_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->di.device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    Buf* all[] = {&c->seq, &c->off, &c->mask, &c->tile_row, &c->table, &c->consts, &c->ops,
                  &c->codes, &c->pairs, &c->bits, &c->hits, &c->lens, &c->text, &c->fill, &c->recs, &c->spill, &c->failed, &c->seg, &c->segfill, &c->hist};
    for (Buf* b : all) buf_free(*b);
    for (auto& p : c->pinned) cudaFreeHost(p.p);
    for (auto e : c->ev_pool) cudaEventDestroy(e);
    if (c->d_status) cudaFree(c->d_status);
    if (c->h_status) cudaFreeHost(c->h_status);
    if (c->h_ring) cudaFreeHost(c->h_ring);
    for (auto e : c->ev_in) if (e) cudaEventDestroy(e);
    for (auto e : c->ev_leaf) if (e) cudaEventDestroy(e);
    if (c->ev_off) cudaEventDestroy(c->ev_off);
    if (c->s_in) cudaStreamDestroy(c->s_in);
    if (c->s_out) cudaStreamDestroy(c->s_out);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" const kmer_cuda_error* kmer_cuda_last_error(const kmer_cuda_ctx* c) { return c ? &c->err : &g_init_error; }

extern "C" void kmer_cuda_release(kmer_cuda_ctx* c, void* result) {
    if (!c || !result) return;
    for (auto& p : c->pinned)
        if (p.p == result) p.in_use = false;  // kept for reuse; freed at shutdown
}

extern "C" void kmer_cuda_set_profiling(kmer_cuda_ctx* c, int on) {
    if (c) c->profiling = on != 0;
}

extern "C" int kmer_cuda_get_phases(const kmer_cuda_ctx* c, const char** names, float* ms, int capacity) {
    if (!c) return 0;
    int n = (int)c->phase_ms.size();
    for (int i = 0; i < n && i < capacity; i++) {
        if (names) names[i] = c->phase_names[i];
        if (ms) ms[i] = c->phase_ms[i];
    }
    return n;
}

extern "C" uint64_t kmer_cuda_launch_count(const kmer_cuda_ctx* c) { return c ? c->launches : 0; }

extern "C" void kmer_cuda_test_force_window(int w) { partition_force_window(w); }

extern "C" uint64_t kmer_cuda_max_kmers(uint64_t n_bases, uint64_t n_rows, int k) {
    if (k < 1 || k > KMER_CUDA_MAX_K) return 0;
    uint64_t sub = n_rows * (uint64_t)(k - 1);
    return n_bases > sub ? n_bases - sub : 0;
}

// ------------------------------------------------------------------------------------------------
// device-resident operations

// stream argument of the C ABI: NULL = the CUDA default stream (what a caller that never created a
// stream is using); KMER_OWN_STREAM = the context's private stream (used by the submit_* calls).
static const char kOwnStreamTag = 0;                  // its ADDRESS is the sentinel: no CUDA stream handle can equal it
#define KMER_OWN_STREAM ((void*)&kOwnStreamTag)         // ((void*)1 would be cudaStreamLegacy)
static cudaStream_t pick_stream(kmer_cuda_ctx* c, void* stream) {
    return stream == KMER_OWN_STREAM ? c->stream : (cudaStream_t)stream;
}

static int begin_op(kmer_cuda_ctx* c, cudaStream_t st, bool keep_input_findings = false) {
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    if (!keep_input_findings) c->ev_used = 0;
    mark(c, st, keep_input_findings ? "exchange" : "");
    if (keep_input_findings) status_reset_keep_input_kernel<<<1, 1, 0, st>>>(c->d_status);
    else status_reset_kernel<<<1, 1, 0, st>>>(c->d_status);
    c->launches++;
    c->pending = OP_NONE;
    c->p_recountable = false;
    c->p_spectrum = false;
    c->p_canonical = false;
    return KMER_OK;
}

// row mask + short-row check shared by extract and count.  Returns KMER_ERR_INVALID_K immediately for
// k outside 1..32 (generate_kmers, kmer.c:310: `window_size <= 0 || window_size > MAX_KMER_LENGTH`).
static int prepare_rows(kmer_cuda_ctx* c, const uint64_t* d_off, uint64_t n_bases, uint64_t n_rows, int k,
                        cudaStream_t st, ScanArgs* a, const char* d_seq) {
    if (n_rows && (k < 1 || k > KMER_CUDA_MAX_K)) return ref_error(&c->err, KMER_ERR_INVALID_K, 0);
    if ((reinterpret_cast<uintptr_t>(d_seq) & 15) != 0) return bad_arg(c, "d_seq must be 16-byte aligned");
    uint64_t mask_words = (n_bases + 1 + 31) / 32 + MASK_PAD_WORDS;
    int rc = ws(c, c->mask, mask_words * 4);
    if (rc) return rc;
    launch_rows_prepare(d_off, n_rows, n_bases, k, (uint32_t*)c->mask.p, mask_words, c->d_status, st);
    c->launches++;
    mark(c, st, "rows_prepare");
    a->seq = reinterpret_cast<const uint8_t*>(d_seq);
    a->n_bases = n_bases;
    a->row_mask = (const uint32_t*)c->mask.p;
    a->k = k;
    a->status = c->d_status;
    return KMER_OK;
}

extern "C" int kmer_cuda_dev_extract(kmer_cuda_ctx* c, const char* d_seq, uint64_t n_bases, const uint64_t* d_row_off,
                                     uint64_t n_rows, int k, uint64_t* d_codes, uint64_t codes_capacity, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    cudaStream_t st = pick_stream(c, stream);
    int rc = begin_op(c, st);
    if (rc) return rc;
    c->pending = OP_EXTRACT;
    c->p_n_bases = n_bases; c->p_n_rows = n_rows; c->p_k = k;
    c->p_expected_kmers = kmer_cuda_max_kmers(n_bases, n_rows, k);
    if (n_rows == 0 || n_bases == 0) {
        if (n_rows && (k < 1 || k > KMER_CUDA_MAX_K)) return ref_error(&c->err, KMER_ERR_INVALID_K, 0);
        if (n_rows) {  // rows exist but are all empty: len 0 < k
            return ref_error(&c->err, KMER_ERR_INVALID_K, 0);
        }
        return KMER_OK;
    }
    ScanArgs a;
    rc = prepare_rows(c, d_row_off, n_bases, n_rows, k, st, &a, d_seq);
    if (rc) return rc;
    uint64_t n_tiles = (n_bases + TILE - 1) / TILE;
    rc = ws(c, c->tile_row, n_tiles * 4);
    if (rc) return rc;
    launch_tile_row_base(d_row_off, n_rows, n_tiles, (uint32_t*)c->tile_row.p, st);
    mark(c, st, "tile_row_base");
    launch_extract(c->di, a, (const uint32_t*)c->tile_row.p, d_codes, codes_capacity, st);
    mark(c, st, "extract");
    resolve_bad_row_kernel<<<1, 1, 0, st>>>(c->d_status, d_row_off, n_rows);
    c->launches += 3;
    CU(cudaGetLastError(), "extract launch");
    return KMER_OK;
}

struct MarkArg {
    kmer_cuda_ctx* c;
    cudaStream_t st;
};
static void mark_cb(void* arg, const char* name) {
    MarkArg* m = (MarkArg*)arg;
    mark(m->c, m->st, name);
}

static uint64_t next_pow2(uint64_t v) {
    uint64_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

static SpecOut spec_out(uint64_t* d_hist, uint64_t hist_len, kmer_count_pair* d_tail, uint64_t tail_capacity) {
    return SpecOut{reinterpret_cast<unsigned long long*>(d_hist), hist_len, d_tail, tail_capacity};
}

// the spectrum result format: the histogram is overwritten whole (the tail cursor is reset by begin_op)
static int spectrum_begin(kmer_cuda_ctx* c, const SpecOut& o, cudaStream_t st) {
    CU(cudaMemsetAsync(o.hist, 0, o.hist_len * sizeof(uint64_t), st), "memset hist");
    return KMER_OK;
}

// d_uniq != nullptr: split result format (see kmer_cuda_dev_count_split); spec != nullptr: spectrum result format
// (kmer_cuda_dev_count_spectrum; d_pairs / d_uniq unused); canon: canonical k-mers (kmer_cuda_dev_count_canonical; algo 4 runs as 3)
static int dev_count_impl(kmer_cuda_ctx* c, const char* d_seq, uint64_t n_bases, const uint64_t* d_row_off, uint64_t n_rows, int k,
                          kmer_count_pair* d_pairs, uint64_t pairs_capacity, uint64_t* d_uniq, uint64_t uniq_capacity, int algo,
                          void* stream, const SpecOut* spec = nullptr, bool canon = false) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    cudaStream_t st = pick_stream(c, stream);
    int rc = begin_op(c, st);
    if (rc) return rc;
    c->pending = OP_COUNT;
    c->p_n_bases = n_bases; c->p_n_rows = n_rows; c->p_k = k;
    c->p_expected_kmers = kmer_cuda_max_kmers(n_bases, n_rows, k);
    if (spec) {
        rc = spectrum_begin(c, *spec, st);
        if (rc) return rc;
    }
    if (n_rows == 0 || n_bases == 0) {
        if (n_rows) return ref_error(&c->err, KMER_ERR_INVALID_K, 0);
        return KMER_OK;
    }
    ScanArgs a;
    rc = prepare_rows(c, d_row_off, n_bases, n_rows, k, st, &a, d_seq);
    if (rc) return rc;
    if (algo == 0) algo = (k <= 13) ? 1 : 3;
    if (canon && algo == 4) algo = 3;                                   // the two-pass scatter has no canonical minimizer
    c->last_overflow = 0;
    c->last_tier2 = 0;
    if (algo == 3 || algo == 4) {
        if (k < 14) return bad_arg(c, "minimizer-partition counting needs k >= 14");
        PartitionPlan plan = make_partition_plan(c->p_expected_kmers, k, canon);
        ScatterPlan sp{};
        // algo 4: the two write-combining passes of scatter.cuh instead of partition_kernel's scattered record stores.  Measured
        // (1 GB, k=21): 4.2 + 2.4 ms against 6.5 ms -- no gain yet (both passes are instruction bound), so it is opt-in.
        const bool two_pass = algo == 4 && make_scatter_plan(c->di, n_bases, c->p_expected_kmers, plan, sp);
        rc = ws(c, c->fill, (size_t)plan.n_buckets * 8);
        if (!rc) rc = ws(c, c->recs, partition_record_bytes(plan));
        if (!rc) rc = ws(c, c->spill, partition_spill_bytes(plan));
        if (!rc) rc = ws(c, c->failed, (size_t)plan.n_buckets * 4);
        if (!rc && two_pass) rc = ws(c, c->seg, scatter_seg_bytes(plan, sp));
        if (!rc && two_pass) rc = ws(c, c->segfill, scatter_segfill_bytes(sp));
        if (rc) return rc;
        const uint64_t t2_slots = tier2_table_slots(c->p_expected_kmers);
        rc = ws(c, c->table, t2_slots * sizeof(kmer_count_pair));
        if (rc) return rc;
        MarkArg ma{c, st};
        if (two_pass) {
            launch_scatter_refine(c->di, a, plan, sp, (uint32_t*)c->segfill.p, c->seg.p, (unsigned long long*)c->fill.p, c->recs.p,
                                  c->spill.p, st, mark_cb, &ma);
            launch_bucket_count(c->di, plan, k, (const unsigned long long*)c->fill.p, c->recs.p, c->spill.p, (uint32_t*)c->failed.p, d_pairs,
                                pairs_capacity, d_uniq, uniq_capacity, c->d_status, st, 0, 0, spec);
            mark(c, st, "bucket_count");
            c->launches += 3;
        } else {
            launch_count_partition(c->di, a, plan, (unsigned long long*)c->fill.p, c->recs.p, c->spill.p, (uint32_t*)c->failed.p,
                                   d_pairs, pairs_capacity, d_uniq, uniq_capacity, st, mark_cb, &ma, spec, canon);
            c->launches += 2;
        }
        // Tier 2 (buckets that did not fit on chip, spilled records) is decided and run by the device: nothing here waits
        // for the GPU.  Only a batch that overflows even that (DevStatus::n_overflow) is recounted, by kmer_cuda_dev_finish.
        launch_partition_tier2(c->di, plan, k, (const unsigned long long*)c->fill.p, c->recs.p, c->spill.p, (const uint32_t*)c->failed.p,
                               (kmer_count_pair*)c->table.p, t2_slots, d_pairs, pairs_capacity, c->d_status, st, mark_cb, &ma, spec, canon);
        c->launches += 4;
        c->p_recountable = true;
        c->p_canonical = canon;
        c->p_seq = d_seq; c->p_off = d_row_off; c->p_pairs = d_pairs; c->p_pairs_cap = pairs_capacity;
        c->p_spectrum = spec != nullptr;
        if (spec) {
            c->p_hist = reinterpret_cast<uint64_t*>(spec->hist); c->p_hist_len = spec->hist_len;
            c->p_tail = spec->tail; c->p_tail_cap = spec->tail_cap;
        }
        algo = -1;
    }
    if (algo == 1) {
        if (k > 15) return bad_arg(c, "dense counting needs k <= 15");
        uint64_t nbins = 1ull << (2 * k);
        rc = ws(c, c->table, nbins * 8);
        if (rc) return rc;
        if (spec) {
            launch_dense_table(c->di, a, (unsigned long long*)c->table.p, st, canon);
            launch_dense_spectrum(c->di, (const unsigned long long*)c->table.p, k, 0, 1, *spec, c->d_status, st);
        } else
            launch_count_dense(c->di, a, (unsigned long long*)c->table.p, d_pairs, pairs_capacity, st, canon);
        c->launches += 2;
        mark(c, st, spec ? "count_dense+spectrum" : "count_dense+compact");
    } else if (algo == 2) {
        uint64_t maxd = c->p_expected_kmers;
        if (k < 32 && (1ull << (2 * k)) < maxd) maxd = 1ull << (2 * k);
        uint64_t n_slots = next_pow2(std::max<uint64_t>(1024, maxd * 2));
        rc = ws(c, c->table, n_slots * sizeof(kmer_count_pair));
        if (rc) return rc;
        launch_hash_clear((kmer_count_pair*)c->table.p, n_slots, st);
        mark(c, st, "hash_clear");
        launch_count_hash_insert(c->di, a, (kmer_count_pair*)c->table.p, n_slots, st, canon);
        mark(c, st, "count_hash_insert");
        if (spec) launch_hash_spectrum(c->di, (const kmer_count_pair*)c->table.p, n_slots, k, *spec, c->d_status, st);
        else launch_hash_compact(c->di, (const kmer_count_pair*)c->table.p, n_slots, k, d_pairs, pairs_capacity, c->d_status, st);
        c->launches += 2;
        mark(c, st, spec ? "hash_spectrum" : "hash_compact");
    } else if (algo != -1)
        return bad_arg(c, "unknown counting algorithm");
    resolve_bad_row_kernel<<<1, 1, 0, st>>>(c->d_status, d_row_off, n_rows);
    c->launches++;
    CU(cudaGetLastError(), "count launch");
    return KMER_OK;
}

extern "C" int kmer_cuda_dev_count(kmer_cuda_ctx* c, const char* d_seq, uint64_t n_bases, const uint64_t* d_row_off,
                                   uint64_t n_rows, int k, kmer_count_pair* d_pairs, uint64_t pairs_capacity, int algo,
                                   void* stream) {
    return dev_count_impl(c, d_seq, n_bases, d_row_off, n_rows, k, d_pairs, pairs_capacity, nullptr, 0, algo, stream);
}

extern "C" int kmer_cuda_dev_count_split(kmer_cuda_ctx* c, const char* d_seq, uint64_t n_bases, const uint64_t* d_row_off,
                                         uint64_t n_rows, int k, uint64_t* d_uniq, uint64_t uniq_capacity,
                                         kmer_count_pair* d_pairs, uint64_t pairs_capacity, void* stream) {
    if (c && !d_uniq && uniq_capacity) return bad_arg(c, "d_uniq");
    return dev_count_impl(c, d_seq, n_bases, d_row_off, n_rows, k, d_pairs, pairs_capacity, d_uniq, d_uniq ? uniq_capacity : 0, 0,
                          stream);
}

static int spectrum_args(kmer_cuda_ctx* c, const uint64_t* d_hist, uint64_t hist_len, const kmer_count_pair* d_tail, uint64_t tail_capacity) {
    if (!d_hist || hist_len < 2) return bad_arg(c, "d_hist / hist_len (>= 2)");
    if (!d_tail && tail_capacity) return bad_arg(c, "d_tail");
    return KMER_OK;
}

extern "C" int kmer_cuda_dev_count_spectrum(kmer_cuda_ctx* c, const char* d_seq, uint64_t n_bases, const uint64_t* d_row_off,
                                            uint64_t n_rows, int k, uint64_t* d_hist, uint64_t hist_len, kmer_count_pair* d_tail,
                                            uint64_t tail_capacity, int algo, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    int rc = spectrum_args(c, d_hist, hist_len, d_tail, tail_capacity);
    if (rc) return rc;
    const SpecOut o = spec_out(d_hist, hist_len, d_tail, tail_capacity);
    return dev_count_impl(c, d_seq, n_bases, d_row_off, n_rows, k, nullptr, 0, nullptr, 0, algo, stream, &o);
}

// canonical counting: the strand-specific entry points' contracts with min(code, reverse complement) as the group key
extern "C" int kmer_cuda_dev_count_canonical(kmer_cuda_ctx* c, const char* d_seq, uint64_t n_bases, const uint64_t* d_row_off,
                                             uint64_t n_rows, int k, uint64_t* d_uniq, uint64_t uniq_capacity, kmer_count_pair* d_pairs,
                                             uint64_t pairs_capacity, int algo, void* stream) {
    if (c && !d_uniq && uniq_capacity) return bad_arg(c, "d_uniq");
    return dev_count_impl(c, d_seq, n_bases, d_row_off, n_rows, k, d_pairs, pairs_capacity, d_uniq, d_uniq ? uniq_capacity : 0, algo,
                          stream, nullptr, true);
}

extern "C" int kmer_cuda_dev_count_canonical_spectrum(kmer_cuda_ctx* c, const char* d_seq, uint64_t n_bases, const uint64_t* d_row_off,
                                                      uint64_t n_rows, int k, uint64_t* d_hist, uint64_t hist_len, kmer_count_pair* d_tail,
                                                      uint64_t tail_capacity, int algo, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    int rc = spectrum_args(c, d_hist, hist_len, d_tail, tail_capacity);
    if (rc) return rc;
    const SpecOut o = spec_out(d_hist, hist_len, d_tail, tail_capacity);
    return dev_count_impl(c, d_seq, n_bases, d_row_off, n_rows, k, nullptr, 0, nullptr, 0, algo, stream, &o, true);
}

extern "C" int kmer_cuda_dev_pairs_spectrum(kmer_cuda_ctx* c, const kmer_count_pair* d_pairs, uint64_t n, uint64_t* d_hist,
                                            uint64_t hist_len, kmer_count_pair* d_tail, uint64_t tail_capacity, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    int rc = spectrum_args(c, d_hist, hist_len, d_tail, tail_capacity);
    if (rc) return rc;
    if (n && !d_pairs) return bad_arg(c, "d_pairs");
    cudaStream_t st = pick_stream(c, stream);
    rc = begin_op(c, st);
    if (rc) return rc;
    c->pending = OP_PAIRS_SPECTRUM;
    const SpecOut o = spec_out(d_hist, hist_len, d_tail, tail_capacity);
    rc = spectrum_begin(c, o, st);
    if (rc) return rc;
    if (n) {
        launch_pairs_spectrum(c->di, d_pairs, n, o, c->d_status, st);
        c->launches++;
        mark(c, st, "pairs_spectrum");
    }
    CU(cudaGetLastError(), "pairs spectrum launch");
    return KMER_OK;
}

static int upload_consts(kmer_cuda_ctx* c, int op, const int* ops, const char* const* consts, uint32_t n_consts,
                         cudaStream_t st, bool* any_contains, const int** d_ops_out) {
    std::vector<MatchConst> mc(n_consts ? n_consts : 1);
    *any_contains = false;
    for (uint32_t i = 0; i < n_consts; i++) {
        int o = ops ? ops[i] : op;
        int rc = compile_const(c, o, consts[i], (int64_t)i, &mc[i]);
        if (rc) return rc;
        if (o == KMER_OP_CONTAINS) *any_contains = true;
    }
    int rc = ws(c, c->consts, sizeof(MatchConst) * (size_t)n_consts);
    if (rc) return rc;
    // staged through pinned memory so the async copy really is asynchronous and the vector may die
    size_t bytes = sizeof(MatchConst) * (size_t)n_consts + (ops ? sizeof(int) * (size_t)n_consts : 0);
    char* stage = (char*)pinned_get(c, bytes);
    if (!stage) return c->err.status;
    memcpy(stage, mc.data(), sizeof(MatchConst) * (size_t)n_consts);
    CU(cudaMemcpyAsync(c->consts.p, stage, sizeof(MatchConst) * (size_t)n_consts, cudaMemcpyHostToDevice, st), "H2D consts");
    *d_ops_out = nullptr;
    if (ops) {
        rc = ws(c, c->ops, sizeof(int) * (size_t)n_consts);
        if (rc) return rc;
        memcpy(stage + sizeof(MatchConst) * (size_t)n_consts, ops, sizeof(int) * (size_t)n_consts);
        CU(cudaMemcpyAsync(c->ops.p, stage + sizeof(MatchConst) * (size_t)n_consts, sizeof(int) * (size_t)n_consts,
                           cudaMemcpyHostToDevice, st), "H2D ops");
        *d_ops_out = (const int*)c->ops.p;
    }
    CU(cudaStreamSynchronize(st), "consts sync");
    kmer_cuda_release(c, stage);
    return KMER_OK;
}

extern "C" int kmer_cuda_dev_match(kmer_cuda_ctx* c, int op, const int* ops, const uint64_t* d_codes, const uint8_t* d_lens,
                                   uint64_t m, int k, const char* const* consts, uint32_t n_consts, uint32_t* d_bits,
                                   uint64_t* d_hits, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    cudaStream_t st = pick_stream(c, stream);
    int rc = begin_op(c, st);
    if (rc) return rc;
    c->pending = OP_MATCH;
    if (!d_lens && (k < 0 || k > KMER_CUDA_MAX_K)) return bad_arg(c, "k-mer length must be 0..32");
    if (n_consts > 4096) return bad_arg(c, "at most 4096 constants per call");
    bool any_contains = false;
    const int* d_ops = nullptr;
    rc = upload_consts(c, op, ops, consts, n_consts, st, &any_contains, &d_ops);
    if (rc) return rc;
    uint64_t wpr = (m + 31) / 32;
    launch_match(c->di, op, d_ops, any_contains, d_codes, d_lens, m, k, (const MatchConst*)c->consts.p, n_consts, d_bits,
                 wpr, (unsigned long long*)d_hits, st);
    c->launches++;
    mark(c, st, "match");
    CU(cudaGetLastError(), "match launch");
    return KMER_OK;
}

extern "C" int kmer_cuda_dev_decode(kmer_cuda_ctx* c, const uint64_t* d_codes, uint64_t n, int k, int with_header,
                                    char* d_text, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    cudaStream_t st = pick_stream(c, stream);
    int rc = begin_op(c, st);
    if (rc) return rc;
    c->pending = OP_DECODE;
    if (k < 0 || k > KMER_CUDA_MAX_K) return bad_arg(c, "k-mer length must be 0..32");
    launch_decode(c->di, d_codes, n, k, with_header, d_text, st);
    c->launches++;
    CU(cudaGetLastError(), "decode launch");
    return KMER_OK;
}

// seeded synthetic reads written straight into HBM (synth.cu): the benchmark shapes of SURVEY 8d2 without host generation
extern "C" int kmer_cuda_dev_synth_reads(kmer_cuda_ctx* c, uint64_t seed, uint64_t first_row, uint64_t n_rows, uint64_t read_len,
                                         char* d_seq, uint64_t* d_row_off, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    if (!d_row_off || (n_rows * read_len && !d_seq)) return bad_arg(c, "d_seq / d_row_off");
    if ((reinterpret_cast<uintptr_t>(d_seq) & 15) != 0) return bad_arg(c, "d_seq must be 16-byte aligned");
    if (read_len && n_rows > (~0ull >> 1) / read_len) return bad_arg(c, "n_rows * read_len overflows");
    cudaStream_t st = pick_stream(c, stream);
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    launch_synth_reads(c->di, seed, first_row, n_rows, read_len, d_seq, d_row_off, st);
    c->launches += n_rows * read_len ? 2 : 1;
    CU(cudaGetLastError(), "synth launch");
    return KMER_OK;
}

extern "C" int kmer_cuda_dev_pack_codes(kmer_cuda_ctx* c, const uint64_t* d_codes, uint64_t n, int k, uint8_t* d_packed, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    if (k < 1 || k > KMER_CUDA_MAX_K) return bad_arg(c, "k-mer length must be 1..32");
    if ((reinterpret_cast<uintptr_t>(d_packed) & 15) != 0) return bad_arg(c, "d_packed must be 16-byte aligned");
    cudaStream_t st = pick_stream(c, stream);
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    launch_pack_codes(c->di, d_codes, n, (2 * k + 7) / 8, d_packed, st);
    c->launches++;
    CU(cudaGetLastError(), "pack launch");
    return KMER_OK;
}

extern "C" int kmer_cuda_dev_finish(kmer_cuda_ctx* c, void* stream, kmer_dev_result* result) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    cudaStream_t st = pick_stream(c, stream);
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    CU(cudaMemcpyAsync(c->h_status, c->d_status, sizeof(DevStatus), cudaMemcpyDeviceToHost, st), "D2H status");
    CU(cudaStreamSynchronize(st), "stream sync");
    c->phase_ms.clear();
    c->phase_names.clear();
    for (size_t i = 1; i < c->ev_used; i++) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, c->ev_pool[i - 1], c->ev_pool[i]) != cudaSuccess) cudaGetLastError();
        c->phase_ms.push_back(ms);
        c->phase_names.push_back(c->ev_names[i]);
    }
    c->ev_used = 0;
    const DevStatus& s = *c->h_status;
    if (result) {
        result->n_kmers = 0;
        result->n_distinct = 0;
        result->n_overflow = 0;
        result->n_tier2 = 0;
        result->n_unique = 0;
    }
    PendingOp op = c->pending;
    c->pending = OP_NONE;
    if (op == OP_COUNT && c->p_recountable) {
        c->p_recountable = false;
        c->last_tier2 = s.t2_mode == 1ull ? s.failed_kmers + s.n_spill : 0;
        if (s.n_overflow != 0 && s.bad_char_pos == kNoError && s.short_row == kNoError) {
            // tier 3: even the spill list / the tier-2 table overflowed (highly repetitive input): everything written so far is
            // discarded and the batch is recounted through the global hash table.  The row mask of the batch is still in place.
            c->last_overflow = s.n_overflow;
            const int k = c->p_k;
            uint64_t maxd = c->p_expected_kmers;
            if (k < 32 && (1ull << (2 * k)) < maxd) maxd = 1ull << (2 * k);
            const uint64_t n_slots = next_pow2(std::max<uint64_t>(1024, maxd * 2));
            int rc = ws(c, c->table, n_slots * sizeof(kmer_count_pair));
            if (rc) return rc;
            ScanArgs a;
            a.seq = reinterpret_cast<const uint8_t*>(c->p_seq);
            a.n_bases = c->p_n_bases;
            a.row_mask = (const uint32_t*)c->mask.p;
            a.k = k;
            a.status = c->d_status;
            status_reset_kernel<<<1, 1, 0, st>>>(c->d_status);          // also rewinds the tail cursor of the spectrum format
            launch_hash_clear((kmer_count_pair*)c->table.p, n_slots, st);
            launch_count_hash_insert(c->di, a, (kmer_count_pair*)c->table.p, n_slots, st, c->p_canonical);
            if (c->p_spectrum) {                                        // what the leaf and tier 2 binned so far is void as well
                const SpecOut o = spec_out(c->p_hist, c->p_hist_len, c->p_tail, c->p_tail_cap);
                rc = spectrum_begin(c, o, st);
                if (rc) return rc;
                launch_hash_spectrum(c->di, (const kmer_count_pair*)c->table.p, n_slots, k, o, c->d_status, st);
            } else
                launch_hash_compact(c->di, (const kmer_count_pair*)c->table.p, n_slots, k, c->p_pairs, c->p_pairs_cap, c->d_status, st);
            c->launches += 3;
            CU(cudaMemcpyAsync(c->h_status, c->d_status, sizeof(DevStatus), cudaMemcpyDeviceToHost, st), "D2H status");
            CU(cudaStreamSynchronize(st), "stream sync");
        }
    }
    if (op == OP_EXTRACT || op == OP_COUNT) {
        // the first offending row decides; on the same row dna_in (text -> dna) precedes generate_kmers
        uint64_t bad_row = s.bad_char_pos == kNoError ? kNoError : s.pad;
        if (bad_row != kNoError && bad_row <= s.short_row) return ref_error(&c->err, KMER_ERR_INVALID_DNA, (int64_t)bad_row);
        if (s.short_row != kNoError) return ref_error(&c->err, KMER_ERR_INVALID_K, (int64_t)s.short_row);
        if (s.out_overflow)
            return set_error(&c->err, KMER_ERR_CAPACITY, "XX000", "kmer_cuda: output buffer too small", "", -1);
        if (result) {
            result->n_kmers = op == OP_EXTRACT ? c->p_expected_kmers : s.n_kmers;
            result->n_distinct = s.n_distinct;
            result->n_overflow = c->last_overflow;
            result->n_tier2 = c->last_tier2;
            result->n_unique = s.n_unique;
        }
        if (op == OP_COUNT && s.n_kmers != c->p_expected_kmers)
            return set_error(&c->err, KMER_ERR_CUDA, "XX000", "kmer_cuda: internal error: counted k-mers != windows", "", -1);
    } else if (op == OP_SHARD_PART || op == OP_DENSE_TABLE) {
        uint64_t bad_row = s.bad_char_pos == kNoError ? kNoError : s.pad;
        if (bad_row != kNoError && bad_row <= s.short_row) return ref_error(&c->err, KMER_ERR_INVALID_DNA, (int64_t)bad_row);
        if (s.short_row != kNoError) return ref_error(&c->err, KMER_ERR_INVALID_K, (int64_t)s.short_row);
        if (s.n_overflow)
            return set_error(&c->err, KMER_ERR_CAPACITY, "XX000",
                             "kmer_cuda: a bucket segment overflowed (input too repetitive for the sharded partition path)", "", -1);
        if (result) result->n_kmers = c->p_expected_kmers;
    } else if (op == OP_SHARD_COUNT) {
        if (c->p_chained) {
            c->p_chained = false;
            uint64_t bad_row = s.bad_char_pos == kNoError ? kNoError : s.pad;
            if (bad_row != kNoError && bad_row <= s.short_row) return ref_error(&c->err, KMER_ERR_INVALID_DNA, (int64_t)bad_row);
            if (s.short_row != kNoError) return ref_error(&c->err, KMER_ERR_INVALID_K, (int64_t)s.short_row);
        }
        if (s.out_overflow)
            return set_error(&c->err, KMER_ERR_CAPACITY, "XX000", "kmer_cuda: output buffer too small", "", -1);
        if (s.n_overflow)
            return set_error(&c->err, KMER_ERR_CAPACITY, "XX000",
                             "kmer_cuda: the spill list overflowed (input too repetitive for the sharded partition path)", "", -1);
        c->last_tier2 = s.t2_mode == 1ull ? s.failed_kmers + s.n_spill : 0;
        if (result) {
            result->n_kmers = s.n_kmers;
            result->n_distinct = s.n_distinct;
            result->n_tier2 = c->last_tier2;
            result->n_unique = s.n_unique;
        }
    } else if (op == OP_MERGE || op == OP_PAIRS_SPECTRUM) {
        if (s.out_overflow)
            return set_error(&c->err, KMER_ERR_CAPACITY, "XX000", "kmer_cuda: output buffer too small", "", -1);
        if (s.n_overflow)
            return set_error(&c->err, KMER_ERR_CAPACITY, "XX000", "kmer_cuda: merge table full (max_groups too small)", "", -1);
        if (result) {
            result->n_kmers = s.n_kmers;
            result->n_distinct = s.n_distinct;
        }
    } else if (op == OP_ENCODE) {
        if (s.bad_char_pos != kNoError) return ref_error(&c->err, KMER_ERR_INVALID_DNA, (int64_t)s.bad_char_pos);
    }
    return KMER_OK;
}

// ------------------------------------------------------------------------------------------------
// sharded counting (the caller owns the exchange)

extern "C" int kmer_cuda_shard_plan(uint64_t total_kmers, int k, uint32_t n_ranks, kmer_shard_plan* plan) {
    return kmer_cuda_shard_plan_chunked(total_kmers, k, n_ranks, 1, plan);
}

extern "C" int kmer_cuda_shard_plan_chunked(uint64_t total_kmers, int k, uint32_t n_ranks, uint32_t chunks_per_rank,
                                            kmer_shard_plan* plan) {
    if (!plan || n_ranks < 1 || n_ranks > 16 || chunks_per_rank < 1 || n_ranks * chunks_per_rank > 32 || k < 14 || k > KMER_CUDA_MAX_K)
        return KMER_ERR_BAD_ARGUMENT;
    // fine buckets as on one GPU (about 1000 k-mers each), 2^fine_shift of them per coarse partition
    PartitionPlan p = make_partition_plan(total_kmers, k);
    uint64_t fine_per_rank = ((uint64_t)p.n_buckets + n_ranks - 1) / n_ranks;
    uint32_t fine_shift = 8;
    while (fine_shift > 0 && (1ull << fine_shift) > fine_per_rank) fine_shift--;
    uint64_t coarse_per_rank = (fine_per_rank + (1ull << fine_shift) - 1) >> fine_shift;
    if (coarse_per_rank * n_ranks << fine_shift > 0x7fffffffull) return KMER_ERR_BAD_ARGUMENT;
    memset(plan, 0, sizeof(*plan));
    plan->n_ranks = n_ranks;
    plan->buckets_per_rank = (uint32_t)coarse_per_rank;
    plan->n_buckets = plan->buckets_per_rank * n_ranks;
    plan->fine_shift = fine_shift;
    plan->fine_cap = p.cap;
    plan->chunks_per_rank = chunks_per_rank;
    plan->k = k;
    plan->w = p.w; plan->m = p.m; plan->recw = p.recw; plan->rmax = p.rmax;
    plan->even_spread = (uint32_t)p.even;
    plan->rec_bytes = p.recw == 1 ? 8 : 16;
    {   // records per (coarse partition, source): 1/n_ranks of a partition's k-mers, about 2.1/(w+1) records per k-mer
        double kmers_per_part = (double)total_kmers / (double)plan->n_buckets;
        double rpk = 2.1 / (p.w + 1) + (p.rmax < p.w ? 1.0 / p.rmax : 0.0);
        double mean = kmers_per_part * rpk / (n_ranks * chunks_per_rank);
        // 1.5x: the ranks' shares of the rows are only roughly equal (ragged rows), and a segment that overflows costs the whole
        // job the exact fallback.  The slack is memory only -- the owners read the filled part of a segment, not its capacity.
        double cap = 1.5 * mean + 6.0 * sqrt(3.0 * mean) + 64.0;
        plan->cap = ((uint32_t)cap + 1u) & ~1u;   // even: every (partition, source) segment starts 16-byte aligned
    }
    plan->recs_bytes_per_peer = (uint64_t)plan->buckets_per_rank * plan->cap * plan->rec_bytes;
    plan->fill_bytes_per_peer = (uint64_t)plan->buckets_per_rank * 8;
    return KMER_OK;
}

// the source side scatters into coarse partitions; the hash range is the global number of fine buckets
static PartitionPlan coarse_partition_plan(const kmer_shard_plan* sp) {
    PartitionPlan p{};
    p.n_buckets = sp->n_buckets;
    p.hash_buckets = sp->n_buckets << sp->fine_shift;
    p.fine_shift = (int)sp->fine_shift;
    p.cap = sp->cap;
    p.w = sp->w; p.m = sp->m; p.recw = sp->recw; p.rmax = sp->rmax; p.even = (int)sp->even_spread;
    p.spill_cap = 0;   // no spill list on the source side: a full segment is an error reported by finish()
    return p;
}
// the owner side: this GPU's fine buckets (local numbering), counted like a single-GPU batch
static PartitionPlan fine_partition_plan(const kmer_shard_plan* sp) {
    PartitionPlan p{};
    p.n_buckets = sp->buckets_per_rank << sp->fine_shift;
    p.hash_buckets = sp->n_buckets << sp->fine_shift;
    p.fine_shift = (int)sp->fine_shift;
    p.cap = sp->fine_cap;
    p.w = sp->w; p.m = sp->m; p.recw = sp->recw; p.rmax = sp->rmax; p.even = (int)sp->even_spread;
    uint64_t sc = (uint64_t)p.n_buckets * p.cap / 8;
    p.spill_cap = sc < 4096 ? 4096 : sc;
    return p;
}

extern "C" int kmer_cuda_dev_shard_partition(kmer_cuda_ctx* c, const char* d_seq, uint64_t n_bases, const uint64_t* d_row_off,
                                             uint64_t n_rows, const kmer_shard_plan* sp, void* d_send_recs,
                                             uint64_t* d_send_fill, void* stream) {
    if (!c || !sp) return KMER_ERR_BAD_ARGUMENT;
    cudaStream_t st = pick_stream(c, stream);
    int rc = begin_op(c, st);
    if (rc) return rc;
    c->pending = OP_SHARD_PART;
    c->p_n_bases = n_bases; c->p_n_rows = n_rows; c->p_k = sp->k;
    c->p_expected_kmers = kmer_cuda_max_kmers(n_bases, n_rows, sp->k);
    PartitionPlan plan = coarse_partition_plan(sp);
    if (n_rows == 0 || n_bases == 0) {
        if (n_rows) return ref_error(&c->err, KMER_ERR_INVALID_K, 0);
        CU(cudaMemsetAsync(d_send_fill, 0, (size_t)sp->n_buckets * 8, st), "memset fill");
        return KMER_OK;
    }
    ScanArgs a;
    rc = prepare_rows(c, d_row_off, n_bases, n_rows, sp->k, st, &a, d_seq);
    if (rc) return rc;
    launch_partition(c->di, a, plan, (unsigned long long*)d_send_fill, d_send_recs, nullptr, st);
    mark(c, st, "minimizer_partition");
    resolve_bad_row_kernel<<<1, 1, 0, st>>>(c->d_status, d_row_off, n_rows);
    c->launches += 2;
    CU(cudaGetLastError(), "shard partition launch");
    return KMER_OK;
}

static int dev_shard_count_impl(kmer_cuda_ctx* c, const kmer_shard_plan* sp, const SrcTable& src, uint64_t* d_uniq,
                                uint64_t uniq_capacity, kmer_count_pair* d_pairs, uint64_t pairs_capacity, void* stream,
                                const SpecOut* spec = nullptr) {
    cudaStream_t st = pick_stream(c, stream);
    const bool chained = c->pending == OP_SHARD_PART;    // no finish since the partition: its findings stay in the status block
    int rc = begin_op(c, st, chained);
    if (rc) return rc;
    c->pending = OP_SHARD_COUNT;
    c->p_chained = chained;
    c->last_overflow = 0;
    c->last_tier2 = 0;
    const int k = sp->k;
    if ((sp->cap & 1u) || sp->fine_shift > 12) return bad_arg(c, "shard plan: cap must be even, fine_shift <= 12");
    // coarse partitions (one segment per source GPU) -> this GPU's fine buckets, then counted like a single-GPU batch
    PartitionPlan plan = fine_partition_plan(sp);
    if (spec) {
        rc = spectrum_begin(c, *spec, st);
        if (rc) return rc;
    }
    rc = ws(c, c->fill, (size_t)plan.n_buckets * 8);
    if (!rc) rc = ws(c, c->recs, partition_record_bytes(plan));
    if (!rc) rc = ws(c, c->spill, partition_spill_bytes(plan));
    if (!rc) rc = ws(c, c->failed, (size_t)plan.n_buckets * 4);
    if (rc) return rc;
    const int n_src = (int)(sp->n_ranks * (sp->chunks_per_rank ? sp->chunks_per_rank : 1u));
    launch_refine(c->di, plan, k, n_src, sp->buckets_per_rank, sp->cap, src, (unsigned long long*)c->fill.p, c->recs.p, c->spill.p,
                  c->d_status, st);
    mark(c, st, "refine");
    launch_bucket_count(c->di, plan, k, (const unsigned long long*)c->fill.p, c->recs.p, c->spill.p, (uint32_t*)c->failed.p, d_pairs,
                        pairs_capacity, d_uniq, d_uniq ? uniq_capacity : 0, c->d_status, st, 0, 0, spec);
    mark(c, st, "bucket_count");
    c->launches += 2;
    // tier 2 is decided and run by the device (no host round trip); an overflow of even that is reported by finish()
    const uint64_t t2_slots = tier2_table_slots((uint64_t)plan.n_buckets * 1200ull);
    rc = ws(c, c->table, t2_slots * sizeof(kmer_count_pair));
    if (rc) return rc;
    MarkArg ma{c, st};
    launch_partition_tier2(c->di, plan, k, (const unsigned long long*)c->fill.p, c->recs.p, c->spill.p, (const uint32_t*)c->failed.p,
                           (kmer_count_pair*)c->table.p, t2_slots, d_pairs, pairs_capacity, c->d_status, st, mark_cb, &ma, spec);
    c->launches += 4;
    CU(cudaGetLastError(), "shard count launch");
    return KMER_OK;
}

// the exchanged layout: [source][coarse partition][cap] records and [source][coarse partition] fills in one buffer each
static int dev_shard_count_contiguous(kmer_cuda_ctx* c, const kmer_shard_plan* sp, const void* d_recv_recs, const uint64_t* d_recv_fill,
                                      uint64_t* d_uniq, uint64_t uniq_capacity, kmer_count_pair* d_pairs, uint64_t pairs_capacity,
                                      void* stream) {
    if (!c || !sp) return KMER_ERR_BAD_ARGUMENT;
    const uint32_t n_src = sp->n_ranks * (sp->chunks_per_rank ? sp->chunks_per_rank : 1u);
    if (n_src > (uint32_t)KMER_MAX_SRC) return bad_arg(c, "shard plan: too many sources");
    SrcTable src{};
    for (uint32_t s = 0; s < n_src; s++) {
        src.recs[s] = (const char*)d_recv_recs + (size_t)s * sp->recs_bytes_per_peer;
        src.fill[s] = (const unsigned long long*)d_recv_fill + (size_t)s * sp->buckets_per_rank;
    }
    return dev_shard_count_impl(c, sp, src, d_uniq, uniq_capacity, d_pairs, pairs_capacity, stream);
}

extern "C" int kmer_cuda_dev_shard_count(kmer_cuda_ctx* c, const kmer_shard_plan* sp, const void* d_recv_recs,
                                         const uint64_t* d_recv_fill, kmer_count_pair* d_pairs, uint64_t pairs_capacity,
                                         void* stream) {
    return dev_shard_count_contiguous(c, sp, d_recv_recs, d_recv_fill, nullptr, 0, d_pairs, pairs_capacity, stream);
}

extern "C" int kmer_cuda_dev_shard_count_split(kmer_cuda_ctx* c, const kmer_shard_plan* sp, const void* d_recv_recs,
                                               const uint64_t* d_recv_fill, uint64_t* d_uniq, uint64_t uniq_capacity,
                                               kmer_count_pair* d_pairs, uint64_t pairs_capacity, void* stream) {
    if (c && !d_uniq && uniq_capacity) return bad_arg(c, "d_uniq");
    return dev_shard_count_contiguous(c, sp, d_recv_recs, d_recv_fill, d_uniq, uniq_capacity, d_pairs, pairs_capacity, stream);
}

// The exchange fused into the count: source s's segments for this owner are read where they lie -- src_recs[s] / src_fill[s]
// may be pointers into ANOTHER GPU's send buffers (peer access inside one process, kmer_cuda_ipc_open across processes).  The
// caller orders this call after every source's partition pass (an event, or any collective on the stream) and keeps the
// sources from overwriting their send buffers until this GPU's count has finished.
extern "C" int kmer_cuda_dev_shard_count_peers(kmer_cuda_ctx* c, const kmer_shard_plan* sp, const void* const* src_recs,
                                               const uint64_t* const* src_fill, uint64_t* d_uniq, uint64_t uniq_capacity,
                                               kmer_count_pair* d_pairs, uint64_t pairs_capacity, void* stream) {
    if (!c || !sp) return KMER_ERR_BAD_ARGUMENT;
    if (!src_recs || !src_fill) return bad_arg(c, "src_recs / src_fill");
    if (!d_uniq && uniq_capacity) return bad_arg(c, "d_uniq");
    const uint32_t n_src = sp->n_ranks * (sp->chunks_per_rank ? sp->chunks_per_rank : 1u);
    if (n_src > (uint32_t)KMER_MAX_SRC) return bad_arg(c, "shard plan: too many sources");
    SrcTable src{};
    for (uint32_t s = 0; s < n_src; s++) {
        if (!src_recs[s] || !src_fill[s]) return bad_arg(c, "src_recs / src_fill: null entry");
        src.recs[s] = src_recs[s];
        src.fill[s] = (const unsigned long long*)src_fill[s];
    }
    return dev_shard_count_impl(c, sp, src, d_uniq, uniq_capacity, d_pairs, pairs_capacity, stream);
}

// This rank's share in the spectrum result format.  The owners' groups are disjoint, so the ranks' histograms add up and their
// tails concatenate to the spectrum of the whole job.  The exchanged layout is the same form: src_recs[s] = recv_recs + s *
// recs_bytes_per_peer, src_fill[s] = recv_fill + s * buckets_per_rank.
extern "C" int kmer_cuda_dev_shard_count_spectrum(kmer_cuda_ctx* c, const kmer_shard_plan* sp, const void* const* src_recs,
                                                  const uint64_t* const* src_fill, uint64_t* d_hist, uint64_t hist_len,
                                                  kmer_count_pair* d_tail, uint64_t tail_capacity, void* stream) {
    if (!c || !sp) return KMER_ERR_BAD_ARGUMENT;
    int rc = spectrum_args(c, d_hist, hist_len, d_tail, tail_capacity);
    if (rc) return rc;
    if (!src_recs || !src_fill) return bad_arg(c, "src_recs / src_fill");
    const uint32_t n_src = sp->n_ranks * (sp->chunks_per_rank ? sp->chunks_per_rank : 1u);
    if (n_src > (uint32_t)KMER_MAX_SRC) return bad_arg(c, "shard plan: too many sources");
    SrcTable src{};
    for (uint32_t s = 0; s < n_src; s++) {
        if (!src_recs[s] || !src_fill[s]) return bad_arg(c, "src_recs / src_fill: null entry");
        src.recs[s] = src_recs[s];
        src.fill[s] = (const unsigned long long*)src_fill[s];
    }
    const SpecOut o = spec_out(d_hist, hist_len, d_tail, tail_capacity);
    return dev_shard_count_impl(c, sp, src, nullptr, 0, nullptr, 0, stream, &o);
}

// ---- CUDA IPC: a device buffer of this process opened in another process on the same node (one process per GPU)
typedef int (*cuMemGetAddressRange_fn)(unsigned long long*, size_t*, unsigned long long);

extern "C" int kmer_cuda_ipc_export(kmer_cuda_ctx* c, const void* d_ptr, void* handle64, uint64_t* offset) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    if (!d_ptr || !handle64 || !offset) return bad_arg(c, "ipc_export");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    // the handle names the whole ALLOCATION d_ptr lies in (a caching allocator hands out pieces of larger blocks)
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    CU(cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &qr), "cudaGetDriverEntryPoint");
    if (!fn || qr != cudaDriverEntryPointSuccess) return cuda_error(c, cudaErrorNotSupported, "cuMemGetAddressRange not found");
    unsigned long long base = 0;
    size_t size = 0;
    if (((cuMemGetAddressRange_fn)fn)(&base, &size, (unsigned long long)(uintptr_t)d_ptr) != 0)
        return cuda_error(c, cudaErrorInvalidValue, "cuMemGetAddressRange");
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, (void*)(uintptr_t)base), "cudaIpcGetMemHandle");
    memcpy(handle64, &h, 64);
    *offset = (uint64_t)((uintptr_t)d_ptr - (uintptr_t)base);
    return KMER_OK;
}

extern "C" int kmer_cuda_ipc_open(kmer_cuda_ctx* c, const void* handle64, void** d_base) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    if (!handle64 || !d_base) return bad_arg(c, "ipc_open");
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    // maps the exporter's allocation into this process and enables peer access from this context's GPU to the exporter's
    CU(cudaIpcOpenMemHandle(d_base, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle");
    return KMER_OK;
}

extern "C" int kmer_cuda_ipc_close(kmer_cuda_ctx* c, void* d_base) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    if (!d_base) return KMER_OK;
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    CU(cudaIpcCloseMemHandle(d_base), "cudaIpcCloseMemHandle");
    return KMER_OK;
}

extern "C" int kmer_cuda_dev_dense_table(kmer_cuda_ctx* c, const char* d_seq, uint64_t n_bases, const uint64_t* d_row_off,
                                         uint64_t n_rows, int k, uint64_t* d_table, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    cudaStream_t st = pick_stream(c, stream);
    int rc = begin_op(c, st);
    if (rc) return rc;
    c->pending = OP_DENSE_TABLE;
    c->p_n_bases = n_bases; c->p_n_rows = n_rows; c->p_k = k;
    c->p_expected_kmers = kmer_cuda_max_kmers(n_bases, n_rows, k);
    if (n_rows && (k < 1 || k > 13)) {
        if (k < 1 || k > KMER_CUDA_MAX_K) return ref_error(&c->err, KMER_ERR_INVALID_K, 0);
        return bad_arg(c, "dense counting needs k <= 13");
    }
    if (n_rows == 0 || n_bases == 0) {
        if (n_rows) return ref_error(&c->err, KMER_ERR_INVALID_K, 0);
        if (k >= 1 && k <= 13) CU(cudaMemsetAsync(d_table, 0, (size_t)8 << (2 * k), st), "memset table");
        return KMER_OK;
    }
    ScanArgs a;
    rc = prepare_rows(c, d_row_off, n_bases, n_rows, k, st, &a, d_seq);
    if (rc) return rc;
    launch_dense_table(c->di, a, (unsigned long long*)d_table, st);
    mark(c, st, "count_dense");
    resolve_bad_row_kernel<<<1, 1, 0, st>>>(c->d_status, d_row_off, n_rows);
    c->launches += 2;
    CU(cudaGetLastError(), "dense table launch");
    return KMER_OK;
}

extern "C" int kmer_cuda_dev_dense_emit(kmer_cuda_ctx* c, const uint64_t* d_table, int k, uint32_t rank, uint32_t n_ranks,
                                        kmer_count_pair* d_pairs, uint64_t pairs_capacity, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    cudaStream_t st = pick_stream(c, stream);
    int rc = begin_op(c, st);
    if (rc) return rc;
    c->pending = OP_SHARD_COUNT;
    c->last_overflow = 0;
    c->last_tier2 = 0;
    if (k < 1 || k > 13 || n_ranks < 1 || rank >= n_ranks) return bad_arg(c, "dense emit: k in 1..13, rank < n_ranks");
    launch_dense_emit(c->di, (const unsigned long long*)d_table, k, rank, n_ranks, d_pairs, pairs_capacity, c->d_status, st);
    mark(c, st, "dense_emit");
    c->launches++;
    CU(cudaGetLastError(), "dense emit launch");
    return KMER_OK;
}

// ------------------------------------------------------------------------------------------------
// merge of (k-mer, count) tables by owner (the exact fallback of sharded counting)

extern "C" int kmer_cuda_dev_merge_begin(kmer_cuda_ctx* c, uint64_t max_groups, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    cudaStream_t st = pick_stream(c, stream);
    int rc = begin_op(c, st);
    if (rc) return rc;
    c->pending = OP_MERGE;
    c->merge_slots = next_pow2(std::max<uint64_t>(1024, max_groups * 2));
    rc = ws(c, c->table, c->merge_slots * sizeof(kmer_count_pair));
    if (rc) return rc;
    launch_hash_clear((kmer_count_pair*)c->table.p, c->merge_slots, st);
    CU(cudaGetLastError(), "merge begin");
    return KMER_OK;
}

extern "C" int kmer_cuda_dev_merge_add(kmer_cuda_ctx* c, const kmer_count_pair* d_pairs, uint64_t n, uint32_t rank, uint32_t n_ranks,
                                       void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    if (c->pending != OP_MERGE) return bad_arg(c, "kmer_cuda_dev_merge_add without kmer_cuda_dev_merge_begin");
    if (n_ranks < 1 || rank >= n_ranks) return bad_arg(c, "merge: rank < n_ranks");
    cudaStream_t st = pick_stream(c, stream);
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    launch_merge_pairs(c->di, d_pairs, n, rank, n_ranks, (kmer_count_pair*)c->table.p, c->merge_slots, c->d_status, st);
    c->launches++;
    CU(cudaGetLastError(), "merge add");
    return KMER_OK;
}

extern "C" int kmer_cuda_dev_merge_emit(kmer_cuda_ctx* c, int k, kmer_count_pair* d_pairs, uint64_t pairs_capacity, void* stream) {
    if (!c) return KMER_ERR_BAD_ARGUMENT;
    if (c->pending != OP_MERGE) return bad_arg(c, "kmer_cuda_dev_merge_emit without kmer_cuda_dev_merge_begin");
    cudaStream_t st = pick_stream(c, stream);
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    launch_hash_compact(c->di, (const kmer_count_pair*)c->table.p, c->merge_slots, k, d_pairs, pairs_capacity, c->d_status, st);
    c->launches++;
    CU(cudaGetLastError(), "merge emit");
    return KMER_OK;
}

// ------------------------------------------------------------------------------------------------
// host-buffer batch submit

static int h2d(kmer_cuda_ctx* c, void* dst, const void* src, size_t bytes, cudaStream_t st) {
    if (!bytes) return KMER_OK;
    // pinned (or otherwise device-accessible) source: one asynchronous DMA; pageable: the driver stages it
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st), "H2D copy");
    return KMER_OK;
}

static int upload_rows(kmer_cuda_ctx* c, const char* seq, const uint64_t* row_off, uint64_t n_rows, uint64_t* n_bases) {
    if (n_rows && !row_off) return bad_arg(c, "row_off");
    *n_bases = n_rows ? row_off[n_rows] : 0;
    if (n_rows && row_off[0] != 0) return bad_arg(c, "row_off[0] must be 0");
    if (*n_bases && !seq) return bad_arg(c, "seq");
    int rc = ws(c, c->seq, ((*n_bases + 15) & ~15ull) + 64);
    if (rc) return rc;
    rc = ws(c, c->off, (n_rows + 1) * 8);
    if (rc) return rc;
    rc = h2d(c, c->seq.p, seq, *n_bases, c->stream);
    if (rc) return rc;
    if (n_rows) rc = h2d(c, c->off.p, row_off, (n_rows + 1) * 8, c->stream);
    return rc;
}

extern "C" int kmer_cuda_submit_extract(kmer_cuda_ctx* c, const char* seq, const uint64_t* row_off, uint64_t n_rows, int k,
                                        uint64_t** codes, uint64_t* n_kmers) {
    if (!c || !codes || !n_kmers) return KMER_ERR_BAD_ARGUMENT;
    *codes = nullptr;
    *n_kmers = 0;
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    uint64_t n_bases = 0;
    int rc = upload_rows(c, seq, row_off, n_rows, &n_bases);
    if (rc) return rc;
    uint64_t cap = kmer_cuda_max_kmers(n_bases, n_rows, k);
    rc = ws(c, c->codes, cap * 8);
    if (rc) return rc;
    rc = kmer_cuda_dev_extract(c, (const char*)c->seq.p, n_bases, (const uint64_t*)c->off.p, n_rows, k,
                               (uint64_t*)c->codes.p, cap, KMER_OWN_STREAM);
    if (rc) return rc;
    kmer_dev_result res;
    rc = kmer_cuda_dev_finish(c, KMER_OWN_STREAM, &res);
    if (rc) return rc;
    uint64_t* out = (uint64_t*)pinned_get(c, res.n_kmers * 8);
    if (!out) return c->err.status;
    CU(cudaMemcpyAsync(out, c->codes.p, res.n_kmers * 8, cudaMemcpyDeviceToHost, c->stream), "D2H codes");
    CU(cudaStreamSynchronize(c->stream), "stream sync");
    *codes = out;
    *n_kmers = res.n_kmers;
    return KMER_OK;
}

// ---- GROUP BY through host buffers: one implementation for the four result formats -------------------------------------------
enum CountFormat { FMT_PAIRS = 0, FMT_SPLIT = 1, FMT_PACKED = 2, FMT_SPECTRUM = 3 };

struct CountOut {              // what the four entry points hand back
    void* uniq = nullptr;      // SPLIT: uint64 codes; PACKED: code_bytes-byte integers
    uint64_t n_unique = 0;
    int code_bytes = 0;
    kmer_count_pair* pairs = nullptr;   // SPECTRUM: the tail
    uint64_t n_pairs = 0, n_kmers = 0;
    uint64_t* hist = nullptr;           // SPECTRUM: hist_len counters
};

// a pinned result buffer that goes back to the pool unless it is handed to the caller (no leak on any error return)
struct PinGuard {
    kmer_cuda_ctx* c;
    void* p = nullptr;
    explicit PinGuard(kmer_cuda_ctx* c_) : c(c_) {}
    ~PinGuard() { if (p) kmer_cuda_release(c, p); }
    void* take() { void* r = p; p = nullptr; return r; }
};

static int ensure_copy_streams(kmer_cuda_ctx* c) {
    if (c->s_in) return KMER_OK;
    CU(cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking), "cudaStreamCreate");
    CU(cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking), "cudaStreamCreate");
    for (auto& e : c->ev_in) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "cudaEventCreate");
    for (auto& e : c->ev_leaf) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "cudaEventCreate");
    CU(cudaEventCreateWithFlags(&c->ev_off, cudaEventDisableTiming), "cudaEventCreate");
    CU(cudaHostAlloc((void**)&c->h_ring, sizeof(DevStatus) * 16, cudaHostAllocDefault), "cudaHostAlloc");
    return KMER_OK;
}

// The whole table (any tier, any algorithm) -> pinned host memory after everything is counted: the plain sequence
// upload, count, download.  Used for small batches, k <= 13, and after a tier-3 recount.
static int download_count_result(kmer_cuda_ctx* c, int k, CountFormat fmt, const kmer_dev_result& res, CountOut* o) {
    PinGuard gu(c), gp(c);
    const int nbytes = k >= 1 ? (2 * k + 7) / 8 : 1;
    if (fmt != FMT_PAIRS) {
        const size_t ub = (size_t)res.n_unique * (fmt == FMT_PACKED ? (size_t)nbytes : 8);
        if (fmt == FMT_PACKED) {
            int rc = ws(c, c->text, ub + 16);
            if (rc) return rc;
            launch_pack_codes(c->di, (const uint64_t*)c->codes.p, res.n_unique, nbytes, (uint8_t*)c->text.p, c->stream);
            c->launches++;
        }
        gu.p = pinned_get(c, ub);
        if (!gu.p) return c->err.status;
        CU(cudaMemcpyAsync(gu.p, fmt == FMT_PACKED ? c->text.p : c->codes.p, ub, cudaMemcpyDeviceToHost, c->stream), "D2H codes");
    }
    gp.p = pinned_get(c, res.n_distinct * sizeof(kmer_count_pair));
    if (!gp.p) return c->err.status;
    CU(cudaMemcpyAsync(gp.p, c->pairs.p, res.n_distinct * sizeof(kmer_count_pair), cudaMemcpyDeviceToHost, c->stream), "D2H pairs");
    CU(cudaStreamSynchronize(c->stream), "stream sync");
    o->uniq = gu.take();
    o->n_unique = fmt == FMT_PAIRS ? 0 : res.n_unique;
    o->code_bytes = fmt == FMT_PACKED ? nbytes : (fmt == FMT_SPLIT ? 8 : 0);
    o->pairs = (kmer_count_pair*)gp.take();
    o->n_pairs = res.n_distinct;
    o->n_kmers = res.n_kmers;
    return KMER_OK;
}

// The spectrum format: the histogram and the tail -> pinned host memory.
static int download_spectrum(kmer_cuda_ctx* c, uint64_t hist_len, const kmer_dev_result& res, CountOut* o) {
    PinGuard gh(c), gt(c);
    gh.p = pinned_get(c, hist_len * sizeof(uint64_t));
    if (!gh.p) return c->err.status;
    CU(cudaMemcpyAsync(gh.p, c->hist.p, hist_len * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream), "D2H hist");
    gt.p = pinned_get(c, res.n_distinct * sizeof(kmer_count_pair));
    if (!gt.p) return c->err.status;
    CU(cudaMemcpyAsync(gt.p, c->pairs.p, res.n_distinct * sizeof(kmer_count_pair), cudaMemcpyDeviceToHost, c->stream), "D2H tail");
    CU(cudaStreamSynchronize(c->stream), "stream sync");
    o->hist = (uint64_t*)gh.take();
    o->pairs = (kmer_count_pair*)gt.take();
    o->n_pairs = res.n_distinct;
    o->n_kmers = res.n_kmers;
    return KMER_OK;
}

// Replaces the scan + HashAggregate of a whole column (kmer.c:289-351 + kmer_hash/kmer_equals) from HOST buffers.  For
// 14 <= k <= 32 the three legs overlap: the column arrives in pieces on a copy stream while the pieces already there are
// partitioned; the buckets are counted in groups, and behind every group the part of the result that is final leaves on a
// second copy stream (PCIe is the bound of this call: the kernels hide under the copies).  FMT_SPECTRUM (hist_len >= 2): the
// groups are binned on the device and nothing streams back but the histogram and the tail, once everything is counted.
static int submit_count_common(kmer_cuda_ctx* c, const char* seq, const uint64_t* row_off, uint64_t n_rows, int k, CountFormat fmt,
                               CountOut* o, uint64_t hist_len = 0, bool canon = false) {
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    if (n_rows && !row_off) return bad_arg(c, "row_off");
    const uint64_t n_bases = n_rows ? row_off[n_rows] : 0;
    if (n_rows && row_off[0] != 0) return bad_arg(c, "row_off[0] must be 0");
    if (n_bases && !seq) return bad_arg(c, "seq");
    int rc = ws(c, c->seq, ((n_bases + 15) & ~15ull) + 64);
    if (!rc) rc = ws(c, c->off, (n_rows + 1) * 8);
    if (rc) return rc;
    uint64_t cap = kmer_cuda_max_kmers(n_bases, n_rows, k);
    if (k >= 1 && k < 32 && (1ull << (2 * k)) < cap) cap = 1ull << (2 * k);
    // a k-mer that is not unique occurs at least twice: at most cap/2 pairs next to the unique codes -- unless a fallback
    // tier (which writes pairs only) takes over, so the pair buffer keeps the full size.  The spectrum format needs no buffer
    // of the table's size: at most n_windows / hist_len groups reach the tail.
    const bool spectrum = fmt == FMT_SPECTRUM;
    const uint64_t tail_cap = spectrum ? std::max<uint64_t>(1, kmer_cuda_max_kmers(n_bases, n_rows, k) / hist_len) : 0;
    if (spectrum) {
        rc = ws(c, c->pairs, tail_cap * sizeof(kmer_count_pair));
        if (!rc) rc = ws(c, c->hist, hist_len * sizeof(uint64_t));
    } else {
        rc = ws(c, c->pairs, cap * sizeof(kmer_count_pair));
        if (!rc && fmt != FMT_PAIRS) rc = ws(c, c->codes, cap * sizeof(uint64_t));
    }
    if (rc) return rc;
    const SpecOut so = spec_out((uint64_t*)c->hist.p, hist_len, (kmer_count_pair*)c->pairs.p, tail_cap);
    const bool pipelined = k >= 14 && k <= KMER_CUDA_MAX_K && n_rows && n_bases >= (4ull << 20);
    kmer_dev_result res;
    if (!pipelined) {
        rc = h2d(c, c->seq.p, seq, n_bases, c->stream);
        if (!rc && n_rows) rc = h2d(c, c->off.p, row_off, (n_rows + 1) * 8, c->stream);
        if (rc) return rc;
        if (spectrum)
            rc = dev_count_impl(c, (const char*)c->seq.p, n_bases, (const uint64_t*)c->off.p, n_rows, k, nullptr, 0, nullptr, 0, 0,
                                KMER_OWN_STREAM, &so, canon);
        else
            rc = dev_count_impl(c, (const char*)c->seq.p, n_bases, (const uint64_t*)c->off.p, n_rows, k, (kmer_count_pair*)c->pairs.p, cap,
                                fmt == FMT_PAIRS ? nullptr : (uint64_t*)c->codes.p, fmt == FMT_PAIRS ? 0 : cap, 0, KMER_OWN_STREAM,
                                nullptr, canon);
        if (rc) return rc;
        rc = kmer_cuda_dev_finish(c, KMER_OWN_STREAM, &res);
        if (rc) return rc;
        return spectrum ? download_spectrum(c, hist_len, res, o) : download_count_result(c, k, fmt, res, o);
    }

    // ---------------------------------------------------------------- pipelined: copy-in | kernels | copy-out
    rc = ensure_copy_streams(c);
    if (rc) return rc;
    cudaStream_t st = c->stream;
    const char* d_seq = (const char*)c->seq.p;
    const uint64_t* d_off = (const uint64_t*)c->off.p;
    kmer_count_pair* d_pairs = (kmer_count_pair*)c->pairs.p;
    uint64_t* d_uniq = fmt == FMT_PAIRS || spectrum ? nullptr : (uint64_t*)c->codes.p;
    const int nbytes = (2 * k + 7) / 8;
    const size_t ubytes = fmt == FMT_PACKED ? (size_t)nbytes : 8;
    if (fmt == FMT_PACKED) {
        rc = ws(c, c->text, cap * ubytes + 16);
        if (rc) return rc;
    }
    // the result buffer the final ranges stream into: sized for the most the batch can produce
    PinGuard gout(c);
    if (!spectrum) {
        gout.p = pinned_get(c, fmt == FMT_PAIRS ? cap * sizeof(kmer_count_pair) : cap * ubytes);
        if (!gout.p) return c->err.status;
    }
    // 1. offsets first: the row mask needs nothing else
    CU(cudaMemcpyAsync(c->off.p, row_off, (n_rows + 1) * 8, cudaMemcpyHostToDevice, c->s_in), "H2D offsets");
    CU(cudaEventRecord(c->ev_off, c->s_in), "event");
    CU(cudaStreamWaitEvent(st, c->ev_off, 0), "wait");
    rc = begin_op(c, st);
    if (rc) return rc;
    c->pending = OP_COUNT;
    c->p_n_bases = n_bases; c->p_n_rows = n_rows; c->p_k = k;
    c->p_expected_kmers = kmer_cuda_max_kmers(n_bases, n_rows, k);
    c->last_overflow = 0;
    c->last_tier2 = 0;
    if (spectrum) {
        rc = spectrum_begin(c, so, st);
        if (rc) return rc;
    }
    ScanArgs a;
    rc = prepare_rows(c, d_off, n_bases, n_rows, k, st, &a, d_seq);
    if (rc) return rc;
    PartitionPlan plan = make_partition_plan(c->p_expected_kmers, k, canon);
    rc = ws(c, c->fill, (size_t)plan.n_buckets * 8);
    if (!rc) rc = ws(c, c->recs, partition_record_bytes(plan));
    if (!rc) rc = ws(c, c->spill, partition_spill_bytes(plan));
    if (!rc) rc = ws(c, c->failed, (size_t)plan.n_buckets * 4);
    const uint64_t t2_slots = tier2_table_slots(c->p_expected_kmers);
    if (!rc) rc = ws(c, c->table, t2_slots * sizeof(kmer_count_pair));
    if (rc) return rc;
    CU(cudaMemsetAsync(c->fill.p, 0, (size_t)plan.n_buckets * 8, st), "memset fill");
    // 2. the column in pieces: piece i is partitioned while piece i+1 crosses PCIe (a piece ends on a tile boundary and is
    //    copied with the 64 bytes behind it, which its last windows read)
    const uint64_t n_tiles = (n_bases + TILE - 1) / TILE;
    const int n_pieces = n_tiles >= 8 ? 8 : 1;
    for (int i = 0; i < n_pieces; i++) {
        const uint64_t t0 = n_tiles * i / n_pieces, t1 = n_tiles * (i + 1) / n_pieces;
        const uint64_t b0 = t0 * TILE, b1 = std::min<uint64_t>(n_bases, t1 * TILE), be = std::min<uint64_t>(n_bases, b1 + 64);
        CU(cudaMemcpyAsync((char*)c->seq.p + b0, seq + b0, be - b0, cudaMemcpyHostToDevice, c->s_in), "H2D column");
        CU(cudaEventRecord(c->ev_in[i], c->s_in), "event");
        CU(cudaStreamWaitEvent(st, c->ev_in[i], 0), "wait");
        a.tile_begin = t0;
        a.tile_end = t1;
        launch_partition(c->di, a, plan, (unsigned long long*)c->fill.p, c->recs.p, c->spill.p, st, false, canon);
        c->launches++;
    }
    mark(c, st, "minimizer_partition");
    // 3. the buckets in groups; behind every group a snapshot of the result cursors (the spectrum format: one launch, nothing
    //    streams back before the end)
    const SpecOut* spec = spectrum ? &so : nullptr;
    const int n_groups = !spectrum && plan.n_buckets >= 4096 ? 8 : 1;
    for (int g = 0; g < n_groups; g++) {
        const uint32_t g0 = (uint32_t)((uint64_t)plan.n_buckets * g / n_groups), g1 = (uint32_t)((uint64_t)plan.n_buckets * (g + 1) / n_groups);
        launch_bucket_count(c->di, plan, k, (const unsigned long long*)c->fill.p, c->recs.p, c->spill.p, (uint32_t*)c->failed.p, d_pairs,
                            cap, d_uniq, d_uniq ? cap : 0, c->d_status, st, g0, g1, spec, canon);
        c->launches++;
        if (spectrum) break;
        CU(cudaMemcpyAsync(&c->h_ring[g], c->d_status, sizeof(DevStatus), cudaMemcpyDeviceToHost, st), "D2H status");
        CU(cudaEventRecord(c->ev_leaf[g], st), "event");
    }
    mark(c, st, "bucket_count");
    MarkArg ma{c, st};
    launch_partition_tier2(c->di, plan, k, (const unsigned long long*)c->fill.p, c->recs.p, c->spill.p, (const uint32_t*)c->failed.p,
                           (kmer_count_pair*)c->table.p, t2_slots, d_pairs, cap, c->d_status, st, mark_cb, &ma, spec, canon);
    resolve_bad_row_kernel<<<1, 1, 0, st>>>(c->d_status, d_off, n_rows);
    c->launches += 5;
    CU(cudaGetLastError(), "count launch");
    c->p_recountable = true;
    c->p_seq = d_seq; c->p_off = d_off; c->p_pairs = d_pairs; c->p_pairs_cap = cap;
    c->p_spectrum = spectrum;
    c->p_canonical = canon;
    if (spectrum) {
        c->p_hist = (uint64_t*)c->hist.p; c->p_hist_len = hist_len; c->p_tail = d_pairs; c->p_tail_cap = tail_cap;
        rc = kmer_cuda_dev_finish(c, KMER_OWN_STREAM, &res);      // input errors, tier 2, or a tier-3 recount
        if (rc) return rc;
        return download_spectrum(c, hist_len, res, o);
    }
    // 4. while later groups are counted, what the finished ones wrote leaves (everything below a snapshot's cursor is final)
    uint64_t done = 0;                                             // entries of the streamed array already on their way
    bool input_error = false;
    for (int g = 0; g < n_groups && !input_error; g++) {
        CU(cudaEventSynchronize(c->ev_leaf[g]), "event sync");
        const DevStatus& hs = c->h_ring[g];
        if (hs.bad_char_pos != kNoError || hs.short_row != kNoError || hs.out_overflow) { input_error = true; break; }
        const uint64_t cur = fmt == FMT_PAIRS ? hs.n_distinct : hs.n_unique;
        if (cur <= done) continue;
        CU(cudaStreamWaitEvent(c->s_out, c->ev_leaf[g], 0), "wait");
        if (fmt == FMT_PACKED) {
            const uint64_t p0 = done & ~1023ull;                   // the pack kernel works in steps of 1024 codes
            launch_pack_codes(c->di, d_uniq + p0, cur - p0, nbytes, (uint8_t*)c->text.p + p0 * ubytes, c->s_out);
            c->launches++;
            CU(cudaMemcpyAsync((char*)gout.p + p0 * ubytes, (char*)c->text.p + p0 * ubytes, (cur - p0) * ubytes, cudaMemcpyDeviceToHost, c->s_out),
               "D2H packed codes");
        } else if (fmt == FMT_SPLIT) {
            CU(cudaMemcpyAsync((uint64_t*)gout.p + done, d_uniq + done, (cur - done) * 8, cudaMemcpyDeviceToHost, c->s_out), "D2H codes");
        } else {
            CU(cudaMemcpyAsync((kmer_count_pair*)gout.p + done, d_pairs + done, (cur - done) * sizeof(kmer_count_pair), cudaMemcpyDeviceToHost,
                               c->s_out), "D2H pairs");
        }
        done = cur;
    }
    // 5. the end of the kernels: input errors, tier 2's groups, or a tier-3 recount
    rc = kmer_cuda_dev_finish(c, KMER_OWN_STREAM, &res);
    if (rc) {
        cudaStreamSynchronize(c->s_out);
        return rc;
    }
    if (res.n_overflow) {                                          // recounted: what left so far is void
        CU(cudaStreamSynchronize(c->s_out), "stream sync");
        return download_count_result(c, k, fmt, res, o);
    }
    PinGuard gp(c);
    if (fmt == FMT_PAIRS) {
        if (res.n_distinct > done)                                 // tier 2's groups and the k == 32 special key
            CU(cudaMemcpyAsync((kmer_count_pair*)gout.p + done, d_pairs + done, (res.n_distinct - done) * sizeof(kmer_count_pair),
                               cudaMemcpyDeviceToHost, c->s_out), "D2H pairs");
    } else {
        gp.p = pinned_get(c, res.n_distinct * sizeof(kmer_count_pair));
        if (!gp.p) { cudaStreamSynchronize(c->s_out); return c->err.status; }
        CU(cudaMemcpyAsync(gp.p, d_pairs, res.n_distinct * sizeof(kmer_count_pair), cudaMemcpyDeviceToHost, c->s_out), "D2H pairs");
    }
    CU(cudaStreamSynchronize(c->s_out), "stream sync");
    if (fmt == FMT_PAIRS) {
        o->pairs = (kmer_count_pair*)gout.take();
        o->n_pairs = res.n_distinct;
    } else {
        o->uniq = gout.take();
        o->n_unique = res.n_unique;
        o->code_bytes = (int)ubytes;
        o->pairs = (kmer_count_pair*)gp.take();
        o->n_pairs = res.n_distinct;
    }
    o->n_kmers = res.n_kmers;
    return KMER_OK;
}

extern "C" int kmer_cuda_submit_count(kmer_cuda_ctx* c, const char* seq, const uint64_t* row_off, uint64_t n_rows, int k,
                                      kmer_count_pair** pairs, uint64_t* n_distinct, uint64_t* n_kmers) {
    if (!c || !pairs || !n_distinct) return KMER_ERR_BAD_ARGUMENT;
    *pairs = nullptr;
    *n_distinct = 0;
    if (n_kmers) *n_kmers = 0;
    CountOut o;
    int rc = submit_count_common(c, seq, row_off, n_rows, k, FMT_PAIRS, &o);
    if (rc) return rc;
    *pairs = o.pairs;
    *n_distinct = o.n_pairs;
    if (n_kmers) *n_kmers = o.n_kmers;
    return KMER_OK;
}

extern "C" int kmer_cuda_submit_count_split(kmer_cuda_ctx* c, const char* seq, const uint64_t* row_off, uint64_t n_rows, int k,
                                            uint64_t** uniq_codes, uint64_t* n_unique, kmer_count_pair** pairs,
                                            uint64_t* n_pairs, uint64_t* n_kmers) {
    if (!c || !uniq_codes || !n_unique || !pairs || !n_pairs) return KMER_ERR_BAD_ARGUMENT;
    *uniq_codes = nullptr; *pairs = nullptr;
    *n_unique = 0; *n_pairs = 0;
    if (n_kmers) *n_kmers = 0;
    CountOut o;
    int rc = submit_count_common(c, seq, row_off, n_rows, k, FMT_SPLIT, &o);
    if (rc) return rc;
    *uniq_codes = (uint64_t*)o.uniq;
    *n_unique = o.n_unique;
    *pairs = o.pairs;
    *n_pairs = o.n_pairs;
    if (n_kmers) *n_kmers = o.n_kmers;
    return KMER_OK;
}

extern "C" int kmer_cuda_submit_count_packed(kmer_cuda_ctx* c, const char* seq, const uint64_t* row_off, uint64_t n_rows, int k,
                                             uint8_t** uniq_packed, uint64_t* n_unique, int* code_bytes,
                                             kmer_count_pair** pairs, uint64_t* n_pairs, uint64_t* n_kmers) {
    if (!c || !uniq_packed || !n_unique || !code_bytes || !pairs || !n_pairs) return KMER_ERR_BAD_ARGUMENT;
    *uniq_packed = nullptr; *pairs = nullptr;
    *n_unique = 0; *n_pairs = 0; *code_bytes = 0;
    if (n_kmers) *n_kmers = 0;
    CountOut o;
    int rc = submit_count_common(c, seq, row_off, n_rows, k, FMT_PACKED, &o);
    if (rc) return rc;
    *uniq_packed = (uint8_t*)o.uniq;
    *n_unique = o.n_unique;
    *code_bytes = k >= 1 ? (2 * k + 7) / 8 : 1;
    *pairs = o.pairs;
    *n_pairs = o.n_pairs;
    if (n_kmers) *n_kmers = o.n_kmers;
    return KMER_OK;
}

extern "C" int kmer_cuda_submit_count_spectrum(kmer_cuda_ctx* c, const char* seq, const uint64_t* row_off, uint64_t n_rows, int k,
                                             uint64_t hist_len, uint64_t** hist, kmer_count_pair** tail, uint64_t* n_tail,
                                             uint64_t* n_kmers) {
    if (!c || !hist || !tail || !n_tail || hist_len < 2) return KMER_ERR_BAD_ARGUMENT;
    *hist = nullptr; *tail = nullptr;
    *n_tail = 0;
    if (n_kmers) *n_kmers = 0;
    CountOut o;
    int rc = submit_count_common(c, seq, row_off, n_rows, k, FMT_SPECTRUM, &o, hist_len);
    if (rc) return rc;
    *hist = o.hist;
    *tail = o.pairs;
    *n_tail = o.n_pairs;
    if (n_kmers) *n_kmers = o.n_kmers;
    return KMER_OK;
}

extern "C" int kmer_cuda_submit_count_canonical(kmer_cuda_ctx* c, const char* seq, const uint64_t* row_off, uint64_t n_rows, int k,
                                                uint64_t** uniq_codes, uint64_t* n_unique, kmer_count_pair** pairs, uint64_t* n_pairs,
                                                uint64_t* n_kmers) {
    if (!c || !pairs || !n_pairs || (uniq_codes && !n_unique)) return KMER_ERR_BAD_ARGUMENT;
    if (uniq_codes) { *uniq_codes = nullptr; *n_unique = 0; }
    *pairs = nullptr;
    *n_pairs = 0;
    if (n_kmers) *n_kmers = 0;
    CountOut o;
    int rc = submit_count_common(c, seq, row_off, n_rows, k, uniq_codes ? FMT_SPLIT : FMT_PAIRS, &o, 0, true);
    if (rc) return rc;
    if (uniq_codes) {
        *uniq_codes = (uint64_t*)o.uniq;
        *n_unique = o.n_unique;
    }
    *pairs = o.pairs;
    *n_pairs = o.n_pairs;
    if (n_kmers) *n_kmers = o.n_kmers;
    return KMER_OK;
}

extern "C" int kmer_cuda_submit_count_canonical_spectrum(kmer_cuda_ctx* c, const char* seq, const uint64_t* row_off, uint64_t n_rows,
                                                         int k, uint64_t hist_len, uint64_t** hist, kmer_count_pair** tail,
                                                         uint64_t* n_tail, uint64_t* n_kmers) {
    if (!c || !hist || !tail || !n_tail || hist_len < 2) return KMER_ERR_BAD_ARGUMENT;
    *hist = nullptr; *tail = nullptr;
    *n_tail = 0;
    if (n_kmers) *n_kmers = 0;
    CountOut o;
    int rc = submit_count_common(c, seq, row_off, n_rows, k, FMT_SPECTRUM, &o, hist_len, true);
    if (rc) return rc;
    *hist = o.hist;
    *tail = o.pairs;
    *n_tail = o.n_pairs;
    if (n_kmers) *n_kmers = o.n_kmers;
    return KMER_OK;
}

extern "C" int kmer_cuda_submit_match(kmer_cuda_ctx* c, int op, const int* ops, const uint64_t* codes, const uint8_t* lens,
                                      uint64_t m, int k, const char* const* consts, uint32_t n_consts, uint32_t** bits,
                                      uint64_t* words_per_row, uint64_t** hits) {
    if (!c || !bits || !words_per_row) return KMER_ERR_BAD_ARGUMENT;
    *bits = nullptr;
    if (hits) *hits = nullptr;
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    if (m && !codes) return bad_arg(c, "codes");
    if (n_consts && !consts) return bad_arg(c, "consts");
    uint64_t wpr = (m + 31) / 32;
    *words_per_row = wpr;
    int rc = ws(c, c->codes, m * 8);
    if (!rc && lens) rc = ws(c, c->lens, m);
    if (!rc) rc = ws(c, c->bits, (size_t)n_consts * wpr * 4);
    if (!rc) rc = ws(c, c->hits, (size_t)n_consts * 8);
    if (rc) return rc;
    rc = h2d(c, c->codes.p, codes, m * 8, c->stream);
    if (!rc && lens) rc = h2d(c, c->lens.p, lens, m, c->stream);
    if (rc) return rc;
    rc = kmer_cuda_dev_match(c, op, ops, (const uint64_t*)c->codes.p, lens ? (const uint8_t*)c->lens.p : nullptr, m, k,
                             consts, n_consts, (uint32_t*)c->bits.p, (uint64_t*)c->hits.p, KMER_OWN_STREAM);
    if (rc) return rc;
    size_t bits_bytes = (size_t)n_consts * wpr * 4;
    char* out = (char*)pinned_get(c, bits_bytes);
    if (!out) return c->err.status;
    if (bits_bytes) CU(cudaMemcpyAsync(out, c->bits.p, bits_bytes, cudaMemcpyDeviceToHost, c->stream), "D2H bits");
    uint64_t* hout = (uint64_t*)pinned_get(c, (size_t)n_consts * 8);
    if (!hout) return c->err.status;
    if (n_consts) CU(cudaMemcpyAsync(hout, c->hits.p, (size_t)n_consts * 8, cudaMemcpyDeviceToHost, c->stream), "D2H hits");
    rc = kmer_cuda_dev_finish(c, KMER_OWN_STREAM, nullptr);
    if (rc) return rc;
    *bits = (uint32_t*)out;
    if (hits) *hits = hout; else kmer_cuda_release(c, hout);
    return KMER_OK;
}

extern "C" int kmer_cuda_submit_decode(kmer_cuda_ctx* c, const uint64_t* codes, uint64_t n, int k, int with_header,
                                       char** text) {
    if (!c || !text) return KMER_ERR_BAD_ARGUMENT;
    *text = nullptr;
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    if (k < 0 || k > KMER_CUDA_MAX_K) return bad_arg(c, "k-mer length must be 0..32");
    size_t bytes = (size_t)n * (size_t)(k + (with_header ? 1 : 0));
    int rc = ws(c, c->codes, n * 8);
    if (!rc) rc = ws(c, c->text, bytes);
    if (rc) return rc;
    rc = h2d(c, c->codes.p, codes, n * 8, c->stream);
    if (rc) return rc;
    rc = kmer_cuda_dev_decode(c, (const uint64_t*)c->codes.p, n, k, with_header, (char*)c->text.p, KMER_OWN_STREAM);
    if (rc) return rc;
    char* out = (char*)pinned_get(c, bytes);
    if (!out) return c->err.status;
    if (bytes) CU(cudaMemcpyAsync(out, c->text.p, bytes, cudaMemcpyDeviceToHost, c->stream), "D2H text");
    rc = kmer_cuda_dev_finish(c, KMER_OWN_STREAM, nullptr);
    if (rc) return rc;
    *text = out;
    return KMER_OK;
}

extern "C" int kmer_cuda_submit_encode(kmer_cuda_ctx* c, const char* text, const uint8_t* lens, uint64_t n, int stride,
                                       uint64_t** codes) {
    if (!c || !codes) return KMER_ERR_BAD_ARGUMENT;
    *codes = nullptr;
    CU(cudaSetDevice(c->di.device), "cudaSetDevice");
    if (stride < 0) return bad_arg(c, "stride");
    // kmer_in checks the length before the alphabet (kmer.c:115-122)
    if (lens) {
        for (uint64_t i = 0; i < n; i++)
            if (lens[i] > KMER_CUDA_MAX_K) return ref_error(&c->err, KMER_ERR_KMER_TOO_LONG, (int64_t)i);
    } else if (stride > KMER_CUDA_MAX_K && n)
        return ref_error(&c->err, KMER_ERR_KMER_TOO_LONG, 0);
    size_t bytes = (size_t)n * (size_t)stride;
    int rc = ws(c, c->text, bytes);
    if (!rc) rc = ws(c, c->codes, n * 8);
    if (!rc && lens) rc = ws(c, c->lens, n);
    if (rc) return rc;
    rc = h2d(c, c->text.p, text, bytes, c->stream);
    if (!rc && lens) rc = h2d(c, c->lens.p, lens, n, c->stream);
    if (rc) return rc;
    rc = begin_op(c, c->stream);
    if (rc) return rc;
    c->pending = OP_ENCODE;
    launch_encode(c->di, (const char*)c->text.p, lens ? (const uint8_t*)c->lens.p : nullptr, n, stride,
                  (uint64_t*)c->codes.p, c->d_status, c->stream);
    c->launches++;
    uint64_t* out = (uint64_t*)pinned_get(c, n * 8);
    if (!out) return c->err.status;
    if (n) CU(cudaMemcpyAsync(out, c->codes.p, n * 8, cudaMemcpyDeviceToHost, c->stream), "D2H codes");
    rc = kmer_cuda_dev_finish(c, KMER_OWN_STREAM, nullptr);
    if (rc) {
        kmer_cuda_release(c, out);
        return rc;
    }
    *codes = out;
    return KMER_OK;
}

// ------------------------------------------------------------------------------------------------
// several GPUs behind the C ABI, one process (kmer_cuda_init_multi): the rows are split evenly over the devices, every
// device partitions its share into the coarse minimizer partitions of ALL devices, the segments cross NVLink as peer copies
// (cudaMemcpyPeerAsync: one copy per ordered pair of devices, all pairs at once), every device counts the partitions it
// owns.  Same kernels and plan as the one-process-per-GPU path (sharded.py), no NCCL and no Python: what the PostgreSQL
// glue links.  Input the minimizer exchange refuses (a segment or the spill list overflows) and k <= 13 take the exact
// merge: per-device GROUP BY, then every device keeps the groups it owns, reading its peers' tables over NVLink.

struct kmer_cuda_multi {
    std::vector<kmer_cuda_ctx*> ctx;
    std::vector<int> dev;
    kmer_cuda_error err{};
    bool all_peers = true;           // every device can read every other device's memory (peer access)
    struct PerDev {
        Buf send, sendfill, recv, recvfill, local;
        uint64_t* h_off = nullptr;   // pinned: this device's row offsets, rebased to its first base
        size_t h_off_cap = 0;
        uint64_t n_local = 0;        // groups of the device's own GROUP BY (merge path)
    };
    std::vector<PerDev> d;
};

static int multi_fail(kmer_cuda_multi* m, const kmer_cuda_ctx* c) {
    m->err = c->err;
    return c->err.status ? c->err.status : KMER_ERR_CUDA;
}

extern "C" int kmer_cuda_init_multi(kmer_cuda_multi** out, const int* devices, int n_devices) {
    if (!out || !devices || n_devices < 1 || n_devices > 16)
        return set_error(&g_init_error, KMER_ERR_BAD_ARGUMENT, "XX000", "kmer_cuda: bad argument: device list (1..16 devices)", "", -1);
    *out = nullptr;
    kmer_cuda_multi* m = new (std::nothrow) kmer_cuda_multi();
    if (!m) return set_error(&g_init_error, KMER_ERR_OOM, "53200", "kmer_cuda: out of host memory", "", -1);
    for (int i = 0; i < n_devices; i++) {
        kmer_cuda_ctx* c = nullptr;
        int rc = kmer_cuda_init(&c, devices[i]);
        if (rc) {
            for (auto x : m->ctx) kmer_cuda_shutdown(x);
            delete m;
            return rc;
        }
        m->ctx.push_back(c);
        m->dev.push_back(devices[i]);
    }
    m->d.resize(n_devices);
    // peer access both ways (kernels of the merge path read peer tables directly); the same device twice is fine
    for (int i = 0; i < n_devices; i++)
        for (int j = 0; j < n_devices; j++) {
            if (devices[i] == devices[j]) continue;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, devices[i], devices[j]);
            if (!can) { m->all_peers = false; continue; }
            cudaSetDevice(devices[i]);
            cudaError_t ce = cudaDeviceEnablePeerAccess(devices[j], 0);
            if (ce != cudaSuccess) cudaGetLastError();   // already enabled
        }
    m->err.status = KMER_OK;
    m->err.row = -1;
    *out = m;
    return KMER_OK;
}

extern "C" void kmer_cuda_shutdown_multi(kmer_cuda_multi* m) {
    if (!m) return;
    for (size_t i = 0; i < m->ctx.size(); i++) {
        cudaSetDevice(m->dev[i]);
        cudaStreamSynchronize(m->ctx[i]->stream);
        auto& d = m->d[i];
        Buf* all[] = {&d.send, &d.sendfill, &d.recv, &d.recvfill, &d.local};
        for (Buf* b : all) buf_free(*b);
        if (d.h_off) cudaFreeHost(d.h_off);
        kmer_cuda_shutdown(m->ctx[i]);
    }
    delete m;
}

extern "C" int kmer_cuda_multi_device_count(const kmer_cuda_multi* m) { return m ? (int)m->ctx.size() : 0; }
extern "C" const kmer_cuda_error* kmer_cuda_multi_last_error(const kmer_cuda_multi* m) { return m ? &m->err : &g_init_error; }
extern "C" void kmer_cuda_multi_release(kmer_cuda_multi* m, int device_index, void* result) {
    if (m && device_index >= 0 && device_index < (int)m->ctx.size()) kmer_cuda_release(m->ctx[device_index], result);
}

// per-device GROUP BY of the device's own rows, then the merge by owner over peer memory
static int multi_count_merge(kmer_cuda_multi* m, const std::vector<uint64_t>& nb, const std::vector<uint64_t>& nr, int k,
                             kmer_count_pair** pairs, uint64_t* n_distinct, uint64_t* n_kmers) {
    const int n = (int)m->ctx.size();
    uint64_t total_groups = 0, total_kmers = 0;
    for (int i = 0; i < n; i++) {
        kmer_cuda_ctx* c = m->ctx[i];
        cudaSetDevice(m->dev[i]);
        uint64_t cap = kmer_cuda_max_kmers(nb[i], nr[i], k);
        if (k >= 1 && k < 32 && (1ull << (2 * k)) < cap) cap = 1ull << (2 * k);
        int rc = ws(c, m->d[i].local, (cap ? cap : 1) * sizeof(kmer_count_pair));
        if (rc) return multi_fail(m, c);
        rc = kmer_cuda_dev_count(c, (const char*)c->seq.p, nb[i], (const uint64_t*)c->off.p, nr[i], k, (kmer_count_pair*)m->d[i].local.p, cap, 0,
                                 KMER_OWN_STREAM);
        if (rc) return multi_fail(m, c);
    }
    for (int i = 0; i < n; i++) {
        kmer_dev_result res;
        cudaSetDevice(m->dev[i]);
        int rc = kmer_cuda_dev_finish(m->ctx[i], KMER_OWN_STREAM, &res);
        if (rc) {                                        // rows of device i: report the row index within the whole batch
            m->err = m->ctx[i]->err;
            return rc;
        }
        m->d[i].n_local = res.n_distinct;
        total_groups += res.n_distinct;
        total_kmers += res.n_kmers;
    }
    // the owner hash spreads DISTINCT k-mers evenly whatever their counts: a device owns about total/n groups
    const uint64_t own_cap = (uint64_t)((double)total_groups / n * 1.3) + 65536;
    for (int j = 0; j < n; j++) {
        kmer_cuda_ctx* c = m->ctx[j];
        cudaSetDevice(m->dev[j]);
        int rc = ws(c, c->pairs, own_cap * sizeof(kmer_count_pair));
        if (!rc) rc = kmer_cuda_dev_merge_begin(c, own_cap, KMER_OWN_STREAM);
        for (int i = 0; i < n && !rc; i++)
            rc = kmer_cuda_dev_merge_add(c, (const kmer_count_pair*)m->d[i].local.p, m->d[i].n_local, (uint32_t)j, (uint32_t)n, KMER_OWN_STREAM);
        if (!rc) rc = kmer_cuda_dev_merge_emit(c, k, (kmer_count_pair*)c->pairs.p, own_cap, KMER_OWN_STREAM);
        if (rc) return multi_fail(m, c);
    }
    uint64_t counted = 0;
    for (int j = 0; j < n; j++) {
        kmer_cuda_ctx* c = m->ctx[j];
        cudaSetDevice(m->dev[j]);
        kmer_dev_result res;
        int rc = kmer_cuda_dev_finish(c, KMER_OWN_STREAM, &res);
        if (rc) return multi_fail(m, c);
        kmer_count_pair* out = (kmer_count_pair*)pinned_get(c, res.n_distinct * sizeof(kmer_count_pair));
        if (!out) return multi_fail(m, c);
        if (cudaMemcpyAsync(out, c->pairs.p, res.n_distinct * sizeof(kmer_count_pair), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) {
            kmer_cuda_release(c, out);
            cuda_error(c, cudaGetLastError(), "D2H pairs");
            return multi_fail(m, c);
        }
        pairs[j] = out;
        n_distinct[j] = res.n_distinct;
        counted += res.n_kmers;
    }
    for (int j = 0; j < n; j++) {
        cudaSetDevice(m->dev[j]);
        cudaStreamSynchronize(m->ctx[j]->stream);
    }
    if (counted != total_kmers) {
        set_error(&m->err, KMER_ERR_CUDA, "XX000", "kmer_cuda: internal error: merged k-mers != counted k-mers", "", -1);
        return KMER_ERR_CUDA;
    }
    if (n_kmers) *n_kmers = counted;
    return KMER_OK;
}

extern "C" int kmer_cuda_multi_submit_count(kmer_cuda_multi* m, const char* seq, const uint64_t* row_off, uint64_t n_rows, int k,
                                            kmer_count_pair** pairs, uint64_t* n_distinct, uint64_t* n_kmers) {
    if (!m || !pairs || !n_distinct) return KMER_ERR_BAD_ARGUMENT;
    const int n = (int)m->ctx.size();
    for (int i = 0; i < n; i++) { pairs[i] = nullptr; n_distinct[i] = 0; }
    if (n_kmers) *n_kmers = 0;
    m->err.status = KMER_OK;
    if (n == 1) {
        int rc = kmer_cuda_submit_count(m->ctx[0], seq, row_off, n_rows, k, &pairs[0], &n_distinct[0], n_kmers);
        if (rc) m->err = m->ctx[0]->err;
        return rc;
    }
    if (n_rows && (!row_off || row_off[0] != 0 || (row_off[n_rows] && !seq))) {
        set_error(&m->err, KMER_ERR_BAD_ARGUMENT, "XX000", "kmer_cuda: bad argument: seq / row_off", "", -1);
        return KMER_ERR_BAD_ARGUMENT;
    }
    if (n_rows && (k < 1 || k > KMER_CUDA_MAX_K)) return ref_error(&m->err, KMER_ERR_INVALID_K, 0);
    // 1. rows split evenly; every device gets its slice of the column and its offsets rebased to 0
    std::vector<uint64_t> r0(n + 1), nb(n), nr(n);
    for (int i = 0; i <= n; i++) r0[i] = n_rows * (uint64_t)i / n;
    uint64_t total_kmers = 0;
    for (int i = 0; i < n; i++) {
        kmer_cuda_ctx* c = m->ctx[i];
        auto& d = m->d[i];
        cudaSetDevice(m->dev[i]);
        nr[i] = r0[i + 1] - r0[i];
        const uint64_t base = n_rows ? row_off[r0[i]] : 0;
        nb[i] = n_rows ? row_off[r0[i + 1]] - base : 0;
        total_kmers += kmer_cuda_max_kmers(nb[i], nr[i], k);
        if (d.h_off_cap < nr[i] + 1) {
            if (d.h_off) cudaFreeHost(d.h_off);
            d.h_off = nullptr;
            d.h_off_cap = 0;
            if (cudaHostAlloc((void**)&d.h_off, (nr[i] + 1) * 8, cudaHostAllocDefault) != cudaSuccess) {
                cuda_error(c, cudaGetLastError(), "cudaHostAlloc");
                return multi_fail(m, c);
            }
            d.h_off_cap = nr[i] + 1;
        }
        for (uint64_t r = 0; r <= nr[i]; r++) d.h_off[r] = row_off[r0[i] + r] - base;
        int rc = ws(c, c->seq, ((nb[i] + 15) & ~15ull) + 64);
        if (!rc) rc = ws(c, c->off, (nr[i] + 1) * 8);
        if (!rc) rc = h2d(c, c->seq.p, seq + base, nb[i], c->stream);
        if (!rc) rc = h2d(c, c->off.p, d.h_off, (nr[i] + 1) * 8, c->stream);
        if (rc) return multi_fail(m, c);
    }
    auto rebase_error_row = [&](int i) {                  // a device reports rows of its slice
        if (m->err.row >= 0) m->err.row += (int64_t)r0[i];
    };
    if (k <= 13 || total_kmers == 0) {
        int rc = multi_count_merge(m, nb, nr, k, pairs, n_distinct, n_kmers);
        if (rc && (rc == KMER_ERR_INVALID_DNA || rc == KMER_ERR_INVALID_K))
            for (int i = 0; i < n; i++) if (m->ctx[i]->err.status == rc) { m->err = m->ctx[i]->err; rebase_error_row(i); break; }
        return rc;
    }
    // 2. the sharded path: partition on every device, peer copies, count on every owner
    kmer_shard_plan sp;
    if (kmer_cuda_shard_plan(total_kmers, k, (uint32_t)n, &sp) != KMER_OK) {
        set_error(&m->err, KMER_ERR_BAD_ARGUMENT, "XX000", "kmer_cuda: no shard plan for this job", "", -1);
        return KMER_ERR_BAD_ARGUMENT;
    }
    const size_t rb = sp.recs_bytes_per_peer, fb = sp.fill_bytes_per_peer;
    for (int i = 0; i < n; i++) {
        kmer_cuda_ctx* c = m->ctx[i];
        auto& d = m->d[i];
        cudaSetDevice(m->dev[i]);
        int rc = ws(c, d.send, rb * n);
        if (!rc) rc = ws(c, d.sendfill, fb * n);
        if (!rc) rc = kmer_cuda_dev_shard_partition(c, (const char*)c->seq.p, nb[i], (const uint64_t*)c->off.p, nr[i], &sp, d.send.p,
                                                    (uint64_t*)d.sendfill.p, KMER_OWN_STREAM);
        if (rc) return multi_fail(m, c);
    }
    bool capacity = false;
    int first_err = KMER_OK, first_dev = -1;
    for (int i = 0; i < n; i++) {                         // the first offending ROW of the batch decides, as in a sequential scan
        cudaSetDevice(m->dev[i]);
        int rc = kmer_cuda_dev_finish(m->ctx[i], KMER_OWN_STREAM, nullptr);
        if (rc == KMER_ERR_CAPACITY) capacity = true;
        else if (rc && first_err == KMER_OK) { first_err = rc; first_dev = i; }
    }
    if (first_err) {
        m->err = m->ctx[first_dev]->err;
        rebase_error_row(first_dev);
        return first_err;
    }
    if (!capacity) {
        const uint64_t own_cap = (uint64_t)((double)total_kmers / n * 1.15) + (1u << 20);
        if (m->all_peers) {
            // every owner reads its segments straight out of the sources' send buffers (peer memory over NVLink): the
            // exchange is part of the owner's split kernel.  All partitions have finished (dev_finish above).
            std::vector<const void*> sr(n);
            std::vector<const uint64_t*> sf(n);
            for (int j = 0; j < n; j++) {
                kmer_cuda_ctx* c = m->ctx[j];
                cudaSetDevice(m->dev[j]);
                for (int i = 0; i < n; i++) {
                    sr[i] = (const char*)m->d[i].send.p + rb * j;
                    sf[i] = (const uint64_t*)((const char*)m->d[i].sendfill.p + fb * j);
                }
                int rc = ws(c, c->pairs, own_cap * sizeof(kmer_count_pair));
                if (!rc) rc = kmer_cuda_dev_shard_count_peers(c, &sp, sr.data(), sf.data(), nullptr, 0, (kmer_count_pair*)c->pairs.p, own_cap,
                                                              KMER_OWN_STREAM);
                if (rc) return multi_fail(m, c);
            }
        } else {
            for (int i = 0; i < n; i++) {
                cudaSetDevice(m->dev[i]);
                int rc = ws(m->ctx[i], m->d[i].recv, rb * n);
                if (!rc) rc = ws(m->ctx[i], m->d[i].recvfill, fb * n);
                if (rc) return multi_fail(m, m->ctx[i]);
            }
            for (int i = 0; i < n; i++)                   // segment block j of device i -> slot i of device j (staged by the driver)
                for (int j = 0; j < n; j++) {
                    cudaError_t ce = cudaMemcpyPeerAsync((char*)m->d[j].recv.p + rb * i, m->dev[j], (const char*)m->d[i].send.p + rb * j, m->dev[i], rb,
                                                         m->ctx[i]->stream);
                    if (ce == cudaSuccess)
                        ce = cudaMemcpyPeerAsync((char*)m->d[j].recvfill.p + fb * i, m->dev[j], (const char*)m->d[i].sendfill.p + fb * j, m->dev[i], fb,
                                                 m->ctx[i]->stream);
                    if (ce != cudaSuccess) { cuda_error(m->ctx[i], ce, "cudaMemcpyPeerAsync"); return multi_fail(m, m->ctx[i]); }
                }
            for (int i = 0; i < n; i++) { cudaSetDevice(m->dev[i]); cudaStreamSynchronize(m->ctx[i]->stream); }
            for (int j = 0; j < n; j++) {
                kmer_cuda_ctx* c = m->ctx[j];
                cudaSetDevice(m->dev[j]);
                int rc = ws(c, c->pairs, own_cap * sizeof(kmer_count_pair));
                if (!rc) rc = kmer_cuda_dev_shard_count(c, &sp, m->d[j].recv.p, (const uint64_t*)m->d[j].recvfill.p, (kmer_count_pair*)c->pairs.p,
                                                        own_cap, KMER_OWN_STREAM);
                if (rc) return multi_fail(m, c);
            }
        }
        std::vector<kmer_dev_result> res(n);
        for (int j = 0; j < n; j++) {
            cudaSetDevice(m->dev[j]);
            int rc = kmer_cuda_dev_finish(m->ctx[j], KMER_OWN_STREAM, &res[j]);
            if (rc == KMER_ERR_CAPACITY) capacity = true;
            else if (rc) return multi_fail(m, m->ctx[j]);
        }
        if (!capacity) {
            uint64_t counted = 0;
            for (int j = 0; j < n; j++) {
                kmer_cuda_ctx* c = m->ctx[j];
                cudaSetDevice(m->dev[j]);
                kmer_count_pair* out = (kmer_count_pair*)pinned_get(c, res[j].n_distinct * sizeof(kmer_count_pair));
                if (!out) return multi_fail(m, c);
                cudaMemcpyAsync(out, c->pairs.p, res[j].n_distinct * sizeof(kmer_count_pair), cudaMemcpyDeviceToHost, c->stream);
                pairs[j] = out;
                n_distinct[j] = res[j].n_distinct;
                counted += res[j].n_kmers;
            }
            for (int j = 0; j < n; j++) { cudaSetDevice(m->dev[j]); cudaStreamSynchronize(m->ctx[j]->stream); }
            if (counted != total_kmers) {
                set_error(&m->err, KMER_ERR_CUDA, "XX000", "kmer_cuda: internal error: counted k-mers != windows", "", -1);
                return KMER_ERR_CUDA;
            }
            if (n_kmers) *n_kmers = counted;
            return KMER_OK;
        }
    }
    // 3. the exchange ran out of room somewhere (skewed input): exact merge instead
    return multi_count_merge(m, nb, nr, k, pairs, n_distinct, n_kmers);
}

// equals / starts_with / contains over a host column on every device of the handle (SURVEY 8e: "shard M, replicate patterns, no
// collective").  The column is cut on multiples of 32 k-mers, so every device's words of a bit row are whole 32-bit words of the
// P x M matrix: device i matches its slice against all constants and its words land in place -- one strided copy per device
// straight into the one pinned result matrix -- and the per-constant hit counts are added on the host.  Same result layout as
// kmer_cuda_submit_match; both result buffers belong to device 0's context (kmer_cuda_multi_release(m, 0, ...)).
extern "C" int kmer_cuda_multi_submit_match(kmer_cuda_multi* m, int op, const int* ops, const uint64_t* codes, const uint8_t* lens,
                                            uint64_t n_kmers, int k, const char* const* consts, uint32_t n_consts, uint32_t** bits,
                                            uint64_t* words_per_row, uint64_t** hits) {
    if (!m || !bits || !words_per_row) return KMER_ERR_BAD_ARGUMENT;
    *bits = nullptr;
    if (hits) *hits = nullptr;
    m->err.status = KMER_OK;
    const int n = (int)m->ctx.size();
    if (n == 1) {
        int rc = kmer_cuda_submit_match(m->ctx[0], op, ops, codes, lens, n_kmers, k, consts, n_consts, bits, words_per_row, hits);
        if (rc) m->err = m->ctx[0]->err;
        return rc;
    }
    if ((n_kmers && !codes) || (n_consts && !consts)) {
        set_error(&m->err, KMER_ERR_BAD_ARGUMENT, "XX000", "kmer_cuda: bad argument: codes / consts", "", -1);
        return KMER_ERR_BAD_ARGUMENT;
    }
    const uint64_t wpr = (n_kmers + 31) / 32;
    *words_per_row = wpr;
    std::vector<uint64_t> cut(n + 1);
    for (int i = 0; i <= n; i++) cut[i] = i == n ? n_kmers : ((n_kmers / n * i + n_kmers % n * i / n) & ~31ull);
    kmer_cuda_ctx* c0 = m->ctx[0];
    cudaSetDevice(m->dev[0]);
    PinGuard g_bits(c0), g_hits(c0);
    g_bits.p = pinned_get(c0, (size_t)n_consts * wpr * 4);
    if (!g_bits.p) return multi_fail(m, c0);
    g_hits.p = pinned_get(c0, (size_t)n_consts * 8);
    if (!g_hits.p) return multi_fail(m, c0);
    std::vector<uint64_t*> part(n, nullptr);      // every device's own hit counters, pinned in its context
    auto drop_parts = [&]() {
        for (int i = 0; i < n; i++)
            if (part[i]) { kmer_cuda_release(m->ctx[i], part[i]); part[i] = nullptr; }
    };
    for (int i = 0; i < n; i++) {
        kmer_cuda_ctx* c = m->ctx[i];
        cudaSetDevice(m->dev[i]);
        const uint64_t ml = cut[i + 1] - cut[i], wl = (ml + 31) / 32;
        int rc = ws(c, c->codes, ml * 8);
        if (!rc && lens) rc = ws(c, c->lens, ml);
        if (!rc) rc = ws(c, c->bits, (size_t)n_consts * wl * 4);
        if (!rc) rc = ws(c, c->hits, (size_t)n_consts * 8);
        if (!rc) rc = h2d(c, c->codes.p, codes + cut[i], ml * 8, c->stream);
        if (!rc && lens) rc = h2d(c, c->lens.p, lens + cut[i], ml, c->stream);
        // a bad constant is found on the host before anything is launched, on the first device: reported once
        if (!rc) rc = kmer_cuda_dev_match(c, op, ops, (const uint64_t*)c->codes.p, lens ? (const uint8_t*)c->lens.p : nullptr, ml, k, consts,
                                          n_consts, (uint32_t*)c->bits.p, (uint64_t*)c->hits.p, KMER_OWN_STREAM);
        if (!rc && !(part[i] = (uint64_t*)pinned_get(c, (size_t)n_consts * 8))) rc = c->err.status;
        cudaError_t ce = cudaSuccess;
        if (!rc && wl && n_consts) {
            char* dst = (char*)g_bits.p + (cut[i] / 32) * 4;
            if (wpr * 4 < (1ull << 31))
                ce = cudaMemcpy2DAsync(dst, wpr * 4, c->bits.p, wl * 4, wl * 4, n_consts, cudaMemcpyDeviceToHost, c->stream);
            else                                  // a row longer than the largest pitch: row by row
                for (uint32_t p = 0; p < n_consts && ce == cudaSuccess; p++)
                    ce = cudaMemcpyAsync(dst + (size_t)p * wpr * 4, (const char*)c->bits.p + (size_t)p * wl * 4, wl * 4, cudaMemcpyDeviceToHost,
                                         c->stream);
        }
        if (!rc && ce == cudaSuccess && n_consts)
            ce = cudaMemcpyAsync(part[i], c->hits.p, (size_t)n_consts * 8, cudaMemcpyDeviceToHost, c->stream);
        if (!rc && ce != cudaSuccess) rc = cuda_error(c, ce, "D2H match result");
        if (rc) {
            for (int j = 0; j <= i; j++) {        // let what is queued drain before the buffers go back
                cudaSetDevice(m->dev[j]);
                cudaStreamSynchronize(m->ctx[j]->stream);
            }
            drop_parts();
            return multi_fail(m, c);
        }
    }
    int first = KMER_OK, first_dev = -1;
    for (int i = 0; i < n; i++) {
        cudaSetDevice(m->dev[i]);
        int rc = kmer_cuda_dev_finish(m->ctx[i], KMER_OWN_STREAM, nullptr);
        if (rc && first == KMER_OK) { first = rc; first_dev = i; }
    }
    if (first) {
        drop_parts();
        return multi_fail(m, m->ctx[first_dev]);
    }
    uint64_t* hsum = (uint64_t*)g_hits.p;
    for (uint32_t p = 0; p < n_consts; p++) {
        uint64_t s = 0;
        for (int i = 0; i < n; i++) s += part[i][p];
        hsum[p] = s;
    }
    drop_parts();
    *bits = (uint32_t*)g_bits.take();
    if (hits) *hits = (uint64_t*)g_hits.take();
    return KMER_OK;
}
