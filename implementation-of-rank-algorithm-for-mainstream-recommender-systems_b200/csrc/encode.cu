// encode.cu — the WeChat frame's categorical columns encoded on the device, straight from Arrow string
// buffers: rank_b200.loader.EncodedWechat's `index[v] if v in index else 0` per value (encode_column) and
// DIN's `str.split(",")` + lookup per history item (EncodedWechat._din_history), which the host does with
// a Python dict probe per value.
//
// A vocabulary is an open-addressing table of 2^k >= 2 * n_keys 64-bit slots over its unique keys (the
// host's dict keeps the semantics: stripped lines, a duplicated line keeps its last position).  A slot
// holds (hash >> 32) << 32 | key index, so a probe compares key bytes only when the upper hash bits agree;
// ~0 marks an empty slot.  Insertion claims a slot with atomicCAS and probes linearly; keys are unique, so
// it never compares strings.  Lookups probe linearly until the key or an empty slot: at a load factor of at
// most 1/2 a miss ends after ~2.5 slots on average.  Values are compared byte for byte: Arrow strings are
// valid UTF-8, so byte equality is Python str equality.
//
// The bound is the latency of the dependent reads of a probe (slot, key offsets, key bytes), not bandwidth.
#include "common.cuh"

namespace rk {

constexpr int kEncodeThreads = 256;
constexpr int64_t kEncodeMaxCtas = 1 << 16;              // grid-stride beyond this
constexpr uint64_t kEmptySlot = ~0ull;

struct Table {
    const char*     bytes;
    const int64_t*  offsets;
    const int64_t*  pos;
    const uint64_t* slots;
    uint64_t        mask;                                 // n_slots - 1
};

// FNV-1a over the bytes, then the murmur3 finaliser so that both the low bits (the slot) and the high bits
// (the tag) depend on every byte.
__device__ __forceinline__ uint64_t key_hash(const char* s, int64_t len) {
    uint64_t h = 0xcbf29ce484222325ull;
    for (int64_t i = 0; i < len; ++i) {
        h ^= (uint8_t)s[i];
        h *= 0x100000001b3ull;
    }
    h ^= h >> 33;
    h *= 0xff51afd7ed558ccdull;
    h ^= h >> 33;
    h *= 0xc4ceb9fe1a85ec53ull;
    h ^= h >> 33;
    return h;
}

__device__ __forceinline__ bool bytes_equal(const char* a, const char* b, int64_t len) {
    for (int64_t i = 0; i < len; ++i)
        if (a[i] != b[i]) return false;
    return true;
}

// The id of the string s[0, len): the key's position on a hit, 0 on a miss.  The one probe of every lookup.
__device__ int64_t vocab_find(const Table& t, const char* s, int64_t len, uint32_t& bits) {
    const uint64_t h = key_hash(s, len);
    const uint32_t tag = (uint32_t)(h >> 32);
    uint64_t at = h & t.mask;
    for (uint64_t probes = 0; probes <= t.mask; ++probes, at = (at + 1) & t.mask) {
        const uint64_t e = __ldg(t.slots + at);
        if (e == kEmptySlot) return 0;
        if ((uint32_t)(e >> 32) != tag) continue;
        const uint32_t k = (uint32_t)e;
        const int64_t b0 = __ldg(t.offsets + k);
        if (__ldg(t.offsets + k + 1) - b0 == len && bytes_equal(t.bytes + b0, s, len)) return __ldg(t.pos + k);
    }
    bits |= RK_ENCODE_TABLE_FULL;                        // no empty slot: not a table rk_vocab_build made
    return 0;
}

__global__ void __launch_bounds__(kEncodeThreads)
vocab_insert_kernel(const char* __restrict__ bytes, const int64_t* __restrict__ offsets, int64_t n_keys,
                    uint64_t* slots, uint64_t mask, uint32_t* status) {
    uint32_t bits = 0;
    for (int64_t k = (int64_t)blockIdx.x * kEncodeThreads + threadIdx.x; k < n_keys;
         k += (int64_t)gridDim.x * kEncodeThreads) {
        const int64_t b0 = offsets[k];
        const uint64_t h = key_hash(bytes + b0, offsets[k + 1] - b0);
        const unsigned long long entry = ((h >> 32) << 32) | (uint64_t)k;
        uint64_t at = h & mask, probes = 0;
        while (atomicCAS(reinterpret_cast<unsigned long long*>(slots + at), kEmptySlot, entry) != kEmptySlot) {
            at = (at + 1) & mask;
            if (++probes > mask) {
                bits |= RK_ENCODE_TABLE_FULL;
                break;
            }
        }
    }
    if (bits) atomicOr(status, bits);
}

__device__ __forceinline__ bool is_valid(const rk_str_col_t& c, int64_t i) {
    if (!c.valid) return true;
    const int64_t b = c.valid_bit0 + i;
    return (c.valid[b >> 3] >> (b & 7)) & 1;
}

__global__ void __launch_bounds__(kEncodeThreads)
encode_strings_kernel(const Table t, const rk_str_col_t c, int64_t* __restrict__ out, int64_t stride,
                      uint32_t* status) {
    uint32_t bits = 0;
    for (int64_t i = (int64_t)blockIdx.x * kEncodeThreads + threadIdx.x; i < c.n;
         i += (int64_t)gridDim.x * kEncodeThreads) {
        int64_t id = 0;                                   // null -> 0, as a missing value
        if (is_valid(c, i)) {
            const int64_t b0 = __ldg(c.offsets + i);
            id = vocab_find(t, c.bytes + b0, __ldg(c.offsets + i + 1) - b0, bits);
        }
        out[i * stride] = id;
    }
    if (bits) atomicOr(status, bits);
}

// One warp per row: 1 + the number of ',' bytes (str.split(",") item count).
__global__ void __launch_bounds__(kEncodeThreads)
split_count_kernel(const rk_str_col_t c, int64_t* __restrict__ counts) {
    const int lane = threadIdx.x % kWarp;
    const int64_t warps = (int64_t)gridDim.x * (kEncodeThreads / kWarp);
    for (int64_t r = ((int64_t)blockIdx.x * kEncodeThreads + threadIdx.x) / kWarp; r < c.n; r += warps) {
        const int64_t b1 = __ldg(c.offsets + r + 1);
        int n = 0;
        for (int64_t p = __ldg(c.offsets + r) + lane; p < b1; p += kWarp) n += __ldg(c.bytes + p) == ',';
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(kFull, n, o);
        if (lane == 0) counts[r] = 1 + (int64_t)n;
    }
}

// One warp per row, 32 bytes per step.  The lane that holds a ',' looks up the item that ends there; it
// starts after the nearest ',' of a lower lane, or where the last step's last item ended.  Lane 0 looks up
// the row's last item.  Item k of row r goes to out[out_offsets[r] + k].
__global__ void __launch_bounds__(kEncodeThreads)
split_encode_kernel(const Table t, const rk_str_col_t c, const int64_t* __restrict__ out_offsets,
                    int64_t* __restrict__ out, uint32_t* status) {
    const int lane = threadIdx.x % kWarp;
    const unsigned below_me = (1u << lane) - 1;
    const int64_t warps = (int64_t)gridDim.x * (kEncodeThreads / kWarp);
    uint32_t bits = 0;
    for (int64_t r = ((int64_t)blockIdx.x * kEncodeThreads + threadIdx.x) / kWarp; r < c.n; r += warps) {
        const int64_t b1 = __ldg(c.offsets + r + 1);
        const int64_t o0 = __ldg(out_offsets + r), cap = __ldg(out_offsets + r + 1) - o0;
        int64_t start = __ldg(c.offsets + r), item = 0;  // warp-uniform: the open item and its index
        for (int64_t base = start; base < b1; base += kWarp) {
            const int64_t p = base + lane;
            const bool sep = p < b1 && __ldg(c.bytes + p) == ',';
            const unsigned seps = __ballot_sync(kFull, sep);
            if (sep) {
                const unsigned lower = seps & below_me;
                const int64_t s = lower ? base + (31 - __clz(lower)) + 1 : start;
                const int64_t k = item + __popc(lower);
                const int64_t id = vocab_find(t, c.bytes + s, p - s, bits);
                if (k < cap) out[o0 + k] = id;
                else bits |= RK_ENCODE_SPLIT_COUNT;
            }
            if (seps) {
                start = base + (31 - __clz(seps)) + 1;
                item += __popc(seps);
            }
        }
        if (lane == 0) {
            const int64_t id = vocab_find(t, c.bytes + start, b1 - start, bits);
            if (item < cap) out[o0 + item] = id;
            if (item + 1 != cap) bits |= RK_ENCODE_SPLIT_COUNT;
        }
    }
    if (bits) atomicOr(status, bits);
}

static unsigned encode_ctas(int64_t units) {
    const int64_t ctas = ceil_div(units, kEncodeThreads);
    return (unsigned)(ctas < kEncodeMaxCtas ? ctas : kEncodeMaxCtas);
}

static Table table_of(const rk_vocab_t& v) {
    return Table{v.bytes, v.offsets, v.pos, v.slots, (uint64_t)v.n_slots - 1};
}

}  // namespace rk

static_assert(sizeof(rk_vocab_t) == 48, "rk_vocab_t layout (mirrored by _lib.RkVocab)");
static_assert(sizeof(rk_str_col_t) == 40, "rk_str_col_t layout (mirrored by _lib.RkStrCol)");

#define RK_CHECK_VOCAB(v, what)                                                                           \
    do {                                                                                                  \
        RK_CHECK_ARG(v, what ": NULL vocabulary");                                                        \
        RK_CHECK_ARG(v->bytes && v->offsets && v->pos && v->slots, what ": NULL bytes / offsets / pos / slots"); \
        RK_CHECK_ARG(v->n_keys >= 0 && v->n_keys < INT32_MAX, what ": n_keys=%lld", (long long)v->n_keys); \
        RK_CHECK_ARG(v->n_slots > 0 && (v->n_slots & (v->n_slots - 1)) == 0 && v->n_slots >= 2 * v->n_keys, \
                     what ": n_slots=%lld is not a power of two >= 2 * n_keys (%lld)", (long long)v->n_slots, \
                     (long long)v->n_keys);                                                               \
    } while (0)

#define RK_CHECK_COL(c, what)                                                                             \
    do {                                                                                                  \
        RK_CHECK_ARG(c && c->bytes && c->offsets, what ": NULL column / bytes / offsets");                \
        RK_CHECK_ARG(c->n >= 0 && c->valid_bit0 >= 0, what ": n=%lld valid_bit0=%lld", (long long)c->n,    \
                     (long long)c->valid_bit0);                                                           \
    } while (0)

extern "C" int64_t rk_vocab_slots(int64_t n_keys) {
    if (n_keys < 0 || n_keys >= INT32_MAX) return -1;
    int64_t s = 1;
    while (s < 2 * n_keys) s <<= 1;
    return s;
}

extern "C" int rk_vocab_build(const rk_vocab_t* vocab, uint32_t* status, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_VOCAB(vocab, "vocab_build");
    RK_CHECK_ARG(status, "vocab_build: NULL status");
    cudaStream_t stream = (cudaStream_t)stream_;
    RK_CUDA(cudaMemsetAsync(vocab->slots, 0xff, (size_t)vocab->n_slots * sizeof(uint64_t), stream));
    if (vocab->n_keys == 0) return 0;
    vocab_insert_kernel<<<encode_ctas(vocab->n_keys), kEncodeThreads, 0, stream>>>(
        vocab->bytes, vocab->offsets, vocab->n_keys, vocab->slots, (uint64_t)vocab->n_slots - 1, status);
    RK_LAUNCH_CHECK();
    return 0;
}

extern "C" int rk_encode_strings(const rk_vocab_t* vocab, const rk_str_col_t* col, int64_t* out,
                                 int64_t out_stride, uint32_t* status, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_VOCAB(vocab, "encode_strings");
    RK_CHECK_COL(col, "encode_strings");
    RK_CHECK_ARG(out && status, "encode_strings: NULL out / status");
    RK_CHECK_ARG(out_stride >= 1, "encode_strings: out_stride=%lld", (long long)out_stride);
    if (col->n == 0) return 0;
    encode_strings_kernel<<<encode_ctas(col->n), kEncodeThreads, 0, (cudaStream_t)stream_>>>(
        table_of(*vocab), *col, out, out_stride, status);
    RK_LAUNCH_CHECK();
    return 0;
}

extern "C" int rk_encode_split_count(const rk_str_col_t* col, int64_t* counts, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_COL(col, "encode_split_count");
    RK_CHECK_ARG(counts, "encode_split_count: NULL counts");
    if (col->n == 0) return 0;
    split_count_kernel<<<encode_ctas(col->n * kWarp), kEncodeThreads, 0, (cudaStream_t)stream_>>>(*col, counts);
    RK_LAUNCH_CHECK();
    return 0;
}

extern "C" int rk_encode_split(const rk_vocab_t* vocab, const rk_str_col_t* col, const int64_t* out_offsets,
                               int64_t* out, uint32_t* status, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_VOCAB(vocab, "encode_split");
    RK_CHECK_COL(col, "encode_split");
    RK_CHECK_ARG(out_offsets && out && status, "encode_split: NULL out_offsets / out / status");
    if (col->n == 0) return 0;
    split_encode_kernel<<<encode_ctas(col->n * kWarp), kEncodeThreads, 0, (cudaStream_t)stream_>>>(
        table_of(*vocab), *col, out_offsets, out, status);
    RK_LAUNCH_CHECK();
    return 0;
}
