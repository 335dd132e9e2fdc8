// scan_kernels.cu -- hand-written sm_100a kernels of the measure scan -> filter -> aggregate path.
//
//   plan_blocks    a1-a3  block selection: sid in query set AND [ts_min,ts_max] overlaps [tmin,tmax]
//                         (banyand/measure/part_iter.go:79-250, query.go:594-639)
//   scan_blocks    a4-a13 one warp per block: timestamps -> row range, tag pages -> row bitmask,
//                         field pages (varint / delta / delta-of-delta, decimal floats) -> per-block
//                         partial aggregates (block.go:299-418,793-870; column.go:287-364;
//                         pkg/encoding/{int.go,delta.go,float.go,dictionary.go};
//                         pkg/query/aggregation/function.go)
//   series_reduce / group_reduce   deterministic (fixed order) combine of the per-block partials
//                         into per-group partial tables (aggregation.go:193-312 fold order is
//                         replaced by a fixed tree; sums stay within the 1e-9 contract)
//   finalize       a13-a14 MEAN finalisation / output typing (function.go:31-40, aggregation.go:425-430)
//
// Pages are streamed from HBM into per-warp shared-memory stages with 1-D TMA bulk copies
// (cp.async.bulk ... mbarrier::complete_tx) and decoded with warp-shuffle scans; no tensor cores
// (there is no dense contraction on this path).
#include "scan_kernels.cuh"
#include "lane_decode.cuh"

#include <atomic>
#include <cub/device/device_merge_sort.cuh>
#include <cfloat>
#include <cmath>
#include <cstring>

#include "../../include/bydb_gpu.h"

namespace bydb {

__constant__ double c_pow10[309];  // Go math.Pow10(n), 0 <= n <= 308 (table product, see upload_pow10_table)

// ------------------------------------------------------------------------------------------------
// small PTX wrappers: mbarrier + 1-D bulk TMA
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// global -> shared bulk copy executed by the TMA unit; completion is signalled on `bar`
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ------------------------------------------------------------------------------------------------
// per-warp shared memory
// ------------------------------------------------------------------------------------------------
constexpr int kSparseQueue = BYDB_SPARSE ? 64 : 1;  // at most 32 windows of the previous chunk + 32 of the current one

struct __align__(128) WarpSmem {
    uint8_t stage[kStages][kStageBytes];
    uint64_t bar[kStages];
    uint32_t mask[kMaskWords + 4];  // +4: the fast paths read a 64- / 96-bit window at the last word
    uint32_t match[8];  // dictionary match set of the predicate being applied
    uint32_t fault;     // set when a TMA wait timed out
    uint32_t seq;       // warp-monotonic count of the TMA stages issued so far (mbarrier phase bookkeeping)
    // result slot of the out-of-line page decoders: handing an accumulator over by reference would put it (and the
    // caller's live registers) into local memory; shared memory costs one broadcast load per field instead
    unsigned long long res_lo;
    long long res_hi, res_mn, res_mx;
    uint32_t res_cnt;
    // argument slot of the same calls (more than a handful of arguments would be marshalled through local memory)
    uint32_t a_len;
    const uint8_t *a_body;
    long long a_first;
    uint32_t a_count, a_r0, a_r1;
    int res_exp;                 // decimal exponent of the page just aggregated (kExpRawFloat for raw float cells)
    const uint8_t *a_page;       // arguments of agg_field_page
    uint32_t a_size, a_flags;    // a_flags: bit 0 = float64 field, bits 1.. = kNeed*
    // the warp's statistics (lane 0 only), flushed to the query's counters once when the warp runs out of work
    unsigned long long st_rows, st_matched, st_bytes;
    uint32_t st_blocks, st_deferred, st_why, pad2;
    // delta_page_sparse: the lane windows that hold an active row, waiting to be decoded 32 at a time
    unsigned long long q_desc[kSparseQueue];  // ring offset | valid range | tail of the previous window (see sparse_desc)
    long long q_base[kSparseQueue];           // value in front of the window's first ending value
    unsigned long long q_aw[kSparseQueue];    // bit i = the i-th value that ends in the window is an active row
};

size_t scan_smem_bytes() { return sizeof(WarpSmem) * kWarpsPerCta; }


struct PageStream {
    const uint8_t *abase;  // 16 B aligned global address at or below the first body byte
    uint32_t total;        // aligned length (multiple of 16)
    uint32_t pstart, pend; // valid byte range inside [0,total)
    uint32_t nstages;
    uint32_t seq0;         // warp-monotonic stage sequence number of stage 0
};

__device__ __forceinline__ void stream_issue(const PageStream &s, WarpSmem *sm, uint32_t k) {
    uint32_t off = k * kStageBytes;
    uint32_t bytes = min(static_cast<uint32_t>(kStageBytes), s.total - off);
    uint32_t slot = (s.seq0 + k) % kStages;
    mbar_expect_tx(&sm->bar[slot], bytes);
    tma_load_1d(sm->stage[slot], s.abase + off, bytes, &sm->bar[slot]);
}
__device__ __forceinline__ void stream_open(PageStream &s, WarpSmem *sm, const uint8_t *body, uint32_t len, int lane) {
    uintptr_t a = reinterpret_cast<uintptr_t>(body);
    s.abase = reinterpret_cast<const uint8_t *>(a & ~static_cast<uintptr_t>(15));
    s.pstart = static_cast<uint32_t>(a & 15);
    s.pend = s.pstart + len;
    s.total = (s.pend + 15u) & ~15u;
    s.nstages = (s.total + kStageBytes - 1) / kStageBytes;
    s.seq0 = sm->seq;
    __syncwarp();  // every lane is done reading the stages of the previous page (and sm->seq)
    if (lane == 0) {
        sm->seq = s.seq0 + s.nstages;
        uint32_t n = min(s.nstages, static_cast<uint32_t>(kStages));
        for (uint32_t k = 0; k < n; ++k) stream_issue(s, sm, k);
    }
}
__device__ __forceinline__ const uint8_t *stream_wait(const PageStream &s, WarpSmem *sm, uint32_t k) {
    uint32_t n = s.seq0 + k;
    uint32_t slot = n % kStages;
    uint32_t parity = (n / kStages) & 1u;
    // bounded spin: a lost transaction must surface as an error, never as a hung GPU
    for (uint32_t spins = 0; !mbar_try_wait(&sm->bar[slot], parity); ++spins) {
        if (spins > (1u << 24)) {
            sm->fault = 1;
            break;
        }
    }
    return sm->stage[slot];
}
__device__ __forceinline__ void stream_release(const PageStream &s, WarpSmem *sm, uint32_t k, int lane) {
    __syncwarp();
    if (lane == 0 && k + kStages < s.nstages) stream_issue(s, sm, k + kStages);
}

// ------------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t zigzag64(uint64_t u) { return static_cast<int64_t>(u >> 1) ^ -static_cast<int64_t>(u & 1); }

__device__ __forceinline__ uint64_t shfl_u64(uint64_t v, int src) {
    uint32_t lo = __shfl_sync(0xffffffffu, static_cast<uint32_t>(v), src);
    uint32_t hi = __shfl_sync(0xffffffffu, static_cast<uint32_t>(v >> 32), src);
    return (static_cast<uint64_t>(hi) << 32) | lo;
}
__device__ __forceinline__ uint64_t shfl_up_u64(uint64_t v, int delta) {
    uint32_t lo = __shfl_up_sync(0xffffffffu, static_cast<uint32_t>(v), delta);
    uint32_t hi = __shfl_up_sync(0xffffffffu, static_cast<uint32_t>(v >> 32), delta);
    return (static_cast<uint64_t>(hi) << 32) | lo;
}
__device__ __forceinline__ uint64_t shfl_xor_u64(uint64_t v, int m) {
    uint32_t lo = __shfl_xor_sync(0xffffffffu, static_cast<uint32_t>(v), m);
    uint32_t hi = __shfl_xor_sync(0xffffffffu, static_cast<uint32_t>(v >> 32), m);
    return (static_cast<uint64_t>(hi) << 32) | lo;
}

// pkg/convert/number.go:93-106 BytesToInt64 (order-preserving form, NOT two's complement)
__device__ __forceinline__ int64_t conv_bytes_to_int64(const uint8_t *b) {
    uint64_t u = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) u = (u << 8) | __ldg(b + k);
    if (u >> 63) return static_cast<int64_t>(u ^ (1ull << 63));
    return static_cast<int64_t>(0ull - ((1ull << 63) - u));
}

// pkg/encoding/int.go:111-148: one zig-zag varint read sequentially (headers only)
__device__ __forceinline__ bool read_varint_seq(const uint8_t *p, uint32_t len, int64_t &out, uint32_t &used) {
    uint64_t u = 0;
    for (uint32_t i = 0; i < len && i < 10; ++i) {
        uint8_t c = __ldg(p + i);
        u |= static_cast<uint64_t>(c & 0x7f) << (7 * i);
        if (c < 0x80) {
            out = zigzag64(u);
            used = i + 1;
            return true;
        }
    }
    return false;
}
__device__ __forceinline__ bool read_varuint_seq(const uint8_t *&p, const uint8_t *end, uint64_t &out) {
    uint64_t u = 0;
    for (uint32_t i = 0; i < 10 && p < end; ++i) {
        uint8_t c = __ldg(p++);
        u |= static_cast<uint64_t>(c & 0x7f) << (7 * i);
        if (c < 0x80) {
            out = u;
            return true;
        }
    }
    return false;
}

__device__ __forceinline__ void set_err(const ScanParams &p, uint32_t code, uint32_t g, int lane) {
    if (lane == 0 && atomicCAS(&p.err[0], 0u, code) == 0u) p.err[1] = g;
}

// pkg/encoding/float.go:69-93: int64 -> float64 by the page exponent; exactly the reference's
// operation sequence (float64(v) * Pow10(e), or float64(v) / d1 / d2 ... with d_i = 10^min(rem,308)).
__device__ __forceinline__ double scale_decimal(double x, int exp) {
    if (exp >= 0) {
        double s = exp <= 308 ? c_pow10[exp] : INFINITY;
        return __dmul_rn(x, s);
    }
    int neg = -exp;
    while (neg > 0) {
        int step = neg < 308 ? neg : 308;
        x = __ddiv_rn(x, c_pow10[step]);
        neg -= step;
    }
    return x;
}

// ------------------------------------------------------------------------------------------------
// row consumers
// ------------------------------------------------------------------------------------------------
enum { kRowsAll = 0, kRowsRange = 1, kRowsMask = 2 };

struct AggAcc {
    uint64_t lo;
    int64_t hi;  // 128-bit exact sum (a block holds <= 2^31 rows of int64)
    int64_t mn, mx;
    uint32_t cnt;
    __device__ __forceinline__ void init() {
        lo = 0;
        hi = 0;
        mn = INT64_MAX;
        mx = INT64_MIN;
        cnt = 0;
    }
    __device__ __forceinline__ void add(int64_t v) {
        uint64_t uv = static_cast<uint64_t>(v);
        lo += uv;
        hi += (v >> 63) + (lo < uv ? 1 : 0);
        mn = v < mn ? v : mn;
        mx = v > mx ? v : mx;
        cnt++;
    }
    __device__ __forceinline__ void add_scaled(int64_t v, uint64_t times) {  // += v * times (exact)
        uint64_t a = static_cast<uint64_t>(v);
        uint64_t plo = a * times;
        int64_t phi = static_cast<int64_t>(__umul64hi(a, times)) - (v < 0 ? static_cast<int64_t>(times) : 0);
        lo += plo;
        hi += phi + (lo < plo ? 1 : 0);
    }
    __device__ __forceinline__ void warp_reduce() {
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            uint64_t olo = shfl_xor_u64(lo, m);
            int64_t ohi = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(hi), m));
            int64_t omn = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(mn), m));
            int64_t omx = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(mx), m));
            uint32_t ocnt = __shfl_xor_sync(0xffffffffu, cnt, m);
            lo += olo;
            hi += ohi + (lo < olo ? 1 : 0);
            mn = omn < mn ? omn : mn;
            mx = omx > mx ? omx : mx;
            cnt += ocnt;
        }
    }
};

// the out-of-line fast decoders leave their (warp-reduced) result in the warp's shared-memory slot
__device__ __forceinline__ void publish_acc(WarpSmem *sm, AggAcc &acc, int lane) {
    acc.warp_reduce();
    if (lane == 0) {
        sm->res_lo = acc.lo;
        sm->res_hi = acc.hi;
        sm->res_mn = acc.mn;
        sm->res_mx = acc.mx;
        sm->res_cnt = acc.cnt;
    }
    __syncwarp();
}
// an accumulator that is already warp-reduced (every lane holds the total)
__device__ __forceinline__ void store_acc(WarpSmem *sm, const AggAcc &acc, int lane) {
    __syncwarp();
    if (lane == 0) {
        sm->res_lo = acc.lo;
        sm->res_hi = acc.hi;
        sm->res_mn = acc.mn;
        sm->res_mx = acc.mx;
        sm->res_cnt = acc.cnt;
    }
    __syncwarp();
}
__device__ __forceinline__ void fetch_acc(const WarpSmem *sm, AggAcc &acc) {
    acc.lo = sm->res_lo;
    acc.hi = sm->res_hi;
    acc.mn = sm->res_mn;
    acc.mx = sm->res_mx;
    acc.cnt = sm->res_cnt;
}

// general-path consumer: the row mode is a runtime value to keep one instantiation of the decoder
struct AggCons {
    AggAcc acc;
    uint32_t r0, r1;
    const uint32_t *mask;
    int mode;
    __device__ __forceinline__ void operator()(uint32_t row, int64_t v) {
        bool a = row >= r0 && row <= r1;
        if (mode == kRowsMask) a = row < kMaskWords * 32 && ((mask[row >> 5] >> (row & 31)) & 1u);
        if (a) acc.add(v);
    }
};

// counts rows with ts < tmin and ts <= tmax (pkg/timestamp/range.go:143-169 on an ascending block)
struct TsCons {
    int64_t tmin, tmax;
    uint32_t lt, le;
    __device__ __forceinline__ void operator()(uint32_t, int64_t v) {
        lt += v < tmin ? 1u : 0u;
        le += v <= tmax ? 1u : 0u;
    }
};

__device__ __forceinline__ bool cmp_op(int op, bool have, int cmp) {
    switch (op) {
        case BYDB_OP_EQ: return have && cmp == 0;
        case BYDB_OP_NE: return !have || cmp != 0;
        case BYDB_OP_LT: return have && cmp < 0;
        case BYDB_OP_LE: return have && cmp <= 0;
        case BYDB_OP_GT: return have && cmp > 0;
        case BYDB_OP_GE: return have && cmp >= 0;
        case kOpEqOrNil: return !have || cmp == 0;
    }
    return false;
}

// int64 tag predicate: clears the mask bit of every non-matching row
struct CmpCons {
    int64_t lit;
    int op;
    uint32_t *mask;
    uint32_t limit;  // rows the mask can hold
    __device__ __forceinline__ void operator()(uint32_t row, int64_t v) {
        int c = v < lit ? -1 : (v > lit ? 1 : 0);
        if (!cmp_op(op, true, c) && row < limit) atomicAnd(&mask[row >> 5], ~(1u << (row & 31)));
    }
};

// ------------------------------------------------------------------------------------------------
// the varint page decoder (pkg/encoding/int.go:111-148 + delta.go:45-70 / :91-118)
//
// One warp; every iteration takes 512 B (16 B per lane) of the body from the staged shared-memory
// tile.  A lane decodes the varints that END inside its 16 bytes; the low bits of a value that
// started in the previous lane arrive by one shuffle of that lane's unfinished tail.  Row indices
// come from a warp scan of the per-lane terminator counts, value prefixes from a warp scan of the
// per-lane delta sums (delta) or of the (count, sum, sum-of-prefix) triple (delta-of-delta).  All
// int64 arithmetic wraps mod 2^64 like Go's, so the result is bit-exact.
// ------------------------------------------------------------------------------------------------
template <bool kDod, class Cons>
__device__ __noinline__ bool decode_varint_page(WarpSmem *sm, const uint8_t *body, uint32_t len, uint32_t count,
                                                 int64_t first, Cons &cons_io, int lane) {
    Cons cons = cons_io;  // register copy: the by-reference object of a noinline call lives in local memory
    if (lane == 0) cons(0u, first);
    if (len == 0) {
        cons_io = cons;
        return count == 1;
    }
    PageStream st;
    stream_open(st, sm, body, len, lane);
    const uint32_t nchunks = (st.total + kChunkBytes - 1) / kChunkBytes;
    constexpr uint32_t kChunksPerStage = kStageBytes / kChunkBytes;
    int64_t V0 = first;  // value of the row before this chunk's first varint (warp-uniform)
    int64_t D0 = 0;      // delta-of-delta: running first difference
    uint64_t carry_acc = 0;
    uint32_t carry_sh = 0;
    uint32_t row_base = 1;
    const uint8_t *buf = nullptr;
    for (uint32_t c = 0; c < nchunks; ++c) {
        const uint32_t k = c / kChunksPerStage;
        if ((c % kChunksPerStage) == 0) buf = stream_wait(st, sm, k);
        const uint32_t o = c * kChunkBytes + lane * 16;
        uint4 w = make_uint4(0, 0, 0, 0);
        if (o < st.total) w = *reinterpret_cast<const uint4 *>(buf + (o % kStageBytes));
        // valid bytes of this lane: [pstart,pend) intersected with [o,o+16)
        int lo_i = static_cast<int>(st.pstart) - static_cast<int>(o);
        int hi_i = static_cast<int>(st.pend) - static_cast<int>(o);
        lo_i = lo_i < 0 ? 0 : (lo_i > 16 ? 16 : lo_i);
        hi_i = hi_i < 0 ? 0 : (hi_i > 16 ? 16 : hi_i);
        const uint32_t valid = ((1u << hi_i) - 1u) & ~((1u << lo_i) - 1u);
        const uint32_t msb = msb4(w.x) | (msb4(w.y) << 4) | (msb4(w.z) << 8) | (msb4(w.w) << 12);
        const uint32_t term = valid & ~msb;
        const uint32_t n = __popc(term);

        // ---- pass A: lane-local sums; the head value is decoded from this lane's bytes only and
        //      corrected below by what the previous lane's unfinished tail contributes
        uint64_t acc = 0;
        uint32_t sh = 0;
        uint64_t head_x = 0;
        bool seen = false;
        int64_t q = 0;  // sum of this lane's values
        int64_t r = 0;  // delta-of-delta: sum of the running prefixes
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const uint32_t wj = j < 4 ? w.x : (j < 8 ? w.y : (j < 12 ? w.z : w.w));
            const uint32_t b = (wj >> (8 * (j & 3))) & 0xffu;
            if ((valid >> j) & 1u) {
                acc |= static_cast<uint64_t>(b & 0x7fu) << (sh & 63u);
                sh += 7;
            }
            if ((term >> j) & 1u) {
                if (!seen) {
                    head_x = acc;
                    seen = true;
                }
                q += zigzag64(acc);
                if (kDod) r += q;
                acc = 0;
                sh = 0;
            }
        }
        uint64_t prev_acc = shfl_up_u64(acc, 1);
        uint32_t prev_sh = __shfl_up_sync(0xffffffffu, sh, 1);
        if (lane == 0) {
            prev_acc = carry_acc;
            prev_sh = carry_sh;
        }
        carry_acc = shfl_u64(acc, 31);
        carry_sh = __shfl_sync(0xffffffffu, sh, 31);
        if (n > 0 && prev_sh != 0) {
            const int64_t dlt = zigzag64(prev_acc | (head_x << (prev_sh & 63u))) - zigzag64(head_x);
            q += dlt;
            if (kDod) r += static_cast<int64_t>(static_cast<uint64_t>(n) * static_cast<uint64_t>(dlt));
        }
        // ---- warp scans (inclusive), then exclusive views
        uint32_t n_in = n;
        int64_t q_in = q, r_in = r;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            uint32_t on = __shfl_up_sync(0xffffffffu, n_in, s);
            int64_t oq = static_cast<int64_t>(shfl_up_u64(static_cast<uint64_t>(q_in), s));
            int64_t orr = 0;
            if (kDod) orr = static_cast<int64_t>(shfl_up_u64(static_cast<uint64_t>(r_in), s));
            if (lane >= s) {
                // (A then B): n = nA+nB, q = qA+qB, r = rA + rB + nB*qA
                if (kDod) r_in = orr + r_in + static_cast<int64_t>(static_cast<uint64_t>(n_in) * static_cast<uint64_t>(oq));
                q_in += oq;
                n_in += on;
            }
        }
        const uint32_t n_ex = n_in - n;
        int64_t q_ex = static_cast<int64_t>(shfl_up_u64(static_cast<uint64_t>(q_in), 1));
        int64_t r_ex = 0;
        if (kDod) r_ex = static_cast<int64_t>(shfl_up_u64(static_cast<uint64_t>(r_in), 1));
        if (lane == 0) {
            q_ex = 0;
            r_ex = 0;
        }
        // ---- pass B: decode again, now starting from the previous lane's tail, with the true base
        uint32_t row = row_base + n_ex;
        int64_t D = D0 + q_ex;
        int64_t v = kDod ? V0 + static_cast<int64_t>(static_cast<uint64_t>(n_ex) * static_cast<uint64_t>(D0)) + r_ex : V0 + q_ex;
        acc = prev_acc;
        sh = prev_sh;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const uint32_t wj = j < 4 ? w.x : (j < 8 ? w.y : (j < 12 ? w.z : w.w));
            const uint32_t b = (wj >> (8 * (j & 3))) & 0xffu;
            if ((valid >> j) & 1u) {
                acc |= static_cast<uint64_t>(b & 0x7fu) << (sh & 63u);
                sh += 7;
            }
            if ((term >> j) & 1u) {
                const int64_t x = zigzag64(acc);
                if (kDod) {
                    D += x;
                    v += D;
                } else {
                    v += x;
                }
                cons(row, v);
                row++;
                acc = 0;
                sh = 0;
            }
        }
        // ---- carries to the next chunk
        const uint32_t n_tot = __shfl_sync(0xffffffffu, n_in, 31);
        const int64_t q_tot = static_cast<int64_t>(shfl_u64(static_cast<uint64_t>(q_in), 31));
        if (!kDod) {
            V0 += q_tot;
        } else {
            const int64_t r_tot = static_cast<int64_t>(shfl_u64(static_cast<uint64_t>(r_in), 31));
            V0 += static_cast<int64_t>(static_cast<uint64_t>(n_tot) * static_cast<uint64_t>(D0)) + r_tot;
            D0 += q_tot;
        }
        row_base += n_tot;
        if ((c % kChunksPerStage) == kChunksPerStage - 1 || c == nchunks - 1) stream_release(st, sm, k, lane);
    }
    cons_io = cons;
    // the body must hold exactly count-1 varints and end on a terminator
    return row_base == count && carry_sh == 0;
}

// ------------------------------------------------------------------------------------------------
// Fast path: EncodeTypeDelta pages whose varints are all <= 3 bytes (|delta| < 2^20 -- the common case
// for metric pages).  One pass per 512 B chunk, everything in 32-bit registers:
//   * a lane decodes its values with no dependency on its neighbour (the head value is decoded from
//     this lane's bytes only and corrected afterwards by the difference the neighbour's tail makes),
//   * it keeps the running LOCAL prefix P_j of its deltas and folds the active rows into
//     (sum of P_j, min P_j, max P_j, count) -- |P_j| < 2^24, so int32 cannot wrap and order is preserved,
//   * one warp scan of the per-lane totals gives the lane's base value; the lane then contributes
//     cnt*base + sum(P), base + min(P), base + max(P) -- exactly the values of the two-pass decoder.
// Returns 0 = done, 1 = a chunk with a longer varint was met (caller re-runs the general decoder
// on the whole page), 2 = corrupt.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void stream_drain(const PageStream &s, WarpSmem *sm, uint32_t k) {
    const uint32_t issued = min(s.nstages, k + static_cast<uint32_t>(kStages));
    for (uint32_t j = k + 1; j < issued; ++j) (void)stream_wait(s, sm, j);
}

// (the lane-level decoders live in lane_decode.cuh: they are plain per-lane functions, also compiled for the host by
// tests/native/lane_decode_test.cc)

// per-chunk front end shared by the two fast decoders: load 32 B per lane, byte masks, narrow check
struct FastChunk {
    uint4 wa, wb;
    uint32_t valid, term, n;
    bool wide;
};

__device__ __forceinline__ void fast_chunk_load(FastChunk &fc, const PageStream &st, const uint8_t *buf, uint32_t c, uint32_t carry_sh, int lane) {
    const uint32_t o = c * kFastChunkBytes + lane * kFastLaneBytes;
    fc.wa = make_uint4(0, 0, 0, 0);
    fc.wb = make_uint4(0, 0, 0, 0);
    if (o < st.total) fc.wa = *reinterpret_cast<const uint4 *>(buf + (o % kStageBytes));
    if (o + 16 < st.total) fc.wb = *reinterpret_cast<const uint4 *>(buf + (o % kStageBytes) + 16);
    int lo_i = static_cast<int>(st.pstart) - static_cast<int>(o);
    int hi_i = static_cast<int>(st.pend) - static_cast<int>(o);
    lo_i = lo_i < 0 ? 0 : (lo_i > 32 ? 32 : lo_i);
    hi_i = hi_i < 0 ? 0 : (hi_i > 32 ? 32 : hi_i);
    fc.valid = low_bits(hi_i) & ~low_bits(lo_i);
    // nibbles gathered with multiply-adds (FMA pipe) instead of shift+or pairs (ALU pipe)
    uint32_t msb = msb4(fc.wa.x);
    msb = imad_u32(msb4(fc.wa.y), 1u << 4, msb);
    msb = imad_u32(msb4(fc.wa.z), 1u << 8, msb);
    msb = imad_u32(msb4(fc.wa.w), 1u << 12, msb);
    msb = imad_u32(msb4(fc.wb.x), 1u << 16, msb);
    msb = imad_u32(msb4(fc.wb.y), 1u << 20, msb);
    msb = imad_u32(msb4(fc.wb.z), 1u << 24, msb);
    msb = imad_u32(msb4(fc.wb.w), 1u << 28, msb);
    fc.term = fc.valid & ~msb;
    const uint32_t cont = fc.valid & msb;
    fc.n = __popc(fc.term);
    // longest varint check: no run of 3 continuation bytes inside the lane, and the run that
    // crosses from the previous lane (its trailing continuation bytes + our leading ones) <= 2
    const uint32_t lead = fc.term ? static_cast<uint32_t>(__ffs(fc.term) - 1 - lo_i) : static_cast<uint32_t>(hi_i - lo_i);
    const uint32_t trail = fc.term ? static_cast<uint32_t>(hi_i - 1 - (31 - __clz(fc.term))) : static_cast<uint32_t>(hi_i - lo_i);
    uint32_t trail_prev = __shfl_up_sync(0xffffffffu, trail, 1);
    if (lane == 0) trail_prev = carry_sh / 7;
    fc.wide = __any_sync(0xffffffffu, (cont & (cont >> 1) & (cont >> 2)) != 0 || (trail_prev + lead) > 2);
}

// rows of the lane -> bit i of the result = i-th value of this lane is an active row
template <int kMode>
__device__ __forceinline__ uint32_t fast_active_window(const WarpSmem *sm, uint32_t row0, uint32_t n, uint32_t r0, uint32_t r1) {
    if (kMode == kRowsAll) return low_bits(n);
    if (kMode == kRowsRange) {
        const uint32_t a = r0 > row0 ? r0 - row0 : 0u;
        const uint32_t b = (r1 + 1u) < (row0 + n) ? (r1 + 1u > row0 ? r1 + 1u - row0 : 0u) : n;
        return a < b ? (low_bits(b) & ~low_bits(a)) : 0u;
    }
    // a corrupt page can hold more varints than the block has rows: never index past the mask
    const uint32_t wi = min(row0 >> 5, static_cast<uint32_t>(kMaskWords));
    const uint64_t m64 = static_cast<uint64_t>(sm->mask[wi]) | (static_cast<uint64_t>(sm->mask[wi + 1]) << 32);
    return static_cast<uint32_t>(m64 >> (row0 & 31)) & low_bits(n);
}

template <int kMode, int kNeed>
__device__ __noinline__ int delta_page_fast(WarpSmem *sm, int lane) {
    const uint8_t *body = sm->a_body;
    const uint32_t len = sm->a_len, count = sm->a_count, r0 = sm->a_r0, r1 = sm->a_r1;
    const int64_t first = sm->a_first;
    AggAcc acc;
    acc.init();
    if (lane == 0) {
        bool a = true;
        if (kMode == kRowsRange) a = r0 == 0;
        if (kMode == kRowsMask) a = sm->mask[0] & 1u;
        if (a) acc.add(first);
    }
    if (len == 0) {
        publish_acc(sm, acc, lane);
        return count == 1 ? 0 : 2;
    }
    PageStream st;
    stream_open(st, sm, body, len, lane);
    const uint32_t nchunks = (st.total + kFastChunkBytes - 1) / kFastChunkBytes;
    constexpr uint32_t kChunksPerStage = kStageBytes / kFastChunkBytes;
    int64_t V0 = first;
    uint32_t carry_acc = 0, carry_sh = 0;
    uint32_t row_base = 1;
    const uint8_t *buf = nullptr;
    for (uint32_t c = 0; c < nchunks; ++c) {
        const uint32_t k = c / kChunksPerStage;
        if ((c % kChunksPerStage) == 0) buf = stream_wait(st, sm, k);
        FastChunk fc;
        fast_chunk_load(fc, st, buf, c, carry_sh, lane);
        if (fc.wide) {
            // give the unissued stage numbers back: the mbarrier phases only advance for stages that
            // were really issued, and the next page must continue from exactly that count
            stream_drain(st, sm, k);
            if (lane == 0) sm->seq = st.seq0 + min(st.nstages, k + static_cast<uint32_t>(kStages));
            __syncwarp();
            return 1;
        }
        const uint32_t n = fc.n;
        // rows of this lane (only the masked / ranged modes need the per-lane row index)
        uint32_t n_tot, aw;
        if (kMode == kRowsAll) {
            n_tot = __reduce_add_sync(0xffffffffu, n);
            aw = low_bits(n);
        } else {
            uint32_t n_in = n;
#pragma unroll
            for (int s = 1; s < 32; s <<= 1) {
                const uint32_t on = __shfl_up_sync(0xffffffffu, n_in, s);
                if (lane >= s) n_in += on;
            }
            n_tot = __shfl_sync(0xffffffffu, n_in, 31);
            aw = fast_active_window<kMode>(sm, row_base + n_in - n, n, r0, r1);
        }
        const uint32_t cntA = __popc(aw);
        // ---- decode: local prefix P, folded over the active rows
        uint32_t accv = 0, sh = 0;
        int32_t P = 0, sumP = 0, minP = INT32_MAX, maxP = INT32_MIN;
        const bool full_chunk = __all_sync(0xffffffffu, fc.valid == 0xffffffffu);
        if (full_chunk) fast_lane_decode<true, kNeed>(fc.wa, fc.wb, fc.valid, fc.term, aw, accv, sh, P, sumP, minP, maxP);
        else fast_lane_decode<false, kNeed>(fc.wa, fc.wb, fc.valid, fc.term, aw, accv, sh, P, sumP, minP, maxP);
        // ---- head correction by the previous lane's unfinished tail
        uint32_t prev_acc = __shfl_up_sync(0xffffffffu, accv, 1);
        uint32_t prev_sh = __shfl_up_sync(0xffffffffu, sh, 1);
        if (lane == 0) {
            prev_acc = carry_acc;
            prev_sh = carry_sh;
        }
        carry_acc = __shfl_sync(0xffffffffu, accv, 31);
        carry_sh = __shfl_sync(0xffffffffu, sh, 31);
        if (n > 0 && prev_sh != 0) {
            const int32_t dlt = head_delta(fc.wa.x, fc.term, prev_acc, prev_sh);
            P += dlt;
            if (kNeed & kNeedSum) sumP += dlt * static_cast<int32_t>(cntA);
            if ((kNeed & kNeedMinMax) && cntA) {
                minP += dlt;
                maxP += dlt;
            }
        }
        // ---- base value of the lane: scan of the lane totals
        int32_t s_in = P;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const int32_t os = __shfl_up_sync(0xffffffffu, s_in, s);
            if (lane >= s) s_in += os;
        }
        const int64_t base = V0 + static_cast<int64_t>(s_in - P);
        if (cntA) {
            if (kNeed & kNeedSum) {
                acc.add_scaled(base, cntA);
                const int64_t sp = sumP;
                const uint64_t usp = static_cast<uint64_t>(sp);
                acc.lo += usp;
                acc.hi += (sp >> 63) + (acc.lo < usp ? 1 : 0);
            }
            if (kNeed & kNeedMinMax) {
                const int64_t vmin = base + minP, vmax = base + maxP;
                acc.mn = vmin < acc.mn ? vmin : acc.mn;
                acc.mx = vmax > acc.mx ? vmax : acc.mx;
            }
            acc.cnt += cntA;
        }
        V0 += static_cast<int64_t>(__shfl_sync(0xffffffffu, s_in, 31));
        row_base += n_tot;
        if ((c % kChunksPerStage) == kChunksPerStage - 1 || c == nchunks - 1) stream_release(st, sm, k, lane);
    }
    publish_acc(sm, acc, lane);
    return (row_base == count && carry_sh == 0) ? 0 : 2;
}

// One 2 KB chunk of a delta page through the SWAR lane decoder: loads the lane's 64 bytes from the staged tile, hands the
// neighbour's last word on, and returns the lane's terminator count n, its byte-linear sums T / R' and the wide flag.
// c: chunk index inside the page window; carry_w: the (masked) last word of the previous chunk, updated.
struct SwarChunk {
    int32_t T, Rp;
    uint32_t n;
    bool wide;
};
// 2 KB per warp iteration, 64 contiguous bytes per lane: the per-chunk work (neighbour shuffle, vote, scan of the terminator
// counts, 64-bit multiply-add, stage bookkeeping: ~160 instructions) is paid once per 16 words instead of once per 8.
constexpr uint32_t kSwarLaneBytes = 64;
constexpr uint32_t kSwarChunkBytes = 32 * kSwarLaneBytes;
static_assert(kStageBytes % kSwarChunkBytes == 0, "a TMA stage holds whole SWAR chunks");
// The lane's 16 words through swar_word.  va / vb: valid bytes 0..31 / 32..63 of a first / last chunk of a page.  The
// three-class pass only runs again over a chunk that holds a class-2 byte (rare), so it stays rolled to keep code small.
template <bool kTwoClass>
__device__ __forceinline__ void swar_chunk_pass(SwarLane &sl, const uint8_t *src, bool interior, uint32_t o, uint32_t total, uint32_t va, uint32_t vb,
                                                uint32_t pw) {
    swar_begin(sl, pw);
    if (interior) {
        // the two halves one after the other so that only 8 data words are live at a time
#pragma unroll(kTwoClass ? 2 : 1)
        for (int half = 0; half < 2; ++half) {
            const uint4 wa = *reinterpret_cast<const uint4 *>(src + 32 * half), wb = *reinterpret_cast<const uint4 *>(src + 32 * half + 16);
            swar_word<false, kTwoClass>(sl, wa.x, 0u);
            swar_word<false, kTwoClass>(sl, wa.y, 0u);
            swar_word<false, kTwoClass>(sl, wa.z, 0u);
            swar_word<false, kTwoClass>(sl, wa.w, 0u);
            swar_word<false, kTwoClass>(sl, wb.x, 0u);
            swar_word<false, kTwoClass>(sl, wb.y, 0u);
            swar_word<false, kTwoClass>(sl, wb.z, 0u);
            swar_word<false, kTwoClass>(sl, wb.w, 0u);
        }
    } else {
#pragma unroll(kTwoClass ? 4 : 1)
        for (int q = 0; q < 4; ++q) {
            uint4 w = make_uint4(0, 0, 0, 0);
            if (o + 16 * q < total) w = *reinterpret_cast<const uint4 *>(src + 16 * q);
            const uint32_t v = (q < 2 ? va : vb) >> (16 * (q & 1));
            swar_word<true, kTwoClass>(sl, w.x, expand4(v));
            swar_word<true, kTwoClass>(sl, w.y, expand4(v >> 4));
            swar_word<true, kTwoClass>(sl, w.z, expand4(v >> 8));
            swar_word<true, kTwoClass>(sl, w.w, expand4(v >> 12));
        }
    }
}
// The two-class pass first; when a byte of the chunk is of class 2 (a lane's guard, or the previous chunk ending in two
// continuation bytes) the warp decodes the chunk again with the three-class word, which also raises `wide`.  Either way
// n, T and R' are those of the three-class word.
__device__ __forceinline__ SwarChunk swar_chunk(const uint8_t *buf, uint32_t c, uint32_t pstart, uint32_t pend, uint32_t total, uint32_t &carry_w, int lane) {
    const uint32_t o = c * kSwarChunkBytes + lane * kSwarLaneBytes;
    const bool interior = c * kSwarChunkBytes >= pstart && (c + 1) * kSwarChunkBytes <= pend;  // warp-uniform
    const uint8_t *src = buf + (o % kStageBytes);
    uint32_t va = 0xffffffffu, vb = 0xffffffffu, lastw;
    if (interior) {
        lastw = *reinterpret_cast<const uint32_t *>(src + kSwarLaneBytes - 4);
    } else {
        int lo_i = static_cast<int>(pstart) - static_cast<int>(o);
        int hi_i = static_cast<int>(pend) - static_cast<int>(o);
        lo_i = lo_i < 0 ? 0 : (lo_i > 64 ? 64 : lo_i);
        hi_i = hi_i < 0 ? 0 : (hi_i > 64 ? 64 : hi_i);
        va = low_bits(hi_i > 32 ? 32 : hi_i) & ~low_bits(lo_i > 32 ? 32 : lo_i);               // bytes 0..31
        vb = low_bits(hi_i > 32 ? hi_i - 32 : 0) & ~low_bits(lo_i > 32 ? lo_i - 32 : 0);       // bytes 32..63
        lastw = o + 48 < total ? *reinterpret_cast<const uint32_t *>(src + kSwarLaneBytes - 4) & expand4(vb >> 28) : 0u;
    }
    // the neighbour only needs this lane's last word: it is fetched first
    uint32_t pw = __shfl_up_sync(0xffffffffu, lastw, 1);
    const uint32_t cw = carry_w;
    if (lane == 0) pw = cw;
    carry_w = __shfl_sync(0xffffffffu, lastw, 31);
    SwarLane sl;
    swar_chunk_pass<true>(sl, src, interior, o, total, va, vb, pw);
    SwarChunk r;
    r.wide = false;
    if (__any_sync(0xffffffffu, (sl.guard & 0x80808080u) != 0) || swar_opens_class2(cw)) {
        swar_chunk_pass<false>(sl, src, interior, o, total, va, vb, pw);
        r.wide = __any_sync(0xffffffffu, (sl.wide & 0x80808080u) != 0);
    }
    r.n = swar_end(sl, r.T, r.Rp);
    return r;
}

// ------------------------------------------------------------------------------------------------
// SWAR sum decoder: EncodeTypeDelta page, every row active, only SUM / MEAN / COUNT wanted (the group-by-sum shape of
// BASELINE configs 3/4).  See lane_decode.cuh (swar_word): the page sum is a weighted sum over BYTES, so nothing is
// carried from byte to byte or from lane to lane except the count of terminators; per 1 KB chunk the warp does one
// shuffle of the neighbour's last word, 8 x swar_word per lane, one scan of the lanes' terminator counts and one
// 64-bit multiply-add.  Returns like delta_page_fast (0 done / 1 a varint of 4+ bytes was met / 2 corrupt).
// ------------------------------------------------------------------------------------------------
__device__ __noinline__ int delta_page_sum_all(WarpSmem *sm, int lane) {
    const uint8_t *body = sm->a_body;
    const uint32_t len = sm->a_len, count = sm->a_count;
    const int64_t first = sm->a_first;
    AggAcc acc;
    acc.init();
    if (lane == 0) {
        acc.add_scaled(first, count);  // n * first, exact in 128 bits
        acc.cnt = count;
    }
    if (len == 0) {
        publish_acc(sm, acc, lane);
        return count == 1 ? 0 : 2;
    }
    PageStream st;
    stream_open(st, sm, body, len, lane);
    const uint32_t nchunks = (st.total + kSwarChunkBytes - 1) / kSwarChunkBytes;
    constexpr uint32_t kChunksPerStage = kStageBytes / kSwarChunkBytes;
    int64_t S = 0;                 // this lane's share of  sum_j d_j * (n - j)
    uint32_t tb = 0, carry_w = 0;  // terminators before this chunk; last (masked) word of the previous chunk
    uint32_t last_byte = 0;
    const uint8_t *buf = nullptr;
    for (uint32_t c = 0; c < nchunks; ++c) {
        const uint32_t k = c / kChunksPerStage;
        if ((c % kChunksPerStage) == 0) buf = stream_wait(st, sm, k);
        const SwarChunk ch = swar_chunk(buf, c, st.pstart, st.pend, st.total, carry_w, lane);
        if (ch.wide) {
            // a varint of four or more bytes: the general decoder takes the page (same bail-out as delta_page_fast)
            stream_drain(st, sm, k);
            if (lane == 0) sm->seq = st.seq0 + min(st.nstages, k + static_cast<uint32_t>(kStages));
            __syncwarp();
            return 1;
        }
        const int32_t T = ch.T, Rp = ch.Rp;
        const uint32_t n = ch.n;
        uint32_t n_in = n;
#pragma unroll
        for (int sft = 1; sft < 32; sft <<= 1) {
            const uint32_t on = __shfl_up_sync(0xffffffffu, n_in, sft);
            if (lane >= sft) n_in += on;
        }
        // weight of a byte = (n - 1) - terminators before it = (count - tb - lb) - (rank + 1)
        const int64_t A1 = static_cast<int64_t>(count) - static_cast<int64_t>(tb) - static_cast<int64_t>(n_in - n);
        S += A1 * static_cast<int64_t>(T) - static_cast<int64_t>(Rp);
        tb += __shfl_sync(0xffffffffu, n_in, 31);
        if (c == nchunks - 1 && lane == 0) last_byte = buf[(st.pend - 1) % kStageBytes];
        if ((c % kChunksPerStage) == kChunksPerStage - 1 || c == nchunks - 1) stream_release(st, sm, k, lane);
    }
    {
        const uint64_t us = static_cast<uint64_t>(S);
        acc.lo += us;
        acc.hi += (S >> 63) + (acc.lo < us ? 1 : 0);
    }
    publish_acc(sm, acc, lane);
    last_byte = __shfl_sync(0xffffffffu, last_byte, 0);
    // the body must hold exactly count-1 varints and end on a terminator
    return (tb + 1 == count && last_byte < 0x80u) ? 0 : 2;
}

// ------------------------------------------------------------------------------------------------
// SWAR sum decoder under a row mask / time range: SUM / MEAN / COUNT of an EncodeTypeDelta page over the ACTIVE rows, without
// decoding a value (lane_decode.cuh: swar_masked_word).  Two passes per 2 KB chunk: (1) the lanes' terminator counts -- a lane
// must know the rows that end in it before it can cut their activity bits out of the row mask; (2) the byte-linear sums with the
// rank taken over active terminators.  Lane contribution: ((A - a_0) - active terminators before the lane + 1) * T - R'.
// One hot loop, like delta_page_sum_all.  Returns like delta_page_fast.
// ------------------------------------------------------------------------------------------------
// Pass 2 of delta_page_sum_masked over the lane's 16 words (va / vb: valid bytes 0..31 / 32..63 of a first / last chunk).
template <bool kTwoClass>
__device__ __forceinline__ void swar_masked_pass(SwarMasked &sl, const uint8_t *src, bool interior, uint32_t o, uint32_t total, uint32_t va, uint32_t vb,
                                                 uint32_t pw, unsigned long long aw) {
    swar_masked_begin(sl, pw, static_cast<uint32_t>(aw), static_cast<uint32_t>(aw >> 32));
    if (interior) {
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
            const uint4 w = *reinterpret_cast<const uint4 *>(src + 16 * q);
            swar_masked_word<false, kTwoClass>(sl, w.x, 0u);
            swar_masked_word<false, kTwoClass>(sl, w.y, 0u);
            swar_masked_word<false, kTwoClass>(sl, w.z, 0u);
            swar_masked_word<false, kTwoClass>(sl, w.w, 0u);
        }
    } else {
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
            uint4 w = make_uint4(0, 0, 0, 0);
            if (o + 16 * q < total) w = *reinterpret_cast<const uint4 *>(src + 16 * q);
            const uint32_t v = (q < 2 ? va : vb) >> (16 * (q & 1));
            swar_masked_word<true, kTwoClass>(sl, w.x, expand4(v));
            swar_masked_word<true, kTwoClass>(sl, w.y, expand4(v >> 4));
            swar_masked_word<true, kTwoClass>(sl, w.z, expand4(v >> 8));
            swar_masked_word<true, kTwoClass>(sl, w.w, expand4(v >> 12));
        }
    }
}

template <int kMode>
__device__ __noinline__ int delta_page_sum_masked(WarpSmem *sm, int lane) {
    static_assert(kMode != kRowsAll, "every row active: delta_page_sum_all");
    const uint8_t *body = sm->a_body;
    const uint32_t len = sm->a_len, count = sm->a_count, r0 = sm->a_r0, r1 = sm->a_r1;
    const int64_t first = sm->a_first;
    uint32_t A_total, a0;
    if (kMode == kRowsRange) {
        A_total = r1 - r0 + 1u;
        a0 = r0 == 0 ? 1u : 0u;
    } else {
        uint32_t c = 0;
        for (uint32_t w = lane; w < ((count + 31u) >> 5); w += 32) c += __popc(sm->mask[w]);
        A_total = __reduce_add_sync(0xffffffffu, c);
        a0 = sm->mask[0] & 1u;
    }
    AggAcc acc;
    acc.init();
    if (lane == 0) {
        acc.add_scaled(first, A_total);
        acc.cnt = A_total;
    }
    if (len == 0) {
        publish_acc(sm, acc, lane);
        return count == 1 ? 0 : 2;
    }
    PageStream st;
    stream_open(st, sm, body, len, lane);
    const uint32_t nchunks = (st.total + kSwarChunkBytes - 1) / kSwarChunkBytes;
    constexpr uint32_t kChunksPerStage = kStageBytes / kSwarChunkBytes;
    int64_t S = 0;
    uint32_t tb = 0, atb = 0, carry_w = 0, last_byte = 0;
    const uint8_t *buf = nullptr;
    for (uint32_t c = 0; c < nchunks; ++c) {
        const uint32_t k = c / kChunksPerStage;
        if ((c % kChunksPerStage) == 0) buf = stream_wait(st, sm, k);
        const uint32_t o = c * kSwarChunkBytes + lane * kSwarLaneBytes;
        const bool interior = c * kSwarChunkBytes >= st.pstart && (c + 1) * kSwarChunkBytes <= st.pend;  // warp-uniform
        const uint8_t *src = buf + (o % kStageBytes);
        int lo_i = static_cast<int>(st.pstart) - static_cast<int>(o);
        int hi_i = static_cast<int>(st.pend) - static_cast<int>(o);
        lo_i = lo_i < 0 ? 0 : (lo_i > 64 ? 64 : lo_i);
        hi_i = hi_i < 0 ? 0 : (hi_i > 64 ? 64 : hi_i);
        const uint32_t va = interior ? 0xffffffffu : (low_bits(hi_i > 32 ? 32 : hi_i) & ~low_bits(lo_i > 32 ? 32 : lo_i));
        const uint32_t vb = interior ? 0xffffffffu : (low_bits(hi_i > 32 ? hi_i - 32 : 0) & ~low_bits(lo_i > 32 ? lo_i - 32 : 0));
        // ---- pass 1: terminators of the lane -> its first row
        uint32_t n_all = 0, lastw = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint4 w = make_uint4(0, 0, 0, 0);
            if (interior || o + 16 * q < st.total) w = *reinterpret_cast<const uint4 *>(src + 16 * q);
            const uint32_t v = (q < 2 ? va : vb) >> (16 * (q & 1));
            n_all += count_terminators(w.x, expand4(v)) + count_terminators(w.y, expand4(v >> 4)) + count_terminators(w.z, expand4(v >> 8)) +
                     count_terminators(w.w, expand4(v >> 12));
            if (q == 3) lastw = w.w & expand4(v >> 12);
        }
        uint32_t n_in = n_all;
#pragma unroll
        for (int sft = 1; sft < 32; sft <<= 1) {
            const uint32_t on = __shfl_up_sync(0xffffffffu, n_in, sft);
            if (lane >= sft) n_in += on;
        }
        const uint32_t row0 = 1u + tb + n_in - n_all;
        unsigned long long aw;
        const unsigned long long nbits = n_all >= 64 ? ~0ull : ((1ull << n_all) - 1ull);
        if (kMode == kRowsRange) {
            const uint32_t a = r0 > row0 ? min(r0 - row0, 64u) : 0u;
            const uint32_t b = r1 + 1u > row0 ? min(r1 + 1u - row0, 64u) : 0u;
            const unsigned long long mb = b >= 64 ? ~0ull : ((1ull << b) - 1ull), ma = a >= 64 ? ~0ull : ((1ull << a) - 1ull);
            aw = mb & ~ma & nbits;
        } else {
            const uint32_t wi = min(row0 >> 5, static_cast<uint32_t>(kMaskWords));
            const uint32_t m0 = sm->mask[wi], m1 = sm->mask[wi + 1], m2 = sm->mask[wi + 2];
            const uint32_t sft = row0 & 31u;
            aw = (static_cast<unsigned long long>(__funnelshift_r(m1, m2, sft)) << 32 | __funnelshift_r(m0, m1, sft)) & nbits;
        }
        uint32_t pw = __shfl_up_sync(0xffffffffu, lastw, 1);
        const uint32_t cw = carry_w;
        if (lane == 0) pw = cw;
        carry_w = __shfl_sync(0xffffffffu, lastw, 31);
        // ---- pass 2: byte-linear sums, ranks over the active terminators (two-class words; the three-class ones again over a
        // chunk that holds a class-2 byte, as in swar_chunk)
        SwarMasked sl;
        swar_masked_pass<true>(sl, src, interior, o, st.total, va, vb, pw, aw);
        if (__any_sync(0xffffffffu, (sl.guard & 0x80808080u) != 0) || swar_opens_class2(cw)) {
            swar_masked_pass<false>(sl, src, interior, o, st.total, va, vb, pw, aw);
            if (__any_sync(0xffffffffu, (sl.wide & 0x80808080u) != 0)) {
                stream_drain(st, sm, k);
                if (lane == 0) sm->seq = st.seq0 + min(st.nstages, k + static_cast<uint32_t>(kStages));
                __syncwarp();
                return 1;
            }
        }
        int32_t T, Rp;
        const uint32_t na = swar_masked_end(sl, T, Rp);
        uint32_t a_in = na;
#pragma unroll
        for (int sft = 1; sft < 32; sft <<= 1) {
            const uint32_t on = __shfl_up_sync(0xffffffffu, a_in, sft);
            if (lane >= sft) a_in += on;
        }
        const int64_t A1a = static_cast<int64_t>(A_total - a0) - static_cast<int64_t>(atb) - static_cast<int64_t>(a_in - na) + 1;
        S += A1a * static_cast<int64_t>(T) - static_cast<int64_t>(Rp);
        tb += __shfl_sync(0xffffffffu, n_in, 31);
        atb += __shfl_sync(0xffffffffu, a_in, 31);
        if (c == nchunks - 1 && lane == 0) last_byte = buf[(st.pend - 1) % kStageBytes];
        if ((c % kChunksPerStage) == kChunksPerStage - 1 || c == nchunks - 1) stream_release(st, sm, k, lane);
    }
    {
        const uint64_t us = static_cast<uint64_t>(S);
        acc.lo += us;
        acc.hi += (S >> 63) + (acc.lo < us ? 1 : 0);
    }
    publish_acc(sm, acc, lane);
    last_byte = __shfl_sync(0xffffffffu, last_byte, 0);
    return (tb + 1 == count && last_byte < 0x80u) ? 0 : 2;
}

// ------------------------------------------------------------------------------------------------
// Sparse masked decode of an EncodeTypeDelta page (row predicate and / or time range, narrow deltas): the selective pass.
// With a dictionary predicate that keeps one row in eight, in runs, two thirds of the 64-byte lane windows of a field page hold
// no active row at all; the serial decoder (delta_page_fast) still walks every byte of every window because the next window's
// values depend on them.  Here every 2 KB chunk first goes through the LIGHT SWAR pass (lane_decode.cuh: swar_lite_word --
// terminator count, byte-linear delta sum, unfinished tail; no per-value work), two warp scans turn that into each window's
// first row and the value in front of it, and only windows with an active row are queued (shared memory: ring offset, base
// value, 64 active bits, the previous window's tail).  When 32 windows are queued -- or the oldest queued chunk has to leave
// the TMA ring -- every lane decodes ONE queued window value by value.  Windows wait at most one chunk: the stage of chunk
// c-1 is handed back to the ring after chunk c's light pass, so the ring needs kStages >= 2 (3 keeps a copy in flight).
// Returns like delta_page_fast.
// ------------------------------------------------------------------------------------------------
static_assert(kStageBytes == kSwarChunkBytes || kStageBytes % kSwarChunkBytes == 0, "a TMA stage holds whole chunks");

__device__ __forceinline__ unsigned long long sparse_desc(uint32_t off, uint32_t lo, uint32_t hi, uint32_t sh, uint32_t accv) {
    return static_cast<unsigned long long>(off) | (static_cast<unsigned long long>(lo) << 16) | (static_cast<unsigned long long>(hi) << 24) |
           (static_cast<unsigned long long>(sh) << 32) | (static_cast<unsigned long long>(accv) << 40);
}

template <int kNeed>
__device__ __forceinline__ void sparse_flush(WarpSmem *sm, uint32_t m, uint32_t &qn, AggAcc &acc, int lane) {
    __syncwarp();
    const bool mine = static_cast<uint32_t>(lane) < m;
    unsigned long long d = 0, aw = 0;
    long long base = 0;
    if (mine) {
        d = sm->q_desc[lane];
        aw = sm->q_aw[lane];
        base = sm->q_base[lane];
    }
    const uint32_t lo = static_cast<uint32_t>(d >> 16) & 0xffu, hi = static_cast<uint32_t>(d >> 24) & 0xffu;
    if (mine) {
        const uint8_t *src = &sm->stage[0][0] + (static_cast<uint32_t>(d) & 0xffffu);
        uint32_t accv = static_cast<uint32_t>(d >> 40) & 0x3fffu, sh = static_cast<uint32_t>(d >> 32) & 0xffu;
        int32_t P = 0, sumP = 0, minP = INT32_MAX, maxP = INT32_MIN;
        unsigned long long a = aw;
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
            const uint4 wa = *reinterpret_cast<const uint4 *>(src + 32 * h), wb = *reinterpret_cast<const uint4 *>(src + 32 * h + 16);
            const int l2 = static_cast<int>(lo) - 32 * h, h2 = static_cast<int>(hi) - 32 * h;
            const uint32_t valid = low_bits(h2 < 0 ? 0 : (h2 > 32 ? 32 : h2)) & ~low_bits(l2 < 0 ? 0 : (l2 > 32 ? 32 : l2));
            uint32_t msb = msb4(wa.x);
            msb = imad_u32(msb4(wa.y), 1u << 4, msb);
            msb = imad_u32(msb4(wa.z), 1u << 8, msb);
            msb = imad_u32(msb4(wa.w), 1u << 12, msb);
            msb = imad_u32(msb4(wb.x), 1u << 16, msb);
            msb = imad_u32(msb4(wb.y), 1u << 20, msb);
            msb = imad_u32(msb4(wb.z), 1u << 24, msb);
            msb = imad_u32(msb4(wb.w), 1u << 28, msb);
            const uint32_t term = valid & ~msb;
            const uint32_t nh = __popc(term);
            const uint32_t a32 = static_cast<uint32_t>(a) & low_bits(nh);
            // one decode variant (the masked one) for interior and edge windows alike: code size, see delta_page_sparse
            fast_lane_decode<false, kNeed>(wa, wb, valid, term, a32, accv, sh, P, sumP, minP, maxP);
            a = nh >= 32 ? (a >> 16) >> 16 : (a >> nh);
        }
        const uint32_t cntA = static_cast<uint32_t>(__popcll(aw));
        if (kNeed & kNeedSum) {
            acc.add_scaled(base, cntA);
            const int64_t sp = sumP;
            const uint64_t usp = static_cast<uint64_t>(sp);
            acc.lo += usp;
            acc.hi += (sp >> 63) + (acc.lo < usp ? 1 : 0);
        }
        if (kNeed & kNeedMinMax) {
            const int64_t vmin = base + minP, vmax = base + maxP;
            acc.mn = vmin < acc.mn ? vmin : acc.mn;
            acc.mx = vmax > acc.mx ? vmax : acc.mx;
        }
        acc.cnt += cntA;
    }
    // the rest of the queue moves to the front
    const uint32_t rest = qn - m;
    unsigned long long rd = 0, ra = 0;
    long long rb = 0;
    if (static_cast<uint32_t>(lane) < rest) {
        rd = sm->q_desc[m + lane];
        ra = sm->q_aw[m + lane];
        rb = sm->q_base[m + lane];
    }
    __syncwarp();
    if (static_cast<uint32_t>(lane) < rest) {
        sm->q_desc[lane] = rd;
        sm->q_aw[lane] = ra;
        sm->q_base[lane] = rb;
    }
    qn = rest;
    __syncwarp();
}

template <int kMode, int kNeed>
__device__ __noinline__ int delta_page_sparse(WarpSmem *sm, int lane) {
    static_assert(kMode != kRowsAll, "every row active: delta_page_sum_all / delta_page_fast");
    const uint8_t *body = sm->a_body;
    const uint32_t len = sm->a_len, count = sm->a_count, r0 = sm->a_r0, r1 = sm->a_r1;
    const int64_t first = sm->a_first;
    AggAcc acc;
    acc.init();
    if (lane == 0) {
        bool a = true;
        if (kMode == kRowsRange) a = r0 == 0;
        if (kMode == kRowsMask) a = sm->mask[0] & 1u;
        if (a) acc.add(first);
    }
    if (len == 0) {
        publish_acc(sm, acc, lane);
        return count == 1 ? 0 : 2;
    }
    PageStream st;
    stream_open(st, sm, body, len, lane);
    const uint32_t nchunks = (st.total + kSwarChunkBytes - 1) / kSwarChunkBytes;
    constexpr uint32_t kChunksPerStage = kStageBytes / kSwarChunkBytes;
    int64_t V0 = first;
    uint32_t row_base = 1, carry_w = 0, carry_acc = 0, carry_sh = 0;
    int32_t carry_pv = 0;
    uint32_t qn = 0;
    const uint8_t *buf = nullptr;
    for (uint32_t c = 0; c < nchunks; ++c) {
        const uint32_t k = c / kChunksPerStage;
        if ((c % kChunksPerStage) == 0) buf = stream_wait(st, sm, k);
        // ---- light pass over the lane's 64 bytes
        const uint32_t o = c * kSwarChunkBytes + lane * kSwarLaneBytes;
        const bool interior = c * kSwarChunkBytes >= st.pstart && (c + 1) * kSwarChunkBytes <= st.pend;  // warp-uniform
        const uint8_t *src = buf + (o % kStageBytes);
        int lo_i = static_cast<int>(st.pstart) - static_cast<int>(o);
        int hi_i = static_cast<int>(st.pend) - static_cast<int>(o);
        lo_i = lo_i < 0 ? 0 : (lo_i > 64 ? 64 : lo_i);
        hi_i = hi_i < 0 ? 0 : (hi_i > 64 ? 64 : hi_i);
        SwarLite sl;
        uint32_t lastw;
        // the word loops stay ROLLED (4 words per trip): unrolled, the two light passes and the two decode variants of one
        // instantiation are ~25 KB of hot code, and a query with two aggregated fields runs two instantiations -- ncu r02l: the
        // warps then wait for instructions 6.8 cycles per issue
        if (interior) {
            lastw = *reinterpret_cast<const uint32_t *>(src + kSwarLaneBytes - 4);
            uint32_t pw = __shfl_up_sync(0xffffffffu, lastw, 1);
            if (lane == 0) pw = carry_w;
            swar_lite_begin(sl, pw);
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {
                const uint4 w = *reinterpret_cast<const uint4 *>(src + 16 * q);
                swar_lite_word<false>(sl, w.x, 0u);
                swar_lite_word<false>(sl, w.y, 0u);
                swar_lite_word<false>(sl, w.z, 0u);
                swar_lite_word<false>(sl, w.w, 0u);
            }
        } else {
            const uint32_t va = low_bits(hi_i > 32 ? 32 : hi_i) & ~low_bits(lo_i > 32 ? 32 : lo_i);
            const uint32_t vb = low_bits(hi_i > 32 ? hi_i - 32 : 0) & ~low_bits(lo_i > 32 ? lo_i - 32 : 0);
            lastw = 0;
            if (o + 48 < st.total) lastw = *reinterpret_cast<const uint32_t *>(src + kSwarLaneBytes - 4) & expand4(vb >> 28);
            uint32_t pw = __shfl_up_sync(0xffffffffu, lastw, 1);
            if (lane == 0) pw = carry_w;
            swar_lite_begin(sl, pw);
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {
                uint4 w = make_uint4(0, 0, 0, 0);
                if (o + 16 * q < st.total) w = *reinterpret_cast<const uint4 *>(src + 16 * q);
                const uint32_t v = (q < 2 ? va : vb) >> (16 * (q & 1));
                swar_lite_word<true>(sl, w.x, expand4(v));
                swar_lite_word<true>(sl, w.y, expand4(v >> 4));
                swar_lite_word<true>(sl, w.z, expand4(v >> 8));
                swar_lite_word<true>(sl, w.w, expand4(v >> 12));
            }
        }
        carry_w = __shfl_sync(0xffffffffu, lastw, 31);
        if (__any_sync(0xffffffffu, (sl.wide & 0x80808080u) != 0)) {
            // a varint of four or more bytes: the general decoder takes the page.  Stages issued so far: the initial kStages
            // plus one per stage handed back (all stages before k - 1)
            const uint32_t kk = k > 0 ? k - 1 : 0;
            stream_drain(st, sm, kk);
            if (lane == 0) sm->seq = st.seq0 + min(st.nstages, kk + static_cast<uint32_t>(kStages));
            __syncwarp();
            return 1;
        }
        int32_t T;
        const uint32_t n = swar_lite_end(sl, T);
        uint32_t t_acc, t_sh;
        int32_t t_pv;
        swar_tail(lastw, t_acc, t_sh, t_pv);
        uint32_t in_acc = __shfl_up_sync(0xffffffffu, t_acc, 1), in_sh = __shfl_up_sync(0xffffffffu, t_sh, 1);
        int32_t in_pv = __shfl_up_sync(0xffffffffu, t_pv, 1);
        if (lane == 0) {
            in_acc = carry_acc;
            in_sh = carry_sh;
            in_pv = carry_pv;
        }
        carry_acc = __shfl_sync(0xffffffffu, t_acc, 31);
        carry_sh = __shfl_sync(0xffffffffu, t_sh, 31);
        carry_pv = __shfl_sync(0xffffffffu, t_pv, 31);
        const int32_t P = T + in_pv - t_pv;  // deltas of the values that END in this window
        uint32_t n_in = n;
        int32_t p_in = P;
#pragma unroll
        for (int sft = 1; sft < 32; sft <<= 1) {
            const uint32_t on = __shfl_up_sync(0xffffffffu, n_in, sft);
            const int32_t op = __shfl_up_sync(0xffffffffu, p_in, sft);
            if (lane >= sft) {
                n_in += on;
                p_in += op;
            }
        }
        const uint32_t row0 = row_base + n_in - n;
        unsigned long long aw;
        const unsigned long long nbits = n >= 64 ? ~0ull : ((1ull << n) - 1ull);
        if (kMode == kRowsRange) {
            const uint32_t a = r0 > row0 ? min(r0 - row0, 64u) : 0u;
            const uint32_t b = r1 + 1u > row0 ? min(r1 + 1u - row0, 64u) : 0u;
            const unsigned long long mb = b >= 64 ? ~0ull : ((1ull << b) - 1ull), ma = a >= 64 ? ~0ull : ((1ull << a) - 1ull);
            aw = mb & ~ma & nbits;
        } else {
            // a corrupt page can hold more varints than the block has rows: never index past the mask
            const uint32_t wi = min(row0 >> 5, static_cast<uint32_t>(kMaskWords));
            const uint32_t m0 = sm->mask[wi], m1 = sm->mask[wi + 1], m2 = sm->mask[wi + 2];
            const uint32_t sft = row0 & 31u;
            aw = (static_cast<unsigned long long>(__funnelshift_r(m1, m2, sft)) << 32 | __funnelshift_r(m0, m1, sft)) & nbits;
        }
        // ---- queue the windows that hold an active row
        const bool act = aw != 0;
        const uint32_t bal = __ballot_sync(0xffffffffu, act);
        const uint32_t q_old = qn;  // everything queued so far belongs to the previous chunk
        if (act) {
            const uint32_t pos = qn + __popc(bal & ((1u << lane) - 1u));
            sm->q_desc[pos] = sparse_desc(static_cast<uint32_t>(src - &sm->stage[0][0]), static_cast<uint32_t>(lo_i), static_cast<uint32_t>(hi_i), in_sh, in_acc);
            sm->q_base[pos] = V0 + static_cast<int64_t>(p_in - P);
            sm->q_aw[pos] = aw;
        }
        qn += __popc(bal);
        V0 += static_cast<int64_t>(__shfl_sync(0xffffffffu, p_in, 31));
        row_base += __shfl_sync(0xffffffffu, n_in, 31);
        const bool stage_done = (c % kChunksPerStage) == kChunksPerStage - 1 || c == nchunks - 1;
        const bool last = c == nchunks - 1;
        // ---- decode: whenever 32 windows wait, and what is left of the previous stage before that stage goes back to the ring
        uint32_t old = q_old;
        while (qn >= 32u || (stage_done && old > 0u) || (last && qn > 0u)) {
            const uint32_t m = qn < 32u ? qn : 32u;
            sparse_flush<kNeed>(sm, m, qn, acc, lane);
            old = old > m ? old - m : 0u;
        }
        if (stage_done && k > 0) stream_release(st, sm, k - 1, lane);
        if (last) stream_release(st, sm, k, lane);
    }
    publish_acc(sm, acc, lane);
    return (row_base == count && carry_sh == 0) ? 0 : 2;
}

// ------------------------------------------------------------------------------------------------
// row mask helpers (per-warp shared memory bitmask)
// ------------------------------------------------------------------------------------------------
// clears bits [a,b) ; cooperative over the warp
__device__ __forceinline__ void warp_clear_range(uint32_t *mask, uint32_t a, uint32_t b, int lane) {
    if (a >= b) return;
    const uint32_t wa = a >> 5, wb = (b - 1) >> 5;
    for (uint32_t w = wa + lane; w <= wb; w += 32) {
        uint32_t keep = 0;
        if (w == wa) keep |= (1u << (a & 31)) - 1u;
        if (w == wb && (b & 31)) keep |= ~((1u << (b & 31)) - 1u);
        atomicAnd(&mask[w], keep);
    }
}
// clears bits [a,b) ; executed by one lane (short runs)
__device__ __forceinline__ void lane_clear_range(uint32_t *mask, uint32_t a, uint32_t b) {
    if (a >= b) return;
    const uint32_t wa = a >> 5, wb = (b - 1) >> 5;
    for (uint32_t w = wa; w <= wb; ++w) {
        uint32_t keep = 0;
        if (w == wa) keep |= (1u << (a & 31)) - 1u;
        if (w == wb && (b & 31)) keep |= ~((1u << (b & 31)) - 1u);
        atomicAnd(&mask[w], keep);
    }
}

__device__ __forceinline__ uint64_t load_be64_unaligned(const uint8_t *p) {
    uint64_t u = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) u = (u << 8) | __ldg(p + k);
    return u;
}

// compressBlock header (bytes.go:291-350): type 0 = [len u8], kBlockRawLong = [len u32 LE] (a zstd frame inflated
// at part admission, unpack_kernels.cu); a type-1 frame that was not inflated surfaces as `zstd_err`.
// Leaves p at the payload and checks that `len` bytes are there.
__device__ __forceinline__ uint32_t read_cblock_header(const uint8_t *&p, const uint8_t *end, uint32_t &len, uint32_t zstd_err) {
    if (end - p < 2) return kErrCorrupt;
    const uint8_t t = __ldg(p++);
    if (t == 1) return zstd_err;
    if (t == 0) {
        len = __ldg(p++);
    } else if (t == kBlockRawLong) {
        if (end - p < 4) return kErrCorrupt;
        len = __ldg(p) | (__ldg(p + 1) << 8) | (__ldg(p + 2) << 16) | (static_cast<uint32_t>(__ldg(p + 3)) << 24);
        p += 4;
    } else {
        return kErrCorrupt;
    }
    if (static_cast<uint64_t>(end - p) < len) return kErrCorrupt;
    return kErrNone;
}

// Plain (high-cardinality) string tag page -> mask: a bytes block of `count` cells (bytes.go:45-127), cell i is
// lens[i]-1 bytes long, 0 = nil.  page points just after the 0x09 type byte.
__device__ __noinline__ uint32_t apply_plain_pred(WarpSmem *sm, const DevPred &pr, const uint8_t *page, uint32_t size, uint32_t count, int lane) {
    const uint8_t *p = page;
    const uint8_t *end = page + size;
    uint32_t llen = 0, dlen = 0;
    uint32_t berr = read_cblock_header(p, end, llen, kErrTagPlain);
    if (berr != kErrNone) return berr;
    if (llen < 1) return kErrCorrupt;
    const uint8_t wt = __ldg(p);
    if (wt > 3) return kErrCorrupt;
    const uint32_t width = 1u << wt;
    if (llen != 1 + static_cast<uint64_t>(count) * width) return kErrCorrupt;
    const uint8_t *lens = p + 1;
    p += llen;
    berr = read_cblock_header(p, end, dlen, kErrTagPlain);
    if (berr != kErrNone) return berr;
    const uint8_t *data = p;
    if (p + dlen != end) return kErrCorrupt;  // bytes.go:121-123
    uint64_t off_carry = 0;
    bool bad = false;
    for (uint32_t base = 0; base < count; base += 32) {
        const uint32_t r = base + lane;
        uint64_t L = 0;
        if (r < count)
            for (uint32_t i = 0; i < width; ++i) L = (L << 8) | __ldg(lens + static_cast<size_t>(r) * width + i);
        const bool have = L > 0;
        const uint64_t vlen = have ? L - 1 : 0;
        uint64_t incl = vlen;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const uint64_t o = shfl_up_u64(incl, s);
            if (lane >= s) incl += o;
        }
        const uint64_t off = off_carry + incl - vlen;
        off_carry += shfl_u64(incl, 31);
        bool pass = true;
        if (r < count) {
            int cmp = 0;
            if (have && off + vlen > dlen) {
                bad = true;
            } else if (have) {
                const uint32_t ml = vlen < pr.lit_len ? static_cast<uint32_t>(vlen) : pr.lit_len;
                for (uint32_t i = 0; i < ml && cmp == 0; ++i) {
                    const int a = __ldg(data + off + i), b = pr.lit[i];
                    cmp = a < b ? -1 : (a > b ? 1 : 0);
                }
                if (cmp == 0) cmp = vlen < pr.lit_len ? -1 : (vlen > pr.lit_len ? 1 : 0);
            }
            pass = cmp_op(pr.op, have, cmp);
        }
        const uint32_t keep = __ballot_sync(0xffffffffu, pass);
        if (lane == 0 && (base >> 5) < kMaskWords) sm->mask[base >> 5] &= keep;
    }
    if (__any_sync(0xffffffffu, bad) || off_carry != dlen) return kErrCorrupt;
    return kErrNone;
}

// Raw-cell numeric page (kEncRawCells, written by unpack_kernels.cu from an EncodeTypePlain fallback page):
// [0x40][has_nulls][6 pad][count x u64 LE][count x u8 valid].  Null cells are skipped (aggregation.go:292-294).
// Floats are arbitrary doubles here (not short decimals), so they are folded in double: each lane its rows in
// order, then a fixed xor tree -- deterministic, within 1e-9 relative of the reference's sequential sum.
// The float result travels in the AggAcc as bit patterns: lo = sum, mn / mx = extremes.
constexpr int kExpRawFloat = INT32_MIN;
__device__ __noinline__ uint32_t agg_raw_page(const uint8_t *page, uint32_t size, bool is_float, int mode, uint32_t count, uint32_t r0, uint32_t r1,
                                              const uint32_t *mask, AggAcc &out, int lane) {
    if (size < 8 + 9ull * count || (reinterpret_cast<uintptr_t>(page) & 7)) return kErrCorrupt;
    const bool nulls = __ldg(page + 1) != 0;
    const unsigned long long *vals = reinterpret_cast<const unsigned long long *>(page + 8);
    const uint8_t *valid = page + 8 + 8ull * count;
    AggAcc acc;
    acc.init();
    double fs = 0.0, fmn = 1.7976931348623157e308, fmx = -1.7976931348623157e308;  // function.go MIN/MAX sentinels
    const uint32_t lo = mode == kRowsMask ? 0 : r0, hi = mode == kRowsMask ? count - 1 : r1;
    for (uint32_t r = lo + lane; r <= hi && r < count; r += 32) {
        bool a = true;
        if (mode == kRowsMask) a = r < kMaskWords * 32 && ((mask[r >> 5] >> (r & 31)) & 1u);
        if (a && nulls) a = __ldg(valid + r) != 0;
        if (!a) continue;
        const unsigned long long u = __ldg(vals + r);
        if (is_float) {
            const double v = __longlong_as_double(static_cast<long long>(u));
            fs += v;
            fmn = v < fmn ? v : fmn;
            fmx = v > fmx ? v : fmx;
            acc.cnt++;
        } else {
            acc.add(static_cast<int64_t>(u));
        }
    }
    if (is_float) {
        uint32_t cnt = acc.cnt;
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            const double os = __longlong_as_double(static_cast<long long>(shfl_xor_u64(static_cast<uint64_t>(__double_as_longlong(fs)), m)));
            const double omn = __longlong_as_double(static_cast<long long>(shfl_xor_u64(static_cast<uint64_t>(__double_as_longlong(fmn)), m)));
            const double omx = __longlong_as_double(static_cast<long long>(shfl_xor_u64(static_cast<uint64_t>(__double_as_longlong(fmx)), m)));
            // lanes pair up symmetrically: add in a fixed (lower lane first) order so both partners get the same bits
            fs = (lane & m) ? os + fs : fs + os;
            fmn = omn < fmn ? omn : fmn;
            fmx = omx > fmx ? omx : fmx;
            cnt += __shfl_xor_sync(0xffffffffu, cnt, m);
        }
        acc.cnt = cnt;
        acc.lo = static_cast<uint64_t>(__double_as_longlong(fs));
        acc.mn = __double_as_longlong(fmn);
        acc.mx = __double_as_longlong(fmx);
    } else {
        acc.warp_reduce();
    }
    out = acc;
    return kErrNone;
}

// A <= 32-bit big-endian bit field at bit offset `bo` of a byte stream (writer.go:25-96): two aligned 32-bit loads
// and a funnel shift instead of eight byte loads.  Touches at most 7 bytes past the field.
__device__ __forceinline__ uint32_t read_bits_be(const uint8_t *base, uint64_t bo, uint32_t wbits, uint64_t vmask) {
    const uint8_t *p = base + (bo >> 3);
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t *w = reinterpret_cast<const uint32_t *>(a & ~static_cast<uintptr_t>(3));
    const uint32_t w0 = __byte_perm(__ldg(w), 0u, 0x0123u), w1 = __byte_perm(__ldg(w + 1), 0u, 0x0123u);  // to big endian
    const uint64_t x = (static_cast<uint64_t>(w0) << 32) | w1;
    const uint32_t off = static_cast<uint32_t>(a & 3) * 8u + static_cast<uint32_t>(bo & 7);
    return static_cast<uint32_t>((x >> (64u - off - wbits)) & vmask);
}

// Dictionary tag page -> mask (pkg/encoding/dictionary.go:69-114, bytes.go:45-127, writer.go/reader.go).
// page points just after the 0x0A type byte.  Returns a DevErr.
__device__ __noinline__ uint32_t apply_dict_pred(WarpSmem *sm, const DevPred &pr, const uint8_t *page, uint32_t size, uint32_t count, int lane) {
    const uint8_t *p = page;
    const uint8_t *end = page + size;
    uint64_t nvals;
    if (!read_varuint_seq(p, end, nvals) || nvals == 0 || nvals > 256) return kErrCorrupt;
    // lens block: compressBlock(encodeUint64List(len+1 | 0 for nil))
    uint32_t llen = 0;
    uint32_t berr = read_cblock_header(p, end, llen, kErrZstdDict);
    if (berr != kErrNone) return berr;
    if (llen < 1) return kErrCorrupt;
    const uint8_t wt = __ldg(p);
    if (wt > 3) return kErrCorrupt;
    const uint32_t width = 1u << wt;
    if (llen != 1 + nvals * width) return kErrCorrupt;
    const uint8_t *lens = p + 1;
    p += llen;
    // data block
    uint32_t dlen = 0;
    berr = read_cblock_header(p, end, dlen, kErrZstdDict);
    if (berr != kErrNone) return berr;
    const uint8_t *data = p;
    p += dlen;
    // ---- match set over the dictionary values
    uint32_t off_carry = 0;
    bool bad = false;  // lane-local; folded warp-wide before any return
    for (uint32_t base = 0; base < nvals; base += 32) {
        const uint32_t k = base + lane;
        uint32_t L = 0;
        if (k < nvals) {
            for (uint32_t i = 0; i < width; ++i) L = (L << 8) | __ldg(lens + k * width + i);
        }
        const bool have = L > 0;
        const uint32_t vlen = have ? L - 1 : 0;
        uint32_t incl = vlen;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            uint32_t o = __shfl_up_sync(0xffffffffu, incl, s);
            if (lane >= s) incl += o;
        }
        const uint32_t off = off_carry + incl - vlen;
        off_carry += __shfl_sync(0xffffffffu, incl, 31);
        bool m = false;
        if (k < nvals) {
            int cmp = 0;
            if (have && off + vlen > dlen) {
                bad = true;
            } else if (have) {
                const uint32_t ml = vlen < pr.lit_len ? vlen : pr.lit_len;
                for (uint32_t i = 0; i < ml && cmp == 0; ++i) {
                    const int a = __ldg(data + off + i), b = pr.lit[i];
                    cmp = a < b ? -1 : (a > b ? 1 : 0);
                }
                if (cmp == 0) cmp = vlen < pr.lit_len ? -1 : (vlen > pr.lit_len ? 1 : 0);
            }
            m = cmp_op(pr.op, have, cmp);
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, m);
        if (lane == 0) sm->match[base >> 5] = bal;
    }
    if (__any_sync(0xffffffffu, bad)) return kErrCorrupt;
    __syncwarp();
    // ---- bit-packed RLE pairs: [u32 BE n][u8 width][n x width bits, MSB first]
    if (end - p < 4) return kErrCorrupt;
    const uint32_t nrle = static_cast<uint32_t>(load_be64_unaligned(p) >> 32);
    p += 4;
    if (nrle == 0) return count == 0 ? kErrNone : kErrCorrupt;
    if (nrle & 1u) return kErrCorrupt;
    if (end - p < 1) return kErrCorrupt;
    const uint32_t wbits = __ldg(p++);
    if (wbits == 0 || wbits > 32) return kErrCorrupt;
    if (static_cast<uint64_t>(end - p) * 8 < static_cast<uint64_t>(nrle) * wbits) return kErrCorrupt;
    const uint8_t *bits = p;
    const uint32_t nruns = nrle >> 1;
    const uint64_t vmask = (wbits == 32) ? 0xffffffffull : ((1ull << wbits) - 1ull);
    uint32_t row_carry = 0;
    for (uint32_t base = 0; base < nruns; base += 32) {
        const uint32_t ri = base + lane;
        uint32_t value = 0, cnt = 0;
        if (ri < nruns) {
            // reads up to 7 bytes past the last needed byte: file images are padded in HBM
            const uint64_t bo = static_cast<uint64_t>(2 * ri) * wbits;
            value = read_bits_be(bits, bo, wbits, vmask);
            cnt = read_bits_be(bits, bo + wbits, wbits, vmask);
        }
        uint32_t incl = cnt;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            uint32_t o = __shfl_up_sync(0xffffffffu, incl, s);
            if (lane >= s) incl += o;
        }
        uint32_t start = row_carry + incl - cnt;
        uint32_t stop = start + cnt;
        row_carry += __shfl_sync(0xffffffffu, incl, 31);
        if (ri < nruns && value >= nvals) {
            bad = true;
            value = 0;
        }
        if (stop > count) stop = count;  // guarded; the total is verified below
        if (start > count) start = count;
        const bool clear = ri < nruns && cnt > 0 && !((sm->match[value >> 5] >> (value & 31)) & 1u);
        const bool is_long = clear && (stop - start) > 128;
        if (clear && !is_long) lane_clear_range(sm->mask, start, stop);
        uint32_t lm = __ballot_sync(0xffffffffu, is_long);
        while (lm) {
            const int src = __ffs(lm) - 1;
            lm &= lm - 1;
            warp_clear_range(sm->mask, __shfl_sync(0xffffffffu, start, src), __shfl_sync(0xffffffffu, stop, src), lane);
        }
    }
    if (__any_sync(0xffffffffu, bad) || row_carry != count) return kErrCorrupt;  // dictionary.go:108-110
    return kErrNone;
}

// Sum of (first + i*d) over the active rows of an arithmetic page (EncodeTypeConst: d = 0,
// EncodeTypeDeltaConst), int_list.go:73-96.  Lanes split the active set.
template <int kMode>
__device__ __forceinline__ void agg_arith_page(AggAcc &acc, int64_t first, int64_t d, uint32_t count, uint32_t r0, uint32_t r1,
                                               const uint32_t *mask, int lane) {
    acc.init();
    if (kMode != kRowsMask) {
        // contiguous rows [r0,r1]: lane 0 owns the closed form
        if (lane == 0) {
            const uint64_t n = static_cast<uint64_t>(r1) - r0 + 1;
            acc.cnt = static_cast<uint32_t>(n);
            acc.add_scaled(first, n);
            // sum of indices r0..r1 = n*(r0+r1)/2 (fits 64 bits: rows < 2^31)
            const uint64_t si = (n * (static_cast<uint64_t>(r0) + r1)) >> 1;
            acc.add_scaled(d, si);
            const int64_t va = first + static_cast<int64_t>(static_cast<uint64_t>(d) * r0);
            const int64_t vb = first + static_cast<int64_t>(static_cast<uint64_t>(d) * r1);
            acc.mn = va < vb ? va : vb;
            acc.mx = va < vb ? vb : va;
        }
        return;
    }
    const uint32_t nwords = (count + 31) >> 5;
    for (uint32_t w = lane; w < nwords; w += 32) {
        uint32_t m = mask[w];
        while (m) {
            const uint32_t b = __ffs(m) - 1;
            m &= m - 1;
            const uint32_t row = (w << 5) + b;
            acc.add(first + static_cast<int64_t>(static_cast<uint64_t>(d) * row));
        }
    }
}

// ------------------------------------------------------------------------------------------------
// plan_blocks: block selection
// ------------------------------------------------------------------------------------------------
__global__ void plan_blocks_kernel(const __grid_constant__ ScanParams p) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    bool sel = false;
    if (g < p.total_blocks) {
        uint32_t pi = 0;
        while (pi + 1 < p.n_parts && g >= p.parts[pi + 1].block_base) ++pi;
        const DevBlock &b = p.parts[pi].blocks[g - p.parts[pi].block_base];
        // binary search of the block's series in the query's ascending series list (query.go:601)
        uint32_t lo = 0, hi = p.n_series;
        const uint64_t sid = b.sid;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (p.q_sids[mid] < sid) lo = mid + 1;
            else hi = mid;
        }
        int32_t qi = -1;
        if (lo < p.n_series && p.q_sids[lo] == sid) qi = static_cast<int32_t>(lo);
        // part_iter.go:232-241: the block must overlap the inclusive time range
        sel = qi >= 0 && !(b.ts_max < p.tmin || b.ts_min > p.tmax);
        p.block_qsid[g] = sel ? qi : -1;
        p.Prows[g] = 0;
        // head of this series' run of blocks inside the part: lets series_reduce skip its binary search
        if (p.first_block && qi >= 0) {
            const uint32_t lb = g - p.parts[pi].block_base;
            if (lb == 0 || p.parts[pi].blocks[lb - 1].sid != sid) p.first_block[static_cast<size_t>(pi) * p.n_series + qi] = g;
        }
    }
    const uint32_t bal = __ballot_sync(0xffffffffu, sel);
    if (bal) {
        const int lane = threadIdx.x & 31;
        uint32_t base = 0;
        if (lane == __ffs(bal) - 1) base = atomicAdd(p.work_count, __popc(bal));
        base = __shfl_sync(0xffffffffu, base, __ffs(bal) - 1);
        if (sel) p.worklist[base + __popc(bal & ((1u << lane) - 1u))] = g;
    }
}

// ------------------------------------------------------------------------------------------------
// scan_blocks: one warp per block
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool find_col(const DevPartRef &part, const DevBlock &blk, uint16_t name_id, DevCol &out, int lane) {
    bool found = false;
    for (uint32_t base = 0; base < blk.n_cols; base += 32) {
        const uint32_t i = base + lane;
        DevCol c{};
        bool hit = false;
        if (i < blk.n_cols) {
            c = part.cols[blk.col_begin + i];
            hit = c.name_id == name_id;
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, hit);
        if (bal) {
            const int src = __ffs(bal) - 1;
            out.off = shfl_u64(c.off, src);
            out.size = __shfl_sync(0xffffffffu, c.size, src);
            out.name_id = name_id;
            out.value_type = static_cast<uint8_t>(__shfl_sync(0xffffffffu, static_cast<uint32_t>(c.value_type), src));
            out.file_id = static_cast<uint8_t>(__shfl_sync(0xffffffffu, static_cast<uint32_t>(c.file_id), src));
            found = true;
            break;
        }
    }
    return found;
}

// ------------------------------------------------------------------------------------------------
// Fast path for EncodeTypeDeltaOfDelta pages with narrow (<= 3 byte) second differences
// (monotone counters, series that start below zero: int_list.go:150-179).  Two light passes per
// chunk: (1) per-lane (count, sum, sum-of-prefixes) of the second differences in 32-bit registers,
// one warp scan of the triple with the composition law r = rA + rB + nB*qA gives every lane its
// (value, first difference) on entry; (2) the lane decodes again and folds the true values.
// The first varint (the first DIFFERENCE, often wide) is read sequentially up front.
// Returns like delta_page_fast.
// ------------------------------------------------------------------------------------------------
template <int kMode, int kNeed>
__device__ __noinline__ int dod_page_fast(WarpSmem *sm, int lane) {
    const uint8_t *body = sm->a_body;
    uint32_t len = sm->a_len;
    const uint32_t count = sm->a_count, r0 = sm->a_r0, r1 = sm->a_r1;
    const int64_t first = sm->a_first;
    AggAcc acc;
    acc.init();
    auto active0 = [&](uint32_t row) -> bool {
        if (kMode == kRowsRange) return row >= r0 && row <= r1;
        if (kMode == kRowsMask) return (sm->mask[row >> 5] >> (row & 31)) & 1u;
        return true;
    };
    if (count < 2) return 2;
    int64_t d1 = 0;
    uint32_t used = 0;
    if (!read_varint_seq(body, len, d1, used)) return 2;
    if (lane == 0) {
        if (active0(0)) acc.add(first);
        if (active0(1)) acc.add(first + d1);
    }
    body += used;
    len -= used;
    if (len == 0) {
        publish_acc(sm, acc, lane);
        return count == 2 ? 0 : 2;
    }
    PageStream st;
    stream_open(st, sm, body, len, lane);
    const uint32_t nchunks = (st.total + kFastChunkBytes - 1) / kFastChunkBytes;
    constexpr uint32_t kChunksPerStage = kStageBytes / kFastChunkBytes;
    int64_t V0 = first + d1;  // value of the row before this chunk's first varint
    int64_t D0 = d1;          // running first difference
    uint32_t carry_acc = 0, carry_sh = 0;
    uint32_t row_base = 2;
    const uint8_t *buf = nullptr;
    for (uint32_t c = 0; c < nchunks; ++c) {
        const uint32_t k = c / kChunksPerStage;
        if ((c % kChunksPerStage) == 0) buf = stream_wait(st, sm, k);
        FastChunk fc;
        fast_chunk_load(fc, st, buf, c, carry_sh, lane);
        if (fc.wide) {
            stream_drain(st, sm, k);
            if (lane == 0) sm->seq = st.seq0 + min(st.nstages, k + static_cast<uint32_t>(kStages));
            __syncwarp();
            return 1;
        }
        const uint32_t n = fc.n;
        // ---- pass 1: lane-local (q, r) with every value counted
        uint32_t accv = 0, sh = 0;
        int32_t P = 0, sumP = 0, mnu = 0, mxu = 0;
        const bool full = __all_sync(0xffffffffu, fc.valid == 0xffffffffu);
        if (full) fast_lane_decode<true, kNeedSum>(fc.wa, fc.wb, fc.valid, fc.term, 0xffffffffu, accv, sh, P, sumP, mnu, mxu);
        else fast_lane_decode<false, kNeedSum>(fc.wa, fc.wb, fc.valid, fc.term, 0xffffffffu, accv, sh, P, sumP, mnu, mxu);
        uint32_t prev_acc = __shfl_up_sync(0xffffffffu, accv, 1);
        uint32_t prev_sh = __shfl_up_sync(0xffffffffu, sh, 1);
        if (lane == 0) {
            prev_acc = carry_acc;
            prev_sh = carry_sh;
        }
        carry_acc = __shfl_sync(0xffffffffu, accv, 31);
        carry_sh = __shfl_sync(0xffffffffu, sh, 31);
        if (n > 0 && prev_sh != 0) {
            const int32_t dlt = head_delta(fc.wa.x, fc.term, prev_acc, prev_sh);
            P += dlt;
            sumP += dlt * static_cast<int32_t>(n);
        }
        // ---- scan of (n, q, r)
        uint32_t n_in = n;
        int64_t q_in = P, r_in = sumP;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const uint32_t on = __shfl_up_sync(0xffffffffu, n_in, s);
            const int64_t oq = static_cast<int64_t>(shfl_up_u64(static_cast<uint64_t>(q_in), s));
            const int64_t orr = static_cast<int64_t>(shfl_up_u64(static_cast<uint64_t>(r_in), s));
            if (lane >= s) {
                r_in = orr + r_in + static_cast<int64_t>(n_in) * oq;  // current lane is B: nB * qA
                q_in += oq;
                n_in += on;
            }
        }
        const uint32_t n_ex = n_in - n;
        int64_t q_ex = static_cast<int64_t>(shfl_up_u64(static_cast<uint64_t>(q_in), 1));
        int64_t r_ex = static_cast<int64_t>(shfl_up_u64(static_cast<uint64_t>(r_in), 1));
        if (lane == 0) {
            q_ex = 0;
            r_ex = 0;
        }
        // ---- pass 2: true values of this lane's rows
        uint32_t aw = fast_active_window<kMode>(sm, row_base + n_ex, n, r0, r1);
        if (__any_sync(0xffffffffu, aw != 0)) {
            int64_t D = D0 + q_ex;
            int64_t v = V0 + static_cast<int64_t>(n_ex) * D0 + r_ex;
            accv = prev_acc;
            sh = prev_sh;
            uint32_t w0 = fc.wa.x, w1 = fc.wa.y, w2 = fc.wa.z, w3 = fc.wa.w, w4 = fc.wb.x, w5 = fc.wb.y, w6 = fc.wb.z, w7 = fc.wb.w;
            uint32_t vm = fc.valid, tm = fc.term;
#pragma unroll 1
            for (int q8 = 0; q8 < 8; ++q8) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t b = (w0 >> (8 * j)) & 0xffu;
                    if ((vm >> j) & 1u) {
                        accv |= (b & 0x7fu) << sh;
                        sh += 7;
                    }
                    if ((tm >> j) & 1u) {
                        D += static_cast<int64_t>(static_cast<int32_t>(accv >> 1) ^ -static_cast<int32_t>(accv & 1u));
                        v += D;
                        if (aw & 1u) {
                            if (kNeed & kNeedSum) {
                                const uint64_t uv = static_cast<uint64_t>(v);
                                acc.lo += uv;
                                acc.hi += (v >> 63) + (acc.lo < uv ? 1 : 0);
                            }
                            if (kNeed & kNeedMinMax) {
                                acc.mn = v < acc.mn ? v : acc.mn;
                                acc.mx = v > acc.mx ? v : acc.mx;
                            }
                            acc.cnt++;
                        }
                        aw >>= 1;
                        accv = 0;
                        sh = 0;
                    }
                }
                w0 = w1;
                w1 = w2;
                w2 = w3;
                w3 = w4;
                w4 = w5;
                w5 = w6;
                w6 = w7;
                vm >>= 4;
                tm >>= 4;
            }
        }
        const uint32_t n_tot = __shfl_sync(0xffffffffu, n_in, 31);
        const int64_t q_tot = static_cast<int64_t>(shfl_u64(static_cast<uint64_t>(q_in), 31));
        const int64_t r_tot = static_cast<int64_t>(shfl_u64(static_cast<uint64_t>(r_in), 31));
        V0 += static_cast<int64_t>(n_tot) * D0 + r_tot;
        D0 += q_tot;
        row_base += n_tot;
        if ((c % kChunksPerStage) == kChunksPerStage - 1 || c == nchunks - 1) stream_release(st, sm, k, lane);
    }
    publish_acc(sm, acc, lane);
    return (row_base == count && carry_sh == 0) ? 0 : 2;
}

// ------------------------------------------------------------------------------------------------
// int64 TAG predicate on a narrow EncodeTypeDelta page, in the fast lane (BASELINE config 5: `code >= 200`).  Two passes per
// 1 KB chunk like dod_page_fast: (1) the lane's delta total with the multiply-add decoder, one warp scan -> the value in
// front of every lane; (2) the lane decodes again, compares each value with the literal and clears the mask bits of the rows
// that fail.  Arguments through the shared slots (a_body, a_len, a_count, a_first; a_r0 = operator, res_lo = literal).
// Returns like delta_page_fast (1 = a varint of 4+ bytes: the block goes to the general lane).
// ------------------------------------------------------------------------------------------------
__device__ __noinline__ int delta_pred_fast(WarpSmem *sm, int lane) {
    const uint8_t *body = sm->a_body;
    const uint32_t len = sm->a_len, count = sm->a_count;
    const int op = static_cast<int>(sm->a_r0);
    const int64_t first = sm->a_first, lit = static_cast<int64_t>(sm->res_lo);
    auto pass = [&](int64_t v) { return cmp_op(op, true, v < lit ? -1 : (v > lit ? 1 : 0)); };
    if (lane == 0 && !pass(first)) atomicAnd(&sm->mask[0], ~1u);
    if (len == 0) return count == 1 ? 0 : 2;
    PageStream st;
    stream_open(st, sm, body, len, lane);
    const uint32_t nchunks = (st.total + kFastChunkBytes - 1) / kFastChunkBytes;
    constexpr uint32_t kChunksPerStage = kStageBytes / kFastChunkBytes;
    int64_t V0 = first;
    uint32_t carry_acc = 0, carry_sh = 0;
    uint32_t row_base = 1;
    const uint8_t *buf = nullptr;
    for (uint32_t c = 0; c < nchunks; ++c) {
        const uint32_t k = c / kChunksPerStage;
        if ((c % kChunksPerStage) == 0) buf = stream_wait(st, sm, k);
        FastChunk fc;
        fast_chunk_load(fc, st, buf, c, carry_sh, lane);
        if (fc.wide) {
            stream_drain(st, sm, k);
            if (lane == 0) sm->seq = st.seq0 + min(st.nstages, k + static_cast<uint32_t>(kStages));
            __syncwarp();
            return 1;
        }
        const uint32_t n = fc.n;
        // ---- pass 1: the lane's delta total
        uint32_t accv = 0, sh = 0;
        int32_t P = 0, sumP = 0, mnu = 0, mxu = 0;
        const bool full = __all_sync(0xffffffffu, fc.valid == 0xffffffffu);
        if (full) fast_lane_decode<true, kNeedSum>(fc.wa, fc.wb, fc.valid, fc.term, 0u, accv, sh, P, sumP, mnu, mxu);
        else fast_lane_decode<false, kNeedSum>(fc.wa, fc.wb, fc.valid, fc.term, 0u, accv, sh, P, sumP, mnu, mxu);
        uint32_t prev_acc = __shfl_up_sync(0xffffffffu, accv, 1);
        uint32_t prev_sh = __shfl_up_sync(0xffffffffu, sh, 1);
        if (lane == 0) {
            prev_acc = carry_acc;
            prev_sh = carry_sh;
        }
        carry_acc = __shfl_sync(0xffffffffu, accv, 31);
        carry_sh = __shfl_sync(0xffffffffu, sh, 31);
        if (n > 0 && prev_sh != 0) P += head_delta(fc.wa.x, fc.term, prev_acc, prev_sh);
        uint32_t n_in = n;
        int32_t s_in = P;
#pragma unroll
        for (int sft = 1; sft < 32; sft <<= 1) {
            const uint32_t on = __shfl_up_sync(0xffffffffu, n_in, sft);
            const int32_t os = __shfl_up_sync(0xffffffffu, s_in, sft);
            if (lane >= sft) {
                n_in += on;
                s_in += os;
            }
        }
        // ---- pass 2: true values of the lane's rows against the literal
        int64_t v = V0 + static_cast<int64_t>(s_in - P);
        uint32_t fail = 0, bit = 1;
        accv = prev_acc;
        sh = prev_sh;
        uint32_t w0 = fc.wa.x, w1 = fc.wa.y, w2 = fc.wa.z, w3 = fc.wa.w, w4 = fc.wb.x, w5 = fc.wb.y, w6 = fc.wb.z, w7 = fc.wb.w;
        uint32_t vm = fc.valid, tm = fc.term;
#pragma unroll 1
        for (int q8 = 0; q8 < 8; ++q8) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t b = (w0 >> (8 * j)) & 0xffu;
                if ((vm >> j) & 1u) {
                    accv |= (b & 0x7fu) << sh;
                    sh += 7;
                }
                if ((tm >> j) & 1u) {
                    v += static_cast<int64_t>(static_cast<int32_t>(accv >> 1) ^ -static_cast<int32_t>(accv & 1u));
                    if (!pass(v)) fail |= bit;
                    bit <<= 1;
                    accv = 0;
                    sh = 0;
                }
            }
            w0 = w1;
            w1 = w2;
            w2 = w3;
            w3 = w4;
            w4 = w5;
            w5 = w6;
            w6 = w7;
            vm >>= 4;
            tm >>= 4;
        }
        // rows row0 .. row0+n-1 of this lane: clear the failing ones (a corrupt page may hold more varints than rows)
        const uint32_t row0 = row_base + n_in - n;
        if (fail && row0 < kMaskWords * 32) {
            const uint32_t w = row0 >> 5, shb = row0 & 31;
            atomicAnd(&sm->mask[w], ~(fail << shb));
            if (shb && w + 1 < kMaskWords) atomicAnd(&sm->mask[w + 1], ~(fail >> (32 - shb)));
        }
        V0 += static_cast<int64_t>(__shfl_sync(0xffffffffu, s_in, 31));
        row_base += __shfl_sync(0xffffffffu, n_in, 31);
        if ((c % kChunksPerStage) == kChunksPerStage - 1 || c == nchunks - 1) stream_release(st, sm, k, lane);
    }
    __syncwarp();
    return (row_base == count && carry_sh == 0) ? 0 : 2;
}

// kDeferSlow is returned by the fast lane when a page needs the general decoder
constexpr uint32_t kDeferSlow = 0xffffffffu;

template <int kMode>
__device__ __forceinline__ int masked_sum_dispatch(WarpSmem *sm, int lane) {
    if constexpr (kMode == kRowsAll) return 2;  // not reached
    else return delta_page_sum_masked<kMode>(sm, lane);
}

template <int kMode>
__device__ __forceinline__ int sparse_dispatch(WarpSmem *sm, uint32_t need, int lane) {
    if constexpr (kMode == kRowsAll) {
        return 2;  // not reached: every-row pages take delta_page_sum_all / delta_page_fast
    } else {
        if (need == kNeedSum) return delta_page_sparse<kMode, kNeedSum>(sm, lane);
        if (need == kNeedMinMax) return delta_page_sparse<kMode, kNeedMinMax>(sm, lane);
        return delta_page_sparse<kMode, kNeedSum | kNeedMinMax>(sm, lane);
    }
}

template <int kMode, bool kFastLane>
// Out of line (one copy per row mode), arguments and result through the warp's shared-memory slots: the block loop of the
// scan kernel then keeps only its own few values live across the call instead of spilling around an inlined decoder.
// In: a_page, a_size, a_flags, a_count, a_r0, a_r1.  Out: res_* (warp-reduced accumulator), res_exp.
__device__ __noinline__ uint32_t agg_field_page(WarpSmem *sm, int lane) {
    const uint8_t *page = sm->a_page;
    const uint32_t size = sm->a_size, count = sm->a_count, r0 = sm->a_r0, r1 = sm->a_r1;
    const bool is_float = (sm->a_flags & 1u) != 0;
    const uint32_t need = sm->a_flags >> 1;
    int exp_out = 0;
    AggAcc out;
    if (size < 1) return kErrCorrupt;
    const uint32_t enc = __ldg(page);
    if (enc == kEncRawCells) {
        if (kFastLane) return kDeferSlow;  // keeps the fast lane's register budget for the varint decoders
        const uint32_t e = agg_raw_page(page, size, is_float, kMode, count, r0, r1, sm->mask, out, lane);
        store_acc(sm, out, lane);
        if (lane == 0) sm->res_exp = is_float ? kExpRawFloat : 0;
        __syncwarp();
        return e;
    }
    if (enc == 9) return kErrPlainPage;  // EncodeTypePlain fallback page that was not unpacked at admission
    const uint32_t hdr = is_float ? 11u : 9u;
    if (size < hdr) return kErrCorrupt;
    if (is_float) exp_out = static_cast<int16_t>((static_cast<uint32_t>(__ldg(page + 1)) << 8) | __ldg(page + 2));
    if (lane == 0) sm->res_exp = exp_out;
    const int64_t first = conv_bytes_to_int64(page + hdr - 8);
    const uint8_t *body = page + hdr;
    const uint32_t blen = size - hdr;
    if (enc == 1 || enc == 2) {
        int64_t d = 0;
        if (enc == 1) {
            if (blen != 0) return kErrCorrupt;
        } else {
            uint32_t used = 0;
            if (!read_varint_seq(body, blen, d, used) || used != blen) return kErrCorrupt;
        }
        agg_arith_page<kMode>(out, first, d, count, r0, r1, sm->mask, lane);
        publish_acc(sm, out, lane);
        return kErrNone;
    }
    if (enc != 3 && enc != 4) return kErrBadEnc;
    {
        int rc;  // warp-uniform: every exit of the fast decoders is taken by the whole warp
        __syncwarp();
        if (lane == 0) {
            sm->a_body = body;
            sm->a_len = blen;
            sm->a_count = count;
            sm->a_first = first;
            sm->a_r0 = r0;
            sm->a_r1 = r1;
        }
        __syncwarp();
        if (enc == 3) {
            if (need == kNeedSum && kMode == kRowsAll) rc = delta_page_sum_all(sm, lane);
            else if (need == kNeedSum && kMode != kRowsAll && kFastLane && BYDB_MASKED_SWAR) rc = masked_sum_dispatch<kMode>(sm, lane);
            else if (kMode != kRowsAll && kFastLane && BYDB_SPARSE) rc = sparse_dispatch<kMode>(sm, need, lane);
            else if (need == kNeedSum) rc = delta_page_fast<kMode, kNeedSum>(sm, lane);
            else if (need == kNeedMinMax) rc = delta_page_fast<kMode, kNeedMinMax>(sm, lane);
            else rc = delta_page_fast<kMode, kNeedSum | kNeedMinMax>(sm, lane);
        } else {
            rc = dod_page_fast<kMode, kNeedSum | kNeedMinMax>(sm, lane);
        }
        if (rc == 0) return kErrNone;  // the decoder left the result in the slot
        if (rc == 2) return kErrCorrupt;
        // rc == 1: a varint longer than 3 bytes -> general two-pass decoder
    }
    if (kFastLane) {
        return kDeferSlow;
    } else {
        AggCons cons;
        cons.acc.init();
        cons.r0 = r0;
        cons.r1 = r1;
        cons.mask = sm->mask;
        cons.mode = kMode;
        bool ok;
        if (enc == 3) ok = decode_varint_page<false>(sm, body, blen, count, first, cons, lane);
        else ok = decode_varint_page<true>(sm, body, blen, count, first, cons, lane);
        ok = __all_sync(0xffffffffu, ok);
        if (!ok) return kErrCorrupt;
        publish_acc(sm, cons.acc, lane);
        return kErrNone;
    }
}

// Guided self-scheduling of the persistent warps: a warp takes up to `most` work items per cursor increment (one atomic
// round trip for several blocks) while plenty of work is left, and single items towards the end, so short work lists -- a
// slice of the cold path, one rank's shard of a strong-scaled query -- still spread over every warp.
__device__ __forceinline__ uint32_t grab_work(uint32_t *cursor, uint32_t nwork, uint32_t most, uint32_t &count, int lane) {
    uint32_t base = 0, want = 1;
    if (lane == 0) {
        const uint32_t seen = *reinterpret_cast<volatile uint32_t *>(cursor);
        const uint32_t left = seen < nwork ? nwork - seen : 0u;
        const uint32_t warps = gridDim.x * (blockDim.x >> 5);
        want = left / (2u * warps);
        want = want < 1u ? 1u : (want > most ? most : want);
        base = atomicAdd(cursor, want);
    }
    base = __shfl_sync(0xffffffffu, base, 0);
    want = __shfl_sync(0xffffffffu, want, 0);
    count = base < nwork ? min(want, nwork - base) : 0u;
    return base;
}

// The value type of aggregated field c must be the same in every block of the query (kErrTypeMix otherwise).  One global word
// per field records it; `known` caches what this thread has already seen (4 bits per field), so the common case costs no
// memory access at all -- a compare-and-swap per block on one hot address used to be a fifth of the kernel's stall samples
// once the page decode got cheap (ncu r02b).  Returns false on a mismatch.
__device__ __forceinline__ bool check_col_type(const ScanParams &p, uint32_t c, uint8_t vt, uint32_t &known) {
    const uint32_t have = (known >> (4 * c)) & 0xfu;
    if (have == vt) return true;
    if (have != 0) return false;
    int32_t old = __ldcg(&p.col_type[c]);
    if (old == 0) old = atomicCAS(&p.col_type[c], 0, static_cast<int32_t>(vt));
    if (old != 0 && old != static_cast<int32_t>(vt)) return false;
    known |= static_cast<uint32_t>(vt) << (4 * c);
    return true;
}

template <bool kFastLane>
__global__ void __launch_bounds__(kWarpsPerCta * 32, kFastLane ? BYDB_FAST_CTAS : 2) scan_blocks_kernel(const __grid_constant__ ScanParams p) {
    // fast lane: the planned work list, or what the express lane left over; slow lane: the blocks the fast lane deferred
    const bool after_express = kFastLane && p.rest_list != nullptr;
    const uint32_t nwork = kFastLane ? (after_express ? *p.rest_count : *p.work_count) : *p.slow_count;
    if (nwork == 0) return;  // the usual case of the lanes behind the express / fast lane: nothing left over (whole grid, uniform)
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    WarpSmem *sm = reinterpret_cast<WarpSmem *>(smem_raw) + warp;
    if (lane == 0) {
        sm->fault = 0;
        sm->seq = 0;
        sm->st_rows = sm->st_matched = sm->st_bytes = 0;
        sm->st_blocks = sm->st_deferred = sm->st_why = 0;
        for (int s = 0; s < kStages; ++s) mbar_init(&sm->bar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint32_t *list = kFastLane ? (after_express ? p.rest_list : p.worklist) : p.slow_list;
    uint32_t *cursor = kFastLane ? (after_express ? p.rest_next : p.work_next) : p.slow_next;
    // per-warp statistics, flushed once at the end: four atomics per block on four hot words serialise in the L2
    uint32_t known_types = 0;
    constexpr uint32_t kGrab = 4;  // blocks per cursor increment: the atomic's round trip is paid once per kGrab blocks
    uint32_t wi_next = 0, wi_end = 0;
    for (;;) {
        if (wi_next == wi_end) {
            uint32_t got = 0;
            wi_next = grab_work(cursor, nwork, kGrab, got, lane);
            if (got == 0) break;
            wi_end = wi_next + got;
        }
        const uint32_t wi = wi_next++;
        const uint32_t g = list[wi];
        bool defer = false;
        uint32_t defer_why = 0;
        uint32_t pi = 0;
        while (pi + 1 < p.n_parts && g >= p.parts[pi + 1].block_base) ++pi;
        const DevPartRef &part = p.parts[pi];
        const DevBlock blk = part.blocks[g - part.block_base];
        const uint32_t count = blk.count;
        uint32_t page_bytes = 0;
        uint32_t err = kErrNone;

        // ---- 1. time range -> rows [r0,r1] (block.go:825-829, range.go:143-169)
        uint32_t r0 = 0, r1 = count - 1;
        bool empty = false;
        if (p.tmin > blk.ts_min || p.tmax < blk.ts_max) {
            const uint8_t *tsp = part.files[0] + blk.ts_off;
            if (blk.ts_enc == 1) {
                // all timestamps equal ts_min, which plan_blocks already proved inside the range
            } else if (blk.ts_enc == 2) {
                int64_t d = 0;
                uint32_t used = 0;
                if (!read_varint_seq(tsp, blk.ver_off, d, used) || used != blk.ver_off || d <= 0) {
                    err = kErrCorrupt;
                } else {
                    const uint64_t ud = static_cast<uint64_t>(d);
                    if (p.tmin > blk.ts_min) {
                        const uint64_t diff = static_cast<uint64_t>(p.tmin) - static_cast<uint64_t>(blk.ts_min);
                        const uint64_t q = (diff + ud - 1) / ud;
                        r0 = q > count ? count : static_cast<uint32_t>(q);
                    }
                    if (p.tmax < blk.ts_max) {
                        const uint64_t diff = static_cast<uint64_t>(p.tmax) - static_cast<uint64_t>(blk.ts_min);
                        const uint64_t q = diff / ud;
                        r1 = q >= count ? count - 1 : static_cast<uint32_t>(q);
                    }
                    empty = r0 > r1;
                }
                page_bytes += blk.ver_off;
            } else if (kFastLane) {
                defer = true;  // irregular timestamps need the general decoder
                defer_why |= 1u;
            } else {
                TsCons tc;
                tc.tmin = p.tmin;
                tc.tmax = p.tmax;
                tc.lt = 0;
                tc.le = 0;
                bool ok;
                if (blk.ts_enc == 3) ok = decode_varint_page<false>(sm, tsp, blk.ver_off, count, blk.ts_min, tc, lane);
                else ok = decode_varint_page<true>(sm, tsp, blk.ver_off, count, blk.ts_min, tc, lane);
                if (!__all_sync(0xffffffffu, ok)) err = kErrCorrupt;
                uint32_t lt = tc.lt, le = tc.le;
#pragma unroll
                for (int m = 16; m >= 1; m >>= 1) {
                    lt += __shfl_xor_sync(0xffffffffu, lt, m);
                    le += __shfl_xor_sync(0xffffffffu, le, m);
                }
                r0 = lt;
                if (le == 0 || lt >= le) empty = true;
                else r1 = le - 1;
                page_bytes += blk.ver_off;
            }
        }

        // ---- 2. tag predicates -> row bitmask
        uint32_t rows = empty ? 0 : (r1 - r0 + 1);
        uint32_t first_row = r0;
        const int32_t ddi = p.dd_index ? p.dd_index[g] : -1;
        const bool use_mask = p.n_preds > 0 || ddi >= 0;
        if (use_mask && !empty && err == kErrNone && !defer) {
            if (count > kMaskWords * 32) {
                err = kErrBigBlock;
            } else {
                const uint32_t nwords = (count + 31) >> 5;
                const uint32_t *shadow = ddi >= 0 ? p.dd_shadow + static_cast<size_t>(ddi) * kMaskWords : nullptr;
                for (uint32_t w = lane; w < kMaskWords; w += 32) {
                    uint32_t v = 0;
                    if (w < nwords) v = (w == nwords - 1 && (count & 31)) ? ((1u << (count & 31)) - 1u) : 0xffffffffu;
                    if (shadow && w < nwords) v &= shadow[w];
                    sm->mask[w] = v;
                }
                __syncwarp();
                for (uint32_t pi2 = 0; pi2 < p.n_preds && err == kErrNone && !defer; ++pi2) {
                    const DevPred &pr = p.preds[pi2];
                    DevCol col;
                    if (!find_col(part, blk, pr.name_id, col, lane)) {
                        // column absent in this block: every cell is nil (block.go:226-233)
                        if (!cmp_op(pr.op, false, 0)) warp_clear_range(sm->mask, 0, count, lane);
                        __syncwarp();
                        continue;
                    }
                    const uint8_t *page = part.files[col.file_id] + col.off;
                    page_bytes += col.size;
                    if (col.size < 1) {
                        err = kErrCorrupt;
                        break;
                    }
                    const uint32_t enc = __ldg(page);
                    if (pr.value_type == BYDB_VT_INT64) {
                        if (col.value_type != BYDB_VT_INT64) {
                            err = kErrPredType;
                        } else if (enc == kEncRawCells && kFastLane) {
                            defer = true;
                            defer_why |= 2u;
                        } else if (enc == kEncRawCells) {
                            if (col.size < 8 + 9ull * count || (reinterpret_cast<uintptr_t>(page) & 7)) {
                                err = kErrCorrupt;
                            } else {
                                const bool nulls = __ldg(page + 1) != 0;
                                const long long *vals = reinterpret_cast<const long long *>(page + 8);
                                const uint8_t *valid = page + 8 + 8ull * count;
                                for (uint32_t row = lane; row < count; row += 32) {
                                    const bool have = !nulls || __ldg(valid + row) != 0;
                                    const int64_t v = __ldg(vals + row);
                                    const int c = v < pr.lit_i64 ? -1 : (v > pr.lit_i64 ? 1 : 0);
                                    if (!cmp_op(pr.op, have, c)) atomicAnd(&sm->mask[row >> 5], ~(1u << (row & 31)));
                                }
                            }
                        } else if (enc == 9) {
                            err = kErrPlainPage;
                        } else if (col.size < 9) {
                            err = kErrCorrupt;
                        } else {
                            const int64_t first = conv_bytes_to_int64(page + 1);
                            const uint8_t *body = page + 9;
                            const uint32_t blen = col.size - 9;
                            if (enc == 1 || enc == 2) {
                                int64_t d = 0;
                                uint32_t used = 0;
                                if (enc == 2 && (!read_varint_seq(body, blen, d, used) || used != blen)) err = kErrCorrupt;
                                if (enc == 1 && blen != 0) err = kErrCorrupt;
                                if (err == kErrNone) {
                                    for (uint32_t row = lane; row < count; row += 32) {
                                        const int64_t v = first + static_cast<int64_t>(static_cast<uint64_t>(d) * row);
                                        const int c = v < pr.lit_i64 ? -1 : (v > pr.lit_i64 ? 1 : 0);
                                        if (!cmp_op(pr.op, true, c)) atomicAnd(&sm->mask[row >> 5], ~(1u << (row & 31)));
                                    }
                                }
                            } else if (enc == 3 && kFastLane) {
                                // narrow delta page: compared in the fast lane; anything wider goes to the general lane
                                __syncwarp();
                                if (lane == 0) {
                                    sm->a_body = body;
                                    sm->a_len = blen;
                                    sm->a_count = count;
                                    sm->a_first = first;
                                    sm->a_r0 = pr.op;
                                    sm->res_lo = static_cast<unsigned long long>(pr.lit_i64);
                                }
                                __syncwarp();
                                const int rc = delta_pred_fast(sm, lane);
                                if (rc == 2) err = kErrCorrupt;
                                if (rc == 1) {
                                    defer = true;
                                    defer_why |= 2u;
                                }
                            } else if (enc == 4 && kFastLane) {
                                defer = true;
                                defer_why |= 2u;
                            } else if (enc == 3 || enc == 4) {
                                CmpCons cc;
                                cc.lit = pr.lit_i64;
                                cc.op = pr.op;
                                cc.mask = sm->mask;
                                cc.limit = count;
                                bool ok;
                                if (enc == 3) ok = decode_varint_page<false>(sm, body, blen, count, first, cc, lane);
                                else ok = decode_varint_page<true>(sm, body, blen, count, first, cc, lane);
                                if (!__all_sync(0xffffffffu, ok)) err = kErrCorrupt;
                            } else {
                                err = kErrBadEnc;
                            }
                        }
                    } else {
                        if (col.value_type != BYDB_VT_STR && col.value_type != BYDB_VT_BINARY) err = kErrPredType;
                        else if (enc == 9 && kFastLane) defer = true, defer_why |= 2u;
                        else if (enc == 9) err = apply_plain_pred(sm, pr, page + 1, col.size - 1, count, lane);
                        else if (enc != 10) err = kErrBadEnc;
                        else err = apply_dict_pred(sm, pr, page + 1, col.size - 1, count, lane);
                        err = __reduce_max_sync(0xffffffffu, err);
                    }
                    __syncwarp();
                }
                // fold the time range into the mask, then count the surviving rows
                if (err == kErrNone && !defer) {
                    warp_clear_range(sm->mask, 0, r0, lane);
                    warp_clear_range(sm->mask, r1 + 1, count, lane);
                    __syncwarp();
                    uint32_t c = 0;
                    for (uint32_t w = lane; w < nwords; w += 32) c += __popc(sm->mask[w]);
#pragma unroll
                    for (int m = 16; m >= 1; m >>= 1) c += __shfl_xor_sync(0xffffffffu, c, m);
                    rows = c;
                    if (p.Pfirst) {  // group-key passes: where the key value first shows in this block
                        uint32_t f = 0xffffffffu;
                        for (uint32_t w = lane; w < nwords && f == 0xffffffffu; w += 32) {
                            const uint32_t m = sm->mask[w];
                            if (m) f = w * 32u + static_cast<uint32_t>(__ffs(m)) - 1u;
                        }
                        first_row = __reduce_min_sync(0xffffffffu, f);
                    }
                }
            }
        }

        // ---- 3. field pages -> per-block partial aggregates
        for (uint32_t c = 0; c < p.n_fcols; ++c) {
            BlockPartial bp;
            bp.sum.i = 0;
            bp.mn.i = 0;
            bp.mx.i = 0;
            bp.cnt = 0;
            DevCol col;
            if (err == kErrNone && !defer && rows > 0 && find_col(part, blk, p.fcol_name[c], col, lane)) {
                const bool is_float = col.value_type == BYDB_VT_FLOAT64;
                if (!is_float && col.value_type != BYDB_VT_INT64) {
                    err = kErrTypeMix;
                } else {
                    if (!check_col_type(p, c, col.value_type, known_types)) err = kErrTypeMix;  // warp-uniform: every lane keeps the cache
                    const uint8_t *page = part.files[col.file_id] + col.off;
                    AggAcc acc;
                    acc.init();
                    int exp = 0;
                    uint32_t e2 = kErrNone;
                    const uint32_t need = p.fcol_need[c];
                    if (need == 0) {
                        // COUNT only: numeric pages hold no nulls (a null forces the Plain fallback page), so the
                        // count is the number of surviving rows and the page body is never read
                        acc.cnt = rows;
                        page_bytes += 1;
                        if (col.size < 2) {
                            e2 = kErrCorrupt;
                        } else if (__ldg(page) == 9) {
                            e2 = kErrPlainPage;
                        } else if (__ldg(page) == kEncRawCells && __ldg(page + 1)) {
                            // a page with null cells: COUNT skips them (aggregation.go:292-294)
                            if (kFastLane) {  // compile-time: the fast lane never instantiates the raw-cell reader
                                e2 = kDeferSlow;
                            } else {
                                const int mode = use_mask ? kRowsMask : kRowsRange;
                                e2 = agg_raw_page(page, col.size, false, mode, count, r0, r1, sm->mask, acc, lane);
                                acc.lo = 0;
                                acc.hi = 0;
                                page_bytes += count;
                            }
                        }
                    } else {
                        page_bytes += col.size;
                        __syncwarp();
                        if (lane == 0) {
                            sm->a_page = page;
                            sm->a_size = col.size;
                            sm->a_flags = (is_float ? 1u : 0u) | (need << 1);
                            sm->a_count = count;
                            sm->a_r0 = r0;
                            sm->a_r1 = r1;
                        }
                        __syncwarp();
                        if (use_mask) e2 = agg_field_page<kRowsMask, kFastLane>(sm, lane);
                        else if (r0 == 0 && r1 == count - 1) e2 = agg_field_page<kRowsAll, kFastLane>(sm, lane);
                        else e2 = agg_field_page<kRowsRange, kFastLane>(sm, lane);
                        if (e2 == kErrNone) {
                            fetch_acc(sm, acc);
                            exp = sm->res_exp;
                        }
                    }
                    if (e2 == kDeferSlow) {
                        defer = true;
                        defer_why |= 4u << c;
                        e2 = kErrNone;
                    }
                    if (err == kErrNone) err = e2;
                    if (err == kErrNone && !defer && acc.cnt > 0) {
                        bp.cnt = acc.cnt;
                        if (is_float && exp == kExpRawFloat) {
                            bp.sum.f = __longlong_as_double(static_cast<long long>(acc.lo));
                            bp.mn.f = __longlong_as_double(acc.mn);
                            bp.mx.f = __longlong_as_double(acc.mx);
                        } else if (is_float) {
                            // block sum in the exact decimal-integer domain, converted once
                            double s;
                            if (acc.hi == (static_cast<int64_t>(acc.lo) >> 63)) s = __ll2double_rn(static_cast<int64_t>(acc.lo));
                            else s = __ll2double_rn(acc.hi) * 18446744073709551616.0 + __ull2double_rn(acc.lo);
                            bp.sum.f = scale_decimal(s, exp);
                            // min/max: int -> float64 conversion and the scaling are monotone, so
                            // converting the integer extreme gives the bit-exact float extreme
                            bp.mn.f = scale_decimal(__ll2double_rn(acc.mn), exp);
                            bp.mx.f = scale_decimal(__ll2double_rn(acc.mx), exp);
                        } else {
                            bp.sum.i = static_cast<int64_t>(acc.lo);  // wraps mod 2^64 like Go's int64 sum
                            bp.mn.i = acc.mn;
                            bp.mx.i = acc.mx;
                        }
                    }
                }
            }
            if (lane == 0 && !defer) p.P[static_cast<size_t>(g) * p.n_fcols + c] = bp;
        }
        if (sm->fault) err = kErrTmaTimeout;
        if (kFastLane && defer && err == kErrNone) {
            // hand the whole block to the slow lane (launched right after this kernel)
            if (lane == 0) {
                p.slow_list[atomicAdd(p.slow_count, 1u)] = g;
                sm->st_deferred += 1;
                sm->st_why |= defer_why;
            }
            continue;
        }
        if (err != kErrNone) {
            set_err(p, err, g, lane);
            rows = 0;
        }
        if (lane == 0) {
            p.Prows[g] = rows;
            if (p.Pfirst) p.Pfirst[g] = first_row;
            sm->st_rows += count;
            sm->st_matched += rows;
            sm->st_bytes += page_bytes;
            sm->st_blocks += 1;
        }
    }
    if (lane == 0) {
        if (sm->st_blocks) {
            atomicAdd(&p.stats[0], sm->st_rows);
            atomicAdd(&p.stats[1], sm->st_matched);
            atomicAdd(&p.stats[2], sm->st_bytes);
            atomicAdd(&p.stats[3], static_cast<unsigned long long>(sm->st_blocks));
        }
        if (sm->st_deferred) {
            atomicAdd(&p.stats[4], static_cast<unsigned long long>(sm->st_deferred));
            atomicOr(&p.stats[5], static_cast<unsigned long long>(sm->st_why));
        }
    }
}


// ------------------------------------------------------------------------------------------------
// Express lane: the all-rows SUM / MEAN / COUNT scan (BASELINE configs 3/4: group-by sum, no row predicate) without the
// per-block latency chain.  With the SWAR decoder a 16 KB page costs ~5 k warp instructions, so the dependent loads in front
// of every page (work cursor -> work list -> DevBlock -> DevCol -> page header -> first TMA stage) weighed as much as the
// decode (ncu r02b: issue slots 46 % busy, long-scoreboard stalls 8 per issue).  Here a warp takes kExpressBatch blocks per
// cursor increment; lane l resolves block l (directory entry, column lookup, page header) -- eight dependent chains overlap in
// the lanes of one warp -- and then the warp streams the batch's pages through ONE continuous TMA ring: the first stages of
// page k+1 are in flight while page k is being decoded.  Blocks that are not plain (cut by the time range, a page that is not
// a narrow EncodeTypeDelta page, nulls, type mix ...) are handed to the regular fast lane through `rest_list`; the express
// lane never reports an error itself.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kExpressBatch = 8;

__device__ __forceinline__ const uint8_t *ring_wait(WarpSmem *sm, uint32_t n) {
    const uint32_t slot = n % kStages;
    const uint32_t parity = (n / kStages) & 1u;
    for (uint32_t spins = 0; !mbar_try_wait(&sm->bar[slot], parity); ++spins) {
        if (spins > (1u << 24)) {
            sm->fault = 1;
            break;
        }
    }
    return sm->stage[slot];
}

__global__ void __launch_bounds__(kWarpsPerCta * 32, BYDB_FAST_CTAS) scan_sum_express_kernel(const __grid_constant__ ScanParams p) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    WarpSmem *sm = reinterpret_cast<WarpSmem *>(smem_raw) + warp;
    if (lane == 0) {
        sm->fault = 0;
        sm->seq = 0;
        sm->st_rows = sm->st_matched = sm->st_bytes = 0;
        sm->st_blocks = sm->st_deferred = sm->st_why = 0;
        for (int s = 0; s < kStages; ++s) mbar_init(&sm->bar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint32_t nwork = *p.work_count;
    constexpr uint32_t kChunksPerStage = kStageBytes / kSwarChunkBytes;
    uint32_t seq = 0;  // stages issued so far by this warp (mbarrier phase bookkeeping; the kernel owns the ring from start to end)
    unsigned long long st_rows = 0, st_bytes = 0;  // per-warp statistics, flushed once at the end
    uint32_t st_blocks = 0, known_types = 0;
    for (;;) {
        uint32_t nb = 0;
        const uint32_t base = grab_work(p.work_next, nwork, kExpressBatch, nb, lane);
        if (nb == 0) break;
        // ---- resolve: lane l < nb owns block l of the batch
        const bool mine = static_cast<uint32_t>(lane) < nb;
        uint32_t g = 0, count = 0, col_begin = 0, n_cols = 0, pi = 0;
        bool ok = mine;
        if (mine) {
            g = p.worklist[base + lane];
            while (pi + 1 < p.n_parts && g >= p.parts[pi + 1].block_base) ++pi;
            const DevBlock *b = p.parts[pi].blocks + (g - p.parts[pi].block_base);
            count = b->count;
            col_begin = b->col_begin;
            n_cols = b->n_cols;
            ok = p.tmin <= b->ts_min && p.tmax >= b->ts_max && count >= 1;  // every row of the block is active
        }
        uint32_t page_bytes = 0;
        for (uint32_t c = 0; c < p.n_fcols; ++c) {
            // ---- this lane's page of field c
            const uint8_t *abase = nullptr;
            uint32_t pstart = 0, pend = 0, total = 0, nst = 0;
            int64_t first = 0;
            int exp = 0;
            bool has_page = false, is_float = false, count_only = false;
            if (ok) {
                const DevCol *cols = p.parts[pi].cols + col_begin;
                DevCol col{};
                bool found = false;
                for (uint32_t i = 0; i < n_cols && !found; ++i) {
                    const DevCol cc = cols[i];
                    if (cc.name_id == p.fcol_name[c]) {
                        col = cc;
                        found = true;
                    }
                }
                if (found) {
                    is_float = col.value_type == BYDB_VT_FLOAT64;
                    if (!is_float && col.value_type != BYDB_VT_INT64) {
                        ok = false;
                    } else if (!check_col_type(p, c, col.value_type, known_types)) {
                        ok = false;  // the regular lane reports the type mix
                    }
                    const uint8_t *page = p.parts[pi].files[col.file_id] + col.off;
                    const uint32_t hdr = is_float ? 11u : 9u;
                    if (ok && p.fcol_need[c] == 0) {
                        // COUNT only: numeric pages hold no nulls unless they are fallback pages
                        if (col.size < 2 || __ldg(page) == 9 || (__ldg(page) == kEncRawCells && __ldg(page + 1))) ok = false;
                        count_only = ok;
                        page_bytes += 1;
                    } else if (ok) {
                        if (col.size < hdr || __ldg(page) != 3) {
                            ok = false;  // not a plain EncodeTypeDelta page
                        } else {
                            if (is_float) exp = static_cast<int16_t>((static_cast<uint32_t>(__ldg(page + 1)) << 8) | __ldg(page + 2));
                            first = conv_bytes_to_int64(page + hdr - 8);
                            const uintptr_t a = reinterpret_cast<uintptr_t>(page + hdr);
                            abase = reinterpret_cast<const uint8_t *>(a & ~static_cast<uintptr_t>(15));
                            pstart = static_cast<uint32_t>(a & 15);
                            pend = pstart + (col.size - hdr);
                            total = (pend + 15u) & ~15u;
                            nst = pend > pstart ? (total + kStageBytes - 1) / kStageBytes : 0;
                            has_page = true;
                            page_bytes += col.size;
                        }
                    }
                }
            }
            const bool streams = ok && has_page && nst > 0;
            // ---- one continuous ring over the batch's pages: stage s of the batch belongs to the lane with sb <= s < sb + nst
            uint32_t sb = streams ? nst : 0;
#pragma unroll
            for (int sft = 1; sft < static_cast<int>(kExpressBatch); sft <<= 1) {
                const uint32_t o = __shfl_up_sync(0xffffffffu, sb, sft);
                if (lane >= sft) sb += o;
            }
            const uint32_t ts = __shfl_sync(0xffffffffu, sb, kExpressBatch - 1);  // stages of the whole batch
            sb -= streams ? nst : 0;                                               // exclusive
            const uint32_t seq0 = seq;
            auto issue = [&](uint32_t s) {
                const uint32_t bal = __ballot_sync(0xffffffffu, streams && s >= sb && s < sb + nst);
                const int src = __ffs(bal) - 1;
                const uint64_t ab = shfl_u64(reinterpret_cast<uint64_t>(abase), src);
                const uint32_t tot = __shfl_sync(0xffffffffu, total, src);
                const uint32_t off = (s - __shfl_sync(0xffffffffu, sb, src)) * kStageBytes;
                if (lane == 0) {
                    const uint32_t bytes = min(static_cast<uint32_t>(kStageBytes), tot - off);
                    const uint32_t slot = (seq0 + s) % kStages;
                    mbar_expect_tx(&sm->bar[slot], bytes);
                    tma_load_1d(sm->stage[slot], reinterpret_cast<const uint8_t *>(ab) + off, bytes, &sm->bar[slot]);
                }
            };
            __syncwarp();
            for (uint32_t s = 0; s < ts && s < static_cast<uint32_t>(kStages); ++s) issue(s);
            seq += ts;
            for (uint32_t k = 0; k < nb; ++k) {
                const bool okk = __shfl_sync(0xffffffffu, ok, k);
                if (!okk) continue;
                const bool pagek = __shfl_sync(0xffffffffu, has_page, k);
                const bool cok = __shfl_sync(0xffffffffu, count_only, k);
                const uint32_t count_k = __shfl_sync(0xffffffffu, count, k);
                AggAcc acc;
                acc.init();
                bool good = true;
                if (pagek) {
                    const uint32_t nst_k = __shfl_sync(0xffffffffu, nst, k), sb_k = __shfl_sync(0xffffffffu, sb, k);
                    const uint32_t ps_k = __shfl_sync(0xffffffffu, pstart, k), pe_k = __shfl_sync(0xffffffffu, pend, k);
                    const uint32_t tot_k = __shfl_sync(0xffffffffu, total, k);
                    const int64_t first_k = static_cast<int64_t>(shfl_u64(static_cast<uint64_t>(first), k));
                    const uint32_t nchunks = (tot_k + kSwarChunkBytes - 1) / kSwarChunkBytes;
                    int64_t S = 0;
                    uint32_t tb = 0, carry_w = 0, last_byte = 0;
                    for (uint32_t j = 0; j < nst_k; ++j) {
                        const uint32_t s = sb_k + j;
                        const uint8_t *buf = ring_wait(sm, seq0 + s);
                        const uint32_t c1 = min(nchunks, (j + 1) * kChunksPerStage);
                        for (uint32_t cc = j * kChunksPerStage; cc < c1; ++cc) {
                            if (good) {
                                const SwarChunk ch = swar_chunk(buf, cc, ps_k, pe_k, tot_k, carry_w, lane);
                                if (ch.wide) {
                                    good = false;  // keep consuming the page's stages (the ring stays in step), stop decoding
                                } else {
                                    uint32_t n_in = ch.n;
#pragma unroll
                                    for (int sft = 1; sft < 32; sft <<= 1) {
                                        const uint32_t on = __shfl_up_sync(0xffffffffu, n_in, sft);
                                        if (lane >= sft) n_in += on;
                                    }
                                    const int64_t A1 = static_cast<int64_t>(count_k) - static_cast<int64_t>(tb) - static_cast<int64_t>(n_in - ch.n);
                                    S += A1 * static_cast<int64_t>(ch.T) - static_cast<int64_t>(ch.Rp);
                                    tb += __shfl_sync(0xffffffffu, n_in, 31);
                                }
                            }
                            if (cc == nchunks - 1 && lane == 0) last_byte = buf[(pe_k - 1) % kStageBytes];
                        }
                        __syncwarp();
                        if (s + kStages < ts) issue(s + kStages);
                    }
                    last_byte = __shfl_sync(0xffffffffu, last_byte, 0);
                    if (nst_k == 0) good = count_k == 1;  // an empty body: the page holds `first` alone
                    else good = good && tb + 1 == count_k && last_byte < 0x80u;
#pragma unroll
                    for (int m = 16; m >= 1; m >>= 1) S += static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(S), m));
                    acc.add_scaled(first_k, count_k);
                    const uint64_t us = static_cast<uint64_t>(S);
                    acc.lo += us;
                    acc.hi += (S >> 63) + (acc.lo < us ? 1 : 0);
                    acc.cnt = count_k;
                } else if (cok) {
                    acc.cnt = count_k;
                }
                if (static_cast<uint32_t>(lane) == k) {
                    if (!good) {
                        ok = false;
                    } else {
                        BlockPartial bp;
                        bp.sum.i = 0;
                        bp.mn.i = 0;
                        bp.mx.i = 0;
                        bp.cnt = acc.cnt;
                        if (acc.cnt > 0 && is_float) {
                            double sd;
                            if (acc.hi == (static_cast<int64_t>(acc.lo) >> 63)) sd = __ll2double_rn(static_cast<int64_t>(acc.lo));
                            else sd = __ll2double_rn(acc.hi) * 18446744073709551616.0 + __ull2double_rn(acc.lo);
                            bp.sum.f = scale_decimal(sd, exp);
                            bp.mn.f = scale_decimal(__ll2double_rn(acc.mn), exp);
                            bp.mx.f = scale_decimal(__ll2double_rn(acc.mx), exp);
                        } else if (acc.cnt > 0) {
                            bp.sum.i = static_cast<int64_t>(acc.lo);
                            bp.mn.i = acc.mn;
                            bp.mx.i = acc.mx;
                        }
                        p.P[static_cast<size_t>(g) * p.n_fcols + c] = bp;
                    }
                }
            }
        }
        // ---- finish: completed blocks are accounted, the others go to the regular fast lane
        const bool done = mine && ok;
        if (done) p.Prows[g] = count;
        const uint32_t rows_sum = __reduce_add_sync(0xffffffffu, done ? count : 0u);
        const uint32_t bytes_sum = __reduce_add_sync(0xffffffffu, done ? page_bytes : 0u);
        const uint32_t done_bal = __ballot_sync(0xffffffffu, done), rest_bal = __ballot_sync(0xffffffffu, mine && !ok);
        uint32_t rbase = 0;
        st_rows += rows_sum;
        st_bytes += bytes_sum;
        st_blocks += __popc(done_bal);
        if (lane == 0 && rest_bal) rbase = atomicAdd(p.rest_count, static_cast<uint32_t>(__popc(rest_bal)));
        rbase = __shfl_sync(0xffffffffu, rbase, 0);
        if (mine && !ok) p.rest_list[rbase + __popc(rest_bal & ((1u << lane) - 1u))] = g;
    }
    if (lane == 0 && st_blocks) {
        atomicAdd(&p.stats[0], st_rows);
        atomicAdd(&p.stats[1], st_rows);
        atomicAdd(&p.stats[2], st_bytes);
        atomicAdd(&p.stats[3], static_cast<unsigned long long>(st_blocks));
    }
    if (sm->fault && lane == 0) atomicCAS(&p.err[0], 0u, static_cast<uint32_t>(kErrTmaTimeout));
}


// ------------------------------------------------------------------------------------------------
// version dedup across parts (banyand/measure/query.go:912-942,995-1004; query_batch.go:151-161):
// a (series, timestamp) present in several parts keeps only the row with the highest version.
//   detect_overlap  thread per query series: parts whose selected time spans intersect -> flag blocks
//   dedup_decode    warp per flagged block: timestamps + versions -> global arrays
//   dedup_shadow    warp per flagged block: binary-search every row's timestamp in the other parts'
//                   blocks of the series; clear the row's bit in the shadow mask when a higher
//                   version (or the same version in an earlier part) exists
// scan_blocks then starts the row mask of a flagged block from its shadow mask.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t series_first_block(const ScanParams &p, uint32_t pi, uint32_t qi, uint64_t sid) {
    const DevPartRef &part = p.parts[pi];
    if (p.first_block) {
        const uint32_t g0 = p.first_block[static_cast<size_t>(pi) * p.n_series + qi];
        return g0 == 0xffffffffu ? part.n_blocks : g0 - part.block_base;
    }
    uint32_t lo = 0, hi = part.n_blocks;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (part.blocks[mid].sid < sid) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__global__ void detect_overlap_kernel(const __grid_constant__ ScanParams p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n_series) return;
    const uint64_t sid = p.q_sids[i];
    // spans of the selected blocks per part; conservative merge beyond 8 parts
    int64_t lo[8], hi[8];
    int ns = 0;
    bool overlap = false;
    for (uint32_t pi = 0; pi < p.n_parts; ++pi) {
        const DevPartRef &part = p.parts[pi];
        int64_t plo = INT64_MAX, phi = INT64_MIN;
        for (uint32_t b = series_first_block(p, pi, i, sid); b < part.n_blocks && part.blocks[b].sid == sid; ++b) {
            if (p.block_qsid[part.block_base + b] < 0) continue;
            plo = part.blocks[b].ts_min < plo ? part.blocks[b].ts_min : plo;
            phi = part.blocks[b].ts_max > phi ? part.blocks[b].ts_max : phi;
        }
        if (plo > phi) continue;
        for (int s = 0; s < ns; ++s)
            if (!(phi < lo[s] || plo > hi[s])) overlap = true;
        if (ns < 8) {
            lo[ns] = plo;
            hi[ns] = phi;
            ++ns;
        } else {
            lo[7] = plo < lo[7] ? plo : lo[7];
            hi[7] = phi > hi[7] ? phi : hi[7];
        }
    }
    if (!overlap) return;
    for (uint32_t pi = 0; pi < p.n_parts; ++pi) {
        const DevPartRef &part = p.parts[pi];
        for (uint32_t b = series_first_block(p, pi, i, sid); b < part.n_blocks && part.blocks[b].sid == sid; ++b) {
            const uint32_t g = part.block_base + b;
            if (p.block_qsid[g] < 0) continue;
            const unsigned long long idx = atomicAdd(&p.dd_counts[0], 1ull);
            p.dd_row_off[g] = atomicAdd(&p.dd_counts[1], static_cast<unsigned long long>(part.blocks[b].count));
            p.dd_index[g] = static_cast<int32_t>(idx);
            p.dd_list[idx] = g;
        }
    }
}

struct StoreCons {
    int64_t *out;
    uint32_t limit;  // rows of the block: a corrupt page may decode more values
    __device__ __forceinline__ void operator()(uint32_t row, int64_t v) {
        if (row < limit) out[row] = v;
    }
};

// decodes one int64 list body (timestamps or versions) into out[0..count)
__device__ __forceinline__ bool decode_list_to(WarpSmem *sm, const uint8_t *body, uint32_t len, uint32_t enc, int64_t first, uint32_t count,
                                               int64_t *out, int lane) {
    if (enc == 1 || enc == 2) {
        int64_t d = 0;
        uint32_t used = 0;
        if (enc == 1 && len != 0) return false;
        if (enc == 2 && (!read_varint_seq(body, len, d, used) || used != len)) return false;
        for (uint32_t r = lane; r < count; r += 32) out[r] = first + static_cast<int64_t>(static_cast<uint64_t>(d) * r);
        return true;
    }
    StoreCons sc;
    sc.out = out;
    sc.limit = count;
    bool ok;
    if (enc == 3) ok = decode_varint_page<false>(sm, body, len, count, first, sc, lane);
    else if (enc == 4) ok = decode_varint_page<true>(sm, body, len, count, first, sc, lane);
    else ok = false;
    return __all_sync(0xffffffffu, ok);
}

__global__ void __launch_bounds__(kWarpsPerCta * 32, 2) dedup_kernel(const __grid_constant__ ScanParams p, int phase) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    WarpSmem *sm = reinterpret_cast<WarpSmem *>(smem_raw) + warp;
    if (lane == 0) {
        sm->fault = 0;
        sm->seq = 0;
        sm->st_rows = sm->st_matched = sm->st_bytes = 0;
        sm->st_blocks = sm->st_deferred = sm->st_why = 0;
        for (int s = 0; s < kStages; ++s) mbar_init(&sm->bar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint32_t gw = blockIdx.x * kWarpsPerCta + warp, nw = gridDim.x * kWarpsPerCta;
    for (uint32_t k = gw; k < p.n_dd_blocks; k += nw) {
        const uint32_t g = p.dd_list[k];
        uint32_t pi = 0;
        while (pi + 1 < p.n_parts && g >= p.parts[pi + 1].block_base) ++pi;
        const DevPartRef &part = p.parts[pi];
        const DevBlock blk = part.blocks[g - part.block_base];
        const unsigned long long off = p.dd_row_off[g];
        if (phase == 0) {
            const uint8_t *tsp = part.files[0] + blk.ts_off;
            bool ok = decode_list_to(sm, tsp, blk.ver_off, blk.ts_enc, blk.ts_min, blk.count, p.dd_ts + off, lane);
            ok = ok && decode_list_to(sm, tsp + blk.ver_off, blk.ts_size - blk.ver_off, blk.ver_enc, blk.ver_first, blk.count, p.dd_ver + off, lane);
            if (!ok || blk.count > kMaskWords * 32) set_err(p, !ok ? kErrCorrupt : kErrBigBlock, g, lane);
            continue;
        }
        // phase 1: shadow mask
        uint32_t *shadow = p.dd_shadow + static_cast<size_t>(k) * kMaskWords;
        const uint32_t nwords = (blk.count + 31) >> 5;
        if (blk.count > kMaskWords * 32) continue;
        const int32_t qi = p.block_qsid[g];
        for (uint32_t w = 0; w < nwords; ++w) {
            const uint32_t row = (w << 5) + lane;
            bool keep = row < blk.count;
            if (keep) {
                const int64_t t = p.dd_ts[off + row], v = p.dd_ver[off + row];
                for (uint32_t qp = 0; qp < p.n_parts && keep; ++qp) {
                    if (qp == pi) continue;
                    const DevPartRef &other = p.parts[qp];
                    for (uint32_t b = series_first_block(p, qp, static_cast<uint32_t>(qi), blk.sid); b < other.n_blocks && other.blocks[b].sid == blk.sid; ++b) {
                        const DevBlock &ob = other.blocks[b];
                        if (ob.ts_min > t) break;
                        if (ob.ts_max < t) continue;
                        const uint32_t og = other.block_base + b;
                        if (p.dd_index[og] < 0) continue;
                        const int64_t *ots = p.dd_ts + p.dd_row_off[og];
                        uint32_t lo = 0, hi = ob.count;
                        while (lo < hi) {
                            const uint32_t mid = (lo + hi) >> 1;
                            if (ots[mid] < t) lo = mid + 1;
                            else hi = mid;
                        }
                        if (lo < ob.count && ots[lo] == t) {
                            const int64_t ov = p.dd_ver[p.dd_row_off[og] + lo];
                            if (ov > v || (ov == v && qp < pi)) keep = false;
                        }
                    }
                }
            }
            const uint32_t bal = __ballot_sync(0xffffffffu, keep);
            if (lane == 0) shadow[w] = bal;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// deterministic reduction of the per-block partials
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void combine(BlockPartial &a, const BlockPartial &b, bool is_float) {
    if (b.cnt == 0) return;
    if (a.cnt == 0) {
        a = b;
        return;
    }
    if (is_float) {
        a.sum.f += b.sum.f;
        a.mn.f = b.mn.f < a.mn.f ? b.mn.f : a.mn.f;
        a.mx.f = b.mx.f > a.mx.f ? b.mx.f : a.mx.f;
    } else {
        a.sum.i = static_cast<int64_t>(static_cast<uint64_t>(a.sum.i) + static_cast<uint64_t>(b.sum.i));
        a.mn.i = b.mn.i < a.mn.i ? b.mn.i : a.mn.i;
        a.mx.i = b.mx.i > a.mx.i ? b.mx.i : a.mx.i;
    }
    a.cnt += b.cnt;
}

// one WARP per query series: the series' blocks are contiguous inside a part (block_metadata.go:170-175),
// so lanes take consecutive blocks, and a fixed shuffle tree combines them (deterministic).  Also detects
// overlapping time spans across parts, which need the version dedup of query.go:995-1004.
__device__ __forceinline__ void warp_combine(BlockPartial &acc, bool is_float, int lane) {
#pragma unroll
    for (int m = 1; m < 32; m <<= 1) {
        BlockPartial o;
        o.sum.i = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.sum.i), m));
        o.mn.i = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.mn.i), m));
        o.mx.i = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.mx.i), m));
        o.cnt = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.cnt), m));
        // lower lane first, so both partners compute the same value and block order is respected
        BlockPartial a = (lane & m) ? o : acc, b = (lane & m) ? acc : o;
        combine(a, b, is_float);
        acc = a;
    }
}

__global__ void __launch_bounds__(256) series_reduce_kernel(const __grid_constant__ ReduceParams p) {
    const int lane = threadIdx.x & 31;
    const uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= p.n_series) return;
    const uint64_t sid = p.q_sids[i];
    BlockPartial acc[kMaxFcols];
    for (uint32_t c = 0; c < p.n_fcols; ++c) {
        acc[c].sum.i = 0;
        acc[c].mn.i = 0;
        acc[c].mx.i = 0;
        acc[c].cnt = 0;
    }
    int64_t rows = 0;
    int64_t kts = INT64_MAX;  // group-key passes: (ts_min, row) of the first surviving row of the series, lane-local until the end
    uint32_t krow = 0;
    int64_t span_lo[4], span_hi[4];
    int nspan = 0;
    bool overlap = false;
    for (uint32_t pi = 0; pi < p.n_parts; ++pi) {
        const DevPartRef &part = p.parts[pi];
        uint32_t lo = 0, hi = part.n_blocks;
        if (p.first_block) {
            const uint32_t g0 = p.first_block[static_cast<size_t>(pi) * p.n_series + i];
            lo = g0 == 0xffffffffu ? part.n_blocks : g0 - part.block_base;
        } else {
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (part.blocks[mid].sid < sid) lo = mid + 1;
                else hi = mid;
            }
        }
        int64_t plo = INT64_MAX, phi = INT64_MIN;
        for (uint32_t base = lo; base < part.n_blocks; base += 32) {
            const uint32_t b = base + lane;
            const bool mine = b < part.n_blocks && part.blocks[b].sid == sid;
            const uint32_t g = part.block_base + b;
            const bool sel = mine && p.block_qsid[g] >= 0;
            int64_t r = 0, tlo = INT64_MAX, thi = INT64_MIN;
            if (sel) {
                r = p.Prows[g];
                tlo = part.blocks[b].ts_min;
                thi = part.blocks[b].ts_max;
            }
            if (p.Kts && r > 0 && tlo < kts) {
                kts = tlo;
                krow = p.Pfirst[g];
            }
#pragma unroll
            for (int m = 16; m >= 1; m >>= 1) {
                r += static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(r), m));
                const int64_t ol = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(tlo), m));
                const int64_t oh = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(thi), m));
                tlo = ol < tlo ? ol : tlo;
                thi = oh > thi ? oh : thi;
            }
            rows += r;
            plo = tlo < plo ? tlo : plo;
            phi = thi > phi ? thi : phi;
            for (uint32_t c = 0; c < p.n_fcols; ++c) {
                BlockPartial bp;
                bp.sum.i = 0;
                bp.mn.i = 0;
                bp.mx.i = 0;
                bp.cnt = 0;
                if (sel) bp = p.P[static_cast<size_t>(g) * p.n_fcols + c];
                const bool is_float = p.col_type[c] == BYDB_VT_FLOAT64;
                warp_combine(bp, is_float, lane);
                combine(acc[c], bp, is_float);
            }
            if (__ballot_sync(0xffffffffu, mine) != 0xffffffffu) break;
        }
        if (plo <= phi) {
            for (int s = 0; s < nspan; ++s)
                if (!(phi < span_lo[s] || plo > span_hi[s])) overlap = true;
            if (nspan < 4) {
                span_lo[nspan] = plo;
                span_hi[nspan] = phi;
                ++nspan;
            } else {  // merge into the last span: conservative
                span_lo[3] = plo < span_lo[3] ? plo : span_lo[3];
                span_hi[3] = phi > span_hi[3] ? phi : span_hi[3];
            }
        }
    }
    if (p.Kts) {
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            const int64_t ot = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(kts), m));
            const uint32_t orow = __shfl_xor_sync(0xffffffffu, krow, m);
            if (ot < kts) {
                kts = ot;
                krow = orow;
            }
        }
        if (lane == 0) {
            p.Kts[i] = kts;
            p.Krow[i] = krow;
        }
    }
    if (lane != 0) return;
    if (overlap && !p.dedup_done && atomicCAS(&p.err[0], 0u, static_cast<uint32_t>(kErrOverlap)) == 0u) p.err[1] = i;
    for (uint32_t c = 0; c < p.n_fcols; ++c) p.S[static_cast<size_t>(i) * p.n_fcols + c] = acc[c];
    p.Srows[i] = rows;
}

// one CTA per group: fixed-stride accumulation + fixed shuffle tree => run-to-run identical sums
__global__ void __launch_bounds__(256) group_reduce_kernel(const __grid_constant__ ReduceParams p) {
    const int32_t g = blockIdx.x;
    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    __shared__ BlockPartial s_part[8];
    __shared__ int64_t s_rows[8];
    const int32_t lo = p.group_start[g], hi = p.group_start[g + 1];
    const size_t GF = static_cast<size_t>(p.n_groups) * p.n_fcols;
    (void)GF;
    int64_t rows = 0;
    for (int32_t k = lo + tid; k < hi; k += blockDim.x) rows += p.Srows[p.order[k]];
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) rows += static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(rows), m));
    if (lane == 0) s_rows[warp] = rows;
    __syncthreads();
    if (tid == 0) {
        int64_t r = 0;
        for (int w = 0; w < 8; ++w) r += s_rows[w];
        p.rows[g] = r;
    }
    for (uint32_t c = 0; c < p.n_fcols; ++c) {
        const bool is_float = p.col_type[c] == BYDB_VT_FLOAT64;
        BlockPartial acc;
        acc.sum.i = 0;
        acc.mn.i = 0;
        acc.mx.i = 0;
        acc.cnt = 0;
        for (int32_t k = lo + tid; k < hi; k += blockDim.x) combine(acc, p.S[static_cast<size_t>(p.order[k]) * p.n_fcols + c], is_float);
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            BlockPartial o;
            o.sum.i = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.sum.i), m));
            o.mn.i = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.mn.i), m));
            o.mx.i = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.mx.i), m));
            o.cnt = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.cnt), m));
            // combine in lane order so that both partners compute the same value
            BlockPartial a = (lane & m) ? o : acc, b = (lane & m) ? acc : o;
            combine(a, b, is_float);
            acc = a;
        }
        __syncthreads();
        if (lane == 0) s_part[warp] = acc;
        __syncthreads();
        if (tid == 0) {
            BlockPartial t = s_part[0];
            for (int w = 1; w < 8; ++w) combine(t, s_part[w], is_float);
            const size_t o = static_cast<size_t>(g) * p.n_fcols + c;
            const bool have = t.cnt > 0;
            p.cnt[o] = t.cnt;
            p.sum_f64[o] = (have && is_float) ? t.sum.f : 0.0;
            p.max_f64[o] = (have && is_float) ? t.mx.f : -INFINITY;
            p.negmin_f64[o] = (have && is_float) ? -t.mn.f : -INFINITY;
            p.sum_i64[o] = (have && !is_float) ? t.sum.i : 0;
            p.max_i64[o] = (have && !is_float) ? t.mx.i : INT64_MIN;
            p.notmin_i64[o] = (have && !is_float) ? ~t.mn.i : INT64_MIN;
            // the scan's status rides in the table (bits 8..): an asynchronous bydb_scan_partials has no other way
            // to tell the rank that finalises that one of its blocks failed
            if (g == 0) p.coltype[c] = static_cast<int64_t>(p.col_type[c]) | (static_cast<int64_t>(p.err[0]) << 8);
        }
    }
}

// The same reduce for groups of at most 32 series (a service with a handful of instances): one WARP per group, eight groups per
// CTA.  The CTA version above degenerates to exactly this tree for such a group (thread k < 32 holds series k, warps 1..7 hold
// nothing), so the sums are bit-identical; what goes away is a thousand 256-thread CTAs with two barriers each.
__global__ void __launch_bounds__(256) group_reduce_small_kernel(const __grid_constant__ ReduceParams p) {
    const int lane = threadIdx.x & 31;
    const int32_t g = static_cast<int32_t>((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (g >= p.n_groups) return;
    const int32_t lo = p.group_start[g], hi = p.group_start[g + 1];
    const int32_t k = lo + lane;
    int64_t rows = k < hi ? p.Srows[p.order[k]] : 0;
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) rows += static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(rows), m));
    if (lane == 0) p.rows[g] = rows;
    for (uint32_t c = 0; c < p.n_fcols; ++c) {
        const bool is_float = p.col_type[c] == BYDB_VT_FLOAT64;
        BlockPartial acc;
        acc.sum.i = 0;
        acc.mn.i = 0;
        acc.mx.i = 0;
        acc.cnt = 0;
        if (k < hi) combine(acc, p.S[static_cast<size_t>(p.order[k]) * p.n_fcols + c], is_float);
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            BlockPartial o;
            o.sum.i = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.sum.i), m));
            o.mn.i = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.mn.i), m));
            o.mx.i = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.mx.i), m));
            o.cnt = static_cast<int64_t>(shfl_xor_u64(static_cast<uint64_t>(acc.cnt), m));
            BlockPartial a = (lane & m) ? o : acc, b = (lane & m) ? acc : o;
            combine(a, b, is_float);
            acc = a;
        }
        if (lane == 0) {
            const BlockPartial &t = acc;
            const size_t o = static_cast<size_t>(g) * p.n_fcols + c;
            const bool have = t.cnt > 0;
            p.cnt[o] = t.cnt;
            p.sum_f64[o] = (have && is_float) ? t.sum.f : 0.0;
            p.max_f64[o] = (have && is_float) ? t.mx.f : -INFINITY;
            p.negmin_f64[o] = (have && is_float) ? -t.mn.f : -INFINITY;
            p.sum_i64[o] = (have && !is_float) ? t.sum.i : 0;
            p.max_i64[o] = (have && !is_float) ? t.mx.i : INT64_MIN;
            p.notmin_i64[o] = (have && !is_float) ? ~t.mn.i : INT64_MIN;
            if (g == 0) p.coltype[c] = static_cast<int64_t>(p.col_type[c]) | (static_cast<int64_t>(p.err[0]) << 8);
        }
    }
}

// finalisation: pkg/query/aggregation/function.go Val() + output typing aggregation.go:425-430
__device__ __forceinline__ void finalize_header(const FinalizeParams &p) {
    for (uint32_t a = 0; a < p.n_aggs; ++a)
        p.out_is_float[a] = ((p.agg_func[a] != BYDB_AGG_COUNT || p.row_path_types) && (p.coltype[p.agg_fcol[a]] & 0xff) == BYDB_VT_FLOAT64) ? 1 : 0;
    uint32_t e = 0;
    for (uint32_t c = 0; c < p.n_fcols; ++c) {
        const uint32_t ec = static_cast<uint32_t>(p.coltype[c] >> 8);
        e = ec > e ? ec : e;
    }
    if (p.err_out) *p.err_out = e;
}
__device__ __forceinline__ void finalize_group(const FinalizeParams &p, int32_t g) {
    for (uint32_t a = 0; a < p.n_aggs; ++a) {
        const uint32_t c = p.agg_fcol[a];
        const size_t o = static_cast<size_t>(g) * p.n_fcols + c;
        const size_t oo = static_cast<size_t>(g) * p.n_aggs + a;
        const int64_t typ = p.coltype[c] & 0xff;
        const int64_t cnt = p.cnt[o];
        int64_t vi = 0;
        double vf = 0.0;
        const int fn = p.agg_func[a];
        if (typ != 0) {
            if (fn == BYDB_AGG_COUNT) {
                vi = cnt;
                if (p.row_path_types && typ == BYDB_VT_FLOAT64) vf = __ll2double_rn(cnt);  // countFunc[float64], function.go:78-93
            } else if (typ == BYDB_VT_FLOAT64) {
                switch (fn) {
                    case BYDB_AGG_SUM: vf = p.sum_f64[o]; break;
                    case BYDB_AGG_MAX: vf = cnt > 0 ? p.max_f64[o] : -DBL_MAX; break;  // aggregation.go:169-191 sentinels
                    case BYDB_AGG_MIN: vf = cnt > 0 ? -p.negmin_f64[o] : DBL_MAX; break;
                    case BYDB_AGG_MEAN: {
                        if (cnt > 0) {
                            vf = __ddiv_rn(p.sum_f64[o], __ll2double_rn(cnt));
                            if (vf < 1.0) vf = 1.0;  // function.go:31-40
                        }
                        break;
                    }
                }
            } else {
                switch (fn) {
                    case BYDB_AGG_SUM: vi = p.sum_i64[o]; break;
                    case BYDB_AGG_MAX: vi = cnt > 0 ? p.max_i64[o] : INT64_MIN; break;
                    case BYDB_AGG_MIN: vi = cnt > 0 ? ~p.notmin_i64[o] : INT64_MAX; break;
                    case BYDB_AGG_MEAN: {
                        if (cnt > 0) {
                            vi = p.sum_i64[o] / cnt;  // Go integer division truncates toward zero
                            if (vi < 1) vi = 1;
                        }
                        break;
                    }
                }
            }
        }
        p.out_i64[oo] = vi;
        p.out_f64[oo] = vf;
    }
}
__global__ void finalize_kernel(const __grid_constant__ FinalizeParams p) {
    const int32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g == 0) finalize_header(p);
    if (g < p.n_groups) finalize_group(p, g);
}


// ------------------------------------------------------------------------------------------------
// select_rows: which groups become output rows, in which order (one CTA; G is small next to the scan)
//   top_n == 0 : stable compaction of the groups with rows > 0 (group-id = first-appearance order,
//                pkg/query/vectorized/measure/aggregation.go:211-213)
//   top_n  > 0 : pkg/query/vectorized/measure/top.go:62-117 -- order by the aggregate, nulls lowest,
//                ties -> earlier row.  MSB-first radix select (8 x 8 bit histograms in shared memory)
//                finds the N-th key, an ordered pass resolves the ties by group id, a bitonic sort
//                orders the <= 2048 selected rows.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *warp_tot, uint32_t &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int s = 1; s < 32; s <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, incl, s);
        if (lane >= s) incl += o;
    }
    __syncthreads();
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    uint32_t base = 0;
    total = 0;
    for (int w = 0; w < nw; ++w) {
        const uint32_t t = warp_tot[w];
        if (w < warp) base += t;
        total += t;
    }
    return base + incl - v;
}

__device__ __forceinline__ uint64_t order_key_i64(int64_t v) { return static_cast<uint64_t>(v) ^ (1ull << 63); }
__device__ __forceinline__ uint64_t order_key_f64(double d) {
    const uint64_t b = static_cast<uint64_t>(__double_as_longlong(d));
    return (b >> 63) ? ~b : (b | (1ull << 63));
}

// kFused: the finalisation runs in this (single) CTA first -- one launch less on the tail of every query with few groups
template <bool kFused>
__global__ void __launch_bounds__(1024) select_rows_kernel(const __grid_constant__ SelectParams p, const __grid_constant__ FinalizeParams fp) {
    if (kFused) {
        if (threadIdx.x == 0) finalize_header(fp);
        for (int32_t g = threadIdx.x; g < fp.n_groups; g += blockDim.x) finalize_group(fp, g);
        __syncthreads();  // global writes of this CTA are visible to its own threads after the barrier
    }
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_hist[256];
    __shared__ uint64_t s_key[kMaxDeviceTopN];
    __shared__ int32_t s_gid[kMaxDeviceTopN];
    __shared__ uint64_t s_prefix;
    __shared__ uint32_t s_remaining, s_count, s_nn, s_nulls;
    const int tid = threadIdx.x;
    const int32_t G = p.n_groups;
    const uint32_t A = p.n_aggs;
    auto emit = [&](uint32_t pos, int32_t g) {
        p.sel_group[pos] = g;
        p.sel_rows[pos] = p.rows[g];
        for (uint32_t a = 0; a < A; ++a) {
            p.sel_i64[static_cast<size_t>(pos) * A + a] = p.val_i64[static_cast<size_t>(g) * A + a];
            p.sel_f64[static_cast<size_t>(pos) * A + a] = p.val_f64[static_cast<size_t>(g) * A + a];
        }
    };
    if (p.top_n <= 0) {
        uint32_t base = 0;
        for (int32_t g0 = 0; g0 < G; g0 += blockDim.x) {
            const int32_t g = g0 + tid;
            const uint32_t f = (g < G && p.rows[g] > 0) ? 1u : 0u;
            uint32_t tot;
            const uint32_t pos = base + block_excl_scan(f, s_warp, tot);
            if (f) emit(pos, g);
            base += tot;
            __syncthreads();
        }
        if (tid == 0) *p.sel_count = base;
        return;
    }
    // ---- keys: 0 for rows that do not compete; nulls are counted apart (they sort lowest as values)
    const bool isf = p.is_float[p.top_agg] != 0;
    uint32_t my_nn = 0, my_null = 0;
    for (int32_t g = tid; g < G; g += blockDim.x) {
        uint64_t k = 0;
        uint8_t st = 0;  // 0 = no output row, 1 = null aggregate, 2 = competes with key k
        if (p.rows[g] > 0) {
            const bool null = !p.top_is_count && p.cnt[static_cast<size_t>(g) * p.n_fcols + p.top_fcol] == 0;
            if (null) {
                st = 1;
                ++my_null;
            } else {
                const size_t o = static_cast<size_t>(g) * A + p.top_agg;
                k = isf ? order_key_f64(p.val_f64[o]) : order_key_i64(p.val_i64[o]);
                if (!p.top_desc) k = ~k;  // ascending: the smallest value gets the largest key
                st = 2;
                ++my_nn;
            }
        }
        p.keys[g] = k;
        p.kstate[g] = st;
    }
    uint32_t tot;
    (void)block_excl_scan(my_nn, s_warp, tot);
    if (tid == 0) s_nn = tot;
    __syncthreads();
    (void)block_excl_scan(my_null, s_warp, tot);
    if (tid == 0) s_nulls = tot;
    __syncthreads();
    const uint32_t N = static_cast<uint32_t>(p.top_n);
    const uint32_t n_nulls_first = p.top_desc ? 0u : min(N, s_nulls);                  // asc: nulls lead
    const uint32_t M = min(N - n_nulls_first, s_nn);                                     // competing rows to take
    const uint32_t n_nulls_last = p.top_desc ? min(N - M, s_nulls) : 0u;               // desc: nulls trail
    const bool few = G <= kMaxDeviceTopN;  // few groups: no selection pass -- all of them go through the bitonic sort below
    // ---- radix select of the M-th largest competing key
    if (tid == 0) {
        s_prefix = 0;
        s_remaining = M;
    }
    __syncthreads();
    if (M > 0 && !few) {
        for (int pass = 7; pass >= 0; --pass) {
            for (int i = tid; i < 256; i += blockDim.x) s_hist[i] = 0;
            __syncthreads();
            const uint64_t prefix = s_prefix;
            for (int32_t g = tid; g < G; g += blockDim.x) {
                if (p.kstate[g] != 2) continue;
                const uint64_t k = p.keys[g];
                if (pass < 7 && (k >> (8 * (pass + 1))) != prefix) continue;
                atomicAdd(&s_hist[(k >> (8 * pass)) & 255u], 1u);
            }
            __syncthreads();
            if (tid == 0) {
                uint32_t rem = s_remaining, above = 0;
                int d = 255;
                for (; d > 0; --d) {
                    if (above + s_hist[d] >= rem) break;
                    above += s_hist[d];
                }
                s_remaining = rem - above;
                s_prefix = (prefix << 8) | static_cast<uint64_t>(d);
            }
            __syncthreads();
        }
    }
    const uint64_t T = s_prefix;
    const uint32_t take_eq = s_remaining;
    // ---- collect: keys above T in any order, keys equal to T in group order
    if (tid == 0) s_count = 0;
    __syncthreads();
    uint32_t eq_base = 0;
    for (int32_t g0 = 0; g0 < G && M > 0 && !few; g0 += blockDim.x) {
        const int32_t g = g0 + tid;
        const uint64_t k = g < G ? p.keys[g] : 0;
        const bool comp = g < G && p.kstate[g] == 2;
        const uint32_t eq = (comp && k == T) ? 1u : 0u;
        uint32_t tot_eq;
        const uint32_t rank = eq_base + block_excl_scan(eq, s_warp, tot_eq);
        if (comp && (k > T || (eq && rank < take_eq))) {
            const uint32_t pos = atomicAdd(&s_count, 1u);
            if (pos < kMaxDeviceTopN) {
                s_key[pos] = k;
                s_gid[pos] = g;
            }
        }
        eq_base += tot_eq;
        __syncthreads();
    }
    __syncthreads();
    // ---- bitonic sort (key desc, group asc) of the selected rows -- or, with few groups, of every group: rows that do not
    //      compete carry (key 0, group INT32_MAX) and sort behind every competing row, the first M entries are the answer
    const uint32_t n_sort = few ? static_cast<uint32_t>(G) : M;
    if (few) {
        for (int32_t g = tid; g < G; g += blockDim.x) {
            const bool comp = p.kstate[g] == 2;
            s_key[g] = comp ? p.keys[g] : 0ull;
            s_gid[g] = comp ? g : INT32_MAX;
        }
    }
    uint32_t P2 = 1;
    while (P2 < n_sort) P2 <<= 1;
    for (uint32_t i = n_sort + tid; i < P2; i += blockDim.x) {
        s_key[i] = 0;
        s_gid[i] = INT32_MAX;
    }
    __syncthreads();
    if (P2 <= blockDim.x) {
        // one element per thread, kept in registers: compare-exchange steps inside a warp (j < 32: 40 of the 55 steps for 1024
        // elements) are two shuffles and no barrier; only the wider steps go through shared memory
        uint64_t mk = 0;
        int32_t mg = INT32_MAX;
        const uint32_t t = static_cast<uint32_t>(tid);
        if (t < P2) {
            mk = s_key[t];
            mg = s_gid[t];
        }
        for (uint32_t k2 = 2; k2 <= P2; k2 <<= 1) {
            for (uint32_t j = k2 >> 1; j > 0; j >>= 1) {
                uint64_t ok;
                int32_t og;
                if (j < 32) {
                    ok = shfl_xor_u64(mk, static_cast<int>(j));
                    og = __shfl_xor_sync(0xffffffffu, mg, static_cast<int>(j));
                } else {
                    __syncthreads();  // the previous wide step's reads are done
                    if (t < P2) {
                        s_key[t] = mk;
                        s_gid[t] = mg;
                    }
                    __syncthreads();
                    ok = t < P2 ? s_key[t ^ j] : 0;
                    og = t < P2 ? s_gid[t ^ j] : INT32_MAX;
                }
                const bool up = (t & k2) == 0, lower = (t & j) == 0;
                const bool mine_first = mk > ok || (mk == ok && mg < og);  // mine precedes the partner in the output
                // the lower position of the pair holds the preceding element when the run ascends (`up`), the other one otherwise
                const bool keep = lower ? (mine_first == up) : (mine_first != up);
                if (!keep) {
                    mk = ok;
                    mg = og;
                }
            }
        }
        __syncthreads();
        if (t < P2) {
            s_key[t] = mk;
            s_gid[t] = mg;
        }
        __syncthreads();
    } else
    for (uint32_t k2 = 2; k2 <= P2; k2 <<= 1) {
        for (uint32_t j = k2 >> 1; j > 0; j >>= 1) {
            for (uint32_t i = tid; i < P2; i += blockDim.x) {
                const uint32_t ixj = i ^ j;
                if (ixj > i) {
                    const bool up = (i & k2) == 0;
                    const uint64_t ka = s_key[i], kb = s_key[ixj];
                    const int32_t ga = s_gid[i], gb = s_gid[ixj];
                    const bool a_first = ka > kb || (ka == kb && ga < gb);  // a precedes b in the output
                    if (a_first != up) {
                        s_key[i] = kb;
                        s_key[ixj] = ka;
                        s_gid[i] = gb;
                        s_gid[ixj] = ga;
                    }
                }
            }
            __syncthreads();
        }
    }
    // ---- emit: [nulls (asc only)] [sorted competing rows] [nulls (desc only)]
    for (uint32_t i = tid; i < M; i += blockDim.x) emit(n_nulls_first + i, s_gid[i]);
    const uint32_t n_nulls = n_nulls_first + n_nulls_last;
    if (n_nulls > 0) {
        uint32_t base = 0;
        const uint32_t at = p.top_desc ? M : 0u;
        for (int32_t g0 = 0; g0 < G; g0 += blockDim.x) {
            const int32_t g = g0 + tid;
            const uint32_t f = (g < G && p.kstate[g] == 1) ? 1u : 0u;
            uint32_t tot2;
            const uint32_t pos = base + block_excl_scan(f, s_warp, tot2);
            if (f && pos < n_nulls) emit(at + pos, g);
            base += tot2;
            __syncthreads();
        }
    }
    if (tid == 0) *p.sel_count = M + n_nulls;
}


// Multi-GPU reduce after ONE all-gather of the per-rank partial tables: every word of the table is
// combined across ranks in rank order (deterministic float sums, unlike a ring all-reduce), which is
// the liaison's reduceAccumulator.Combine (measure_plan_aggregation.go:96-124) done on the device.
__global__ void combine_tables_kernel(uint64_t *t, uint32_t n, uint64_t words, uint64_t stride, uint64_t sf_lo, uint64_t sf_hi, uint64_t mf_lo, uint64_t mf_hi,
                                      uint64_t si_lo, uint64_t si_hi, uint64_t mi_lo, uint64_t mi_hi) {
    const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= words) return;
    uint64_t a = t[i];
    for (uint32_t r = 1; r < n; ++r) {
        const uint64_t b = t[static_cast<uint64_t>(r) * stride + i];
        if (i >= sf_lo && i < sf_hi) {
            a = static_cast<uint64_t>(__double_as_longlong(__longlong_as_double(static_cast<long long>(a)) + __longlong_as_double(static_cast<long long>(b))));
        } else if (i >= mf_lo && i < mf_hi) {
            const double x = __longlong_as_double(static_cast<long long>(a)), y = __longlong_as_double(static_cast<long long>(b));
            a = static_cast<uint64_t>(__double_as_longlong(y > x ? y : x));
        } else if (i >= si_lo && i < si_hi) {
            a += b;  // wraps like Go's int64
        } else if (i >= mi_lo && i < mi_hi) {
            a = static_cast<uint64_t>(static_cast<int64_t>(b) > static_cast<int64_t>(a) ? b : a);
        }
    }
    t[i] = a;
}

// ------------------------------------------------------------------------------------------------
// host launchers
// ------------------------------------------------------------------------------------------------

// ------------------------------------------------------------------------------------------------
// Group key: group-by on a stored dictionary tag, whose value changes from row to row inside a series
// (pkg/query/vectorized/measure/aggregation.go:193-254 Consume: key of the row -> group, new groups appended to the
// insertion list; groupby.go:226-254: a string / bytes key is its length + raw bytes, so a nil cell and "" are one key).
//   1. key_values_kernel: one warp per selected block reads the tag's dictionary page (<= 256 values per block,
//      pkg/encoding/dictionary.go:52-88) and enters every value into a small open-addressing table in global memory; a
//      slot holds the device address and length of the bytes inside the part, the bytes themselves never move.
//   2. the host runs one ordinary scan pass per distinct value v (predicate "tag is v"); group_reduce of pass v writes
//      slice v of a composite partial table of V x G groups, series_reduce records where each series first shows v.
//   3. key_order_kernel / key_perm_kernel put the composite groups into insertion order: the scan order is series by
//      series (ascending series id) and by time inside a series, so a group's first row is (first series that shows the
//      value, rank of the value among that series' values by first row); permute_table_kernel reorders the table and the
//      ordinary finalisation / Top-N runs on it unchanged (ties in Top-N go to the group inserted first, top.go:62-76).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void key_err(const KeyParams &p, uint32_t code, uint32_t g) {
    if (atomicCAS(&p.err[0], 0u, code) == 0u) p.err[1] = g;
}

__device__ void key_insert(const KeyParams &p, const uint8_t *bytes, uint32_t len, uint32_t g) {
    if (len > kMaxLit) {
        key_err(p, kErrKeyLong, g);
        return;
    }
    uint64_t h = 0xcbf29ce484222325ull;  // FNV-1a
    for (uint32_t i = 0; i < len; ++i) h = (h ^ __ldg(bytes + i)) * 0x100000001b3ull;
    const unsigned long long mine =
        (1ull << 63) | (static_cast<unsigned long long>(len) << 48) | (len ? (reinterpret_cast<uintptr_t>(bytes) & 0xffffffffffffull) : 0ull);
    uint32_t s = static_cast<uint32_t>(h ^ (h >> 32)) & (kKeySlots - 1);
    for (uint32_t probe = 0; probe < kKeySlots; ++probe) {
        unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(&p.slots[s]);
        if (cur == 0) {
            cur = atomicCAS(&p.slots[s], 0ull, mine);
            if (cur == 0) {
                if (atomicAdd(p.count, 1u) >= p.cap) key_err(p, kErrKeyCap, g);
                return;
            }
        }
        if (((cur >> 48) & 0x7fffu) == len) {
            const uint8_t *o = reinterpret_cast<const uint8_t *>(static_cast<uintptr_t>(cur & 0xffffffffffffull));
            bool eq = true;
            for (uint32_t i = 0; i < len && eq; ++i) eq = __ldg(o + i) == __ldg(bytes + i);
            if (eq) return;
        }
        s = (s + 1) & (kKeySlots - 1);
    }
    key_err(p, kErrKeyCap, g);
}

__global__ void __launch_bounds__(256) key_values_kernel(const __grid_constant__ KeyParams p) {
    const int lane = threadIdx.x & 31;
    const uint32_t n_warps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); g < p.total_blocks; g += n_warps) {
        uint32_t stop = lane == 0 ? *reinterpret_cast<volatile uint32_t *>(&p.err[0]) : 0u;
        stop = __shfl_sync(0xffffffffu, stop, 0);
        if (stop != 0u) return;  // warp-uniform
        uint32_t pi = 0;
        while (pi + 1 < p.n_parts && g >= p.parts[pi + 1].block_base) ++pi;
        const DevPartRef &part = p.parts[pi];
        const DevBlock blk = part.blocks[g - part.block_base];
        // the selection of plan_blocks_kernel
        uint32_t lo = 0, hi = p.n_series;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (p.q_sids[mid] < blk.sid) lo = mid + 1;
            else hi = mid;
        }
        if (!(lo < p.n_series && p.q_sids[lo] == blk.sid) || blk.ts_max < p.tmin || blk.ts_min > p.tmax) continue;
        DevCol col;
        if (!find_col(part, blk, p.key_name, col, lane)) {
            if (lane == 0) key_insert(p, nullptr, 0, g);  // column absent in this block: every cell is nil (block.go:226-233)
            continue;
        }
        uint32_t err = kErrNone;
        const uint8_t *page = part.files[col.file_id] + col.off;
        const uint8_t *q = page + 1, *end = page + col.size;
        uint64_t nvals = 0;
        uint32_t llen = 0, dlen = 0, width = 1;
        const uint8_t *lens = nullptr, *data = nullptr;
        if (col.value_type != BYDB_VT_STR && col.value_type != BYDB_VT_BINARY) err = kErrPredType;
        else if (col.size < 2) err = kErrCorrupt;
        else if (__ldg(page) == 9) err = kErrTagPlain;
        else if (__ldg(page) != 10) err = kErrBadEnc;
        else if (!read_varuint_seq(q, end, nvals) || nvals == 0 || nvals > 256) err = kErrCorrupt;
        if (err == kErrNone) err = read_cblock_header(q, end, llen, kErrZstdDict);
        if (err == kErrNone) {
            const uint8_t wt = llen >= 1 ? __ldg(q) : 4;
            width = 1u << (wt & 3);
            if (wt > 3 || llen != 1 + nvals * width) err = kErrCorrupt;
            lens = q + 1;
            q += llen;
        }
        if (err == kErrNone) err = read_cblock_header(q, end, dlen, kErrZstdDict);
        data = q;
        if (err != kErrNone) {
            if (lane == 0) key_err(p, err, g);
            continue;
        }
        uint32_t off_carry = 0;
        for (uint32_t base = 0; base < nvals; base += 32) {
            const uint32_t k = base + lane;
            uint32_t L = 0;
            if (k < nvals)
                for (uint32_t i = 0; i < width; ++i) L = (L << 8) | __ldg(lens + k * width + i);
            const uint32_t vlen = L > 0 ? L - 1 : 0;
            uint32_t incl = vlen;
#pragma unroll
            for (int sft = 1; sft < 32; sft <<= 1) {
                const uint32_t o = __shfl_up_sync(0xffffffffu, incl, sft);
                if (lane >= sft) incl += o;
            }
            const uint32_t off = off_carry + incl - vlen;
            off_carry += __shfl_sync(0xffffffffu, incl, 31);
            if (k < nvals) {
                if (off + vlen > dlen) key_err(p, kErrCorrupt, g);
                else key_insert(p, data + off, vlen, g);
            }
        }
    }
}

// one warp: the occupied slots, in slot order, packed into vals / lens (read back by the host: the values become the
// literals of the per-value passes and the key column of the result)
__global__ void key_pack_kernel(const __grid_constant__ KeyParams p) {
    const int lane = threadIdx.x;
    uint32_t n = 0;
    for (uint32_t s = 0; s < kKeySlots && n < p.cap; ++s) {
        const unsigned long long cur = p.slots[s];
        if (cur == 0) continue;
        const uint32_t len = static_cast<uint32_t>((cur >> 48) & 0x7fffu);
        const uint8_t *o = reinterpret_cast<const uint8_t *>(static_cast<uintptr_t>(cur & 0xffffffffffffull));
        for (uint32_t i = lane; i < len; i += 32) p.vals[static_cast<size_t>(n) * kMaxLit + i] = __ldg(o + i);
        if (lane == 0) p.lens[n] = len;
        ++n;
    }
}

void launch_key_values(const KeyParams &p, int grid, cudaStream_t s) {
    if (p.total_blocks) key_values_kernel<<<grid, 256, 0, s>>>(p);
    key_pack_kernel<<<1, 32, 0, s>>>(p);
}

// one warp per composite group (v, g): its first series and the rank of v among that series' values
__global__ void __launch_bounds__(256) key_order_kernel(const __grid_constant__ KeyOrderParams p) {
    const int lane = threadIdx.x & 31;
    const uint32_t gp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t G = static_cast<uint32_t>(p.n_groups);
    if (gp >= G * p.n_values) return;
    const uint32_t v = gp / G, g = gp % G;
    const int64_t *kts = p.Kts + static_cast<size_t>(v) * p.n_series;
    int32_t best = INT32_MAX;
    for (int32_t k = p.group_start[g] + lane; k < p.group_start[g + 1]; k += 32) {
        const int32_t i = p.order[k];
        if (kts[i] != INT64_MAX && i < best) best = i;
    }
    best = __reduce_min_sync(0xffffffffu, best);
    if (best == INT32_MAX) {
        if (lane == 0) p.first_series[gp] = -1;
        return;
    }
    const int64_t mts = kts[best];
    const uint32_t mrow = p.Krow[static_cast<size_t>(v) * p.n_series + best];
    uint32_t rank = 0;
    for (uint32_t v2 = lane; v2 < p.n_values; v2 += 32) {
        const int64_t t = p.Kts[static_cast<size_t>(v2) * p.n_series + best];
        if (t != INT64_MAX && (t < mts || (t == mts && p.Krow[static_cast<size_t>(v2) * p.n_series + best] < mrow))) ++rank;
    }
    rank = __reduce_add_sync(0xffffffffu, rank);
    if (lane == 0) {
        p.first_series[gp] = best;
        p.slot[static_cast<size_t>(best) * p.n_values + rank] = static_cast<int32_t>(gp);
    }
}

// one CTA: ordered compaction of the (series, rank) slots -> perm; the composite groups that never appeared follow
__global__ void __launch_bounds__(1024) key_perm_kernel(const __grid_constant__ KeyOrderParams p) {
    __shared__ uint32_t warp_tot[32];
    const uint32_t tid = threadIdx.x;
    const size_t n_slots = static_cast<size_t>(p.n_series) * p.n_values;
    const uint32_t n_comp = static_cast<uint32_t>(p.n_groups) * p.n_values;
    uint32_t base = 0;
    for (size_t chunk = 0; chunk < n_slots; chunk += 1024) {
        const size_t idx = chunk + tid;
        const int32_t gp = idx < n_slots ? p.slot[idx] : -1;
        uint32_t total = 0;
        const uint32_t pos = block_excl_scan(gp >= 0 ? 1u : 0u, warp_tot, total);
        if (gp >= 0) p.perm[base + pos] = gp;
        base += total;
        __syncthreads();
    }
    if (tid == 0) *p.n_present = base;
    for (uint32_t chunk = 0; chunk < n_comp; chunk += 1024) {
        const uint32_t gp = chunk + tid;
        const bool absent = gp < n_comp && p.first_series[gp] < 0;
        uint32_t total = 0;
        const uint32_t pos = block_excl_scan(absent ? 1u : 0u, warp_tot, total);
        if (absent) p.perm[base + pos] = static_cast<int32_t>(gp);
        base += total;
        __syncthreads();
    }
}

void launch_key_order(const KeyOrderParams &p, cudaStream_t s) {
    const uint32_t n_comp = static_cast<uint32_t>(p.n_groups) * p.n_values;
    if (n_comp == 0) return;
    key_order_kernel<<<(n_comp + 7) / 8, 256, 0, s>>>(p);
    key_perm_kernel<<<1, 1024, 0, s>>>(p);
}

__global__ void permute_table_kernel(TablePtrs dst, TablePtrs src, const int32_t *perm, uint32_t n_groups, uint32_t n_fcols,
                                     const int64_t *pass_coltype, uint32_t n_passes) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_fcols) {
        // column type of the query = the type any pass saw; two passes that disagree are a type mix; the worst status wins
        int64_t typ = 0, err = 0;
        for (uint32_t v = 0; v < n_passes; ++v) {
            const int64_t w = pass_coltype[static_cast<size_t>(v) * n_fcols + t];
            const int64_t wt = w & 0xff, we = w >> 8;
            if (wt != 0 && typ != 0 && wt != typ) err = err > static_cast<int64_t>(kErrTypeMix) ? err : static_cast<int64_t>(kErrTypeMix);
            if (typ == 0) typ = wt;
            err = we > err ? we : err;
        }
        dst.coltype[t] = typ | (err << 8);
    }
    if (t >= n_groups * n_fcols) return;
    const uint32_t j = t / n_fcols, c = t % n_fcols;
    const size_t so = static_cast<size_t>(perm[j]) * n_fcols + c;
    dst.sum_f64[t] = src.sum_f64[so];
    dst.max_f64[t] = src.max_f64[so];
    dst.negmin_f64[t] = src.negmin_f64[so];
    dst.sum_i64[t] = src.sum_i64[so];
    dst.cnt[t] = src.cnt[so];
    dst.max_i64[t] = src.max_i64[so];
    dst.notmin_i64[t] = src.notmin_i64[so];
    if (c == 0) dst.rows[j] = src.rows[perm[j]];
}

void launch_permute_table(const TablePtrs &dst, const TablePtrs &src, const int32_t *perm, uint32_t n_groups, uint32_t n_fcols,
                          const int64_t *pass_coltype, uint32_t n_passes, cudaStream_t s) {
    const uint32_t n = n_groups * n_fcols > n_fcols ? n_groups * n_fcols : n_fcols;
    permute_table_kernel<<<(n + 255) / 256, 256, 0, s>>>(dst, src, perm, n_groups, n_fcols, pass_coltype, n_passes);
}

// ------------------------------------------------------------------------------------------------
// Keyed collective (bydb_scan_reduce_keyed): group-by on a stored tag over the ranks' peer mailboxes.  Each rank finds ITS
// distinct values and runs its per-value passes, so rank r's value v is not rank s's value v; what travels in the slot is
// V_r, the rank's dictionary, the composite table and, per composite group, where it first showed (key_first_kernel).
// The root then
//   1. key_union_kernel: one CTA numbers the distinct values of all ranks in order of first occurrence over (rank, local id)
//      -- a deterministic global dictionary -- and writes the remap (r, v) -> global id and its inverse;
//   2. key_combine_kernel: folds the slices into one Vg x G table in rank order through the inverse (sums add, max / negmin
//      take the maximum, the column types merge like permute_table's), and merges the first appearances (lexicographic
//      minimum of (series id, Kts, Krow));
//   3. launch_key_rank: sorts the composite groups by first appearance.  One context scanning everything inserts group (v, g)
//      at (first series of g that shows v, rank of v among that series' first rows), and series ids ascend in the scan, so
//      the sort gives the same insertion order; permute_table and the ordinary finalisation run on the result unchanged.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) key_first_kernel(const __grid_constant__ KeyFirstParams p) {
    const int lane = threadIdx.x & 31;
    const uint32_t gp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t G = static_cast<uint32_t>(p.n_groups);
    if (gp == 0 && lane == 0) *p.n_values_out = p.n_values;
    if (gp >= G * p.n_values) return;
    const uint32_t v = gp / G, g = gp % G;
    const int64_t *kts = p.Kts + static_cast<size_t>(v) * p.n_series;
    int32_t best = INT32_MAX;  // the query's series ascend: the smallest index is the smallest series id
    for (int32_t k = p.group_start[g] + lane; k < p.group_start[g + 1]; k += 32) {
        const int32_t i = p.order[k];
        if (kts[i] != INT64_MAX && i < best) best = i;
    }
    best = __reduce_min_sync(0xffffffffu, best);
    if (lane != 0) return;
    if (best == INT32_MAX) {
        p.first_sid[gp] = UINT64_MAX;
        p.first_ts[gp] = INT64_MAX;
        p.first_row[gp] = UINT32_MAX;
    } else {
        p.first_sid[gp] = p.q_sids[best];
        p.first_ts[gp] = kts[best];
        p.first_row[gp] = p.Krow[static_cast<size_t>(v) * p.n_series + best];
    }
}

void launch_key_first(const KeyFirstParams &p, cudaStream_t s) {
    const uint32_t n_comp = static_cast<uint32_t>(p.n_groups) * p.n_values;
    key_first_kernel<<<n_comp ? (n_comp + 7) / 8 : 1, 256, 0, s>>>(p);
}

__global__ void __launch_bounds__(1024) key_union_kernel(const __grid_constant__ KeyUnionParams p) {
    __shared__ uint32_t warp_tot[32];
    const uint32_t n = p.n_ranks * p.cap, mask = p.hash_slots - 1;
    // 1. every (rank, value) enters an open-addressing table keyed by its bytes (FNV-1a, as key_insert); the table keeps the
    //    smallest entry index per distinct value.  rep[e] = the table slot for now.
    for (uint32_t e = threadIdx.x; e < n; e += blockDim.x) {
        const uint32_t r = e / p.cap, v = e % p.cap;
        const uint8_t *slot = p.slots + static_cast<size_t>(r) * p.slot_bytes;
        if (v >= *reinterpret_cast<const uint32_t *>(slot + p.off_nv)) {
            p.rep[e] = -1;
            continue;
        }
        const uint32_t len = reinterpret_cast<const uint32_t *>(slot + p.off_lens)[v];
        const uint8_t *b = slot + p.off_vals + static_cast<size_t>(v) * kMaxLit;
        uint64_t h = 0xcbf29ce484222325ull;
        for (uint32_t i = 0; i < len; ++i) h = (h ^ b[i]) * 0x100000001b3ull;
        uint32_t s = static_cast<uint32_t>(h ^ (h >> 32)) & mask;
        for (;;) {  // hash_slots >= 2n: a free slot always exists
            const uint32_t cur = atomicCAS(&p.hash[s], 0u, e + 1);
            if (cur == 0) break;
            const uint32_t o = cur - 1, ro = o / p.cap, vo = o % p.cap;
            const uint8_t *so = p.slots + static_cast<size_t>(ro) * p.slot_bytes;
            bool eq = reinterpret_cast<const uint32_t *>(so + p.off_lens)[vo] == len;
            const uint8_t *bo = so + p.off_vals + static_cast<size_t>(vo) * kMaxLit;
            for (uint32_t i = 0; i < len && eq; ++i) eq = bo[i] == b[i];
            if (eq) {
                atomicMin(&p.hash[s], e + 1);
                break;
            }
            s = (s + 1) & mask;
        }
        p.rep[e] = static_cast<int32_t>(s);
    }
    __syncthreads();
    // 2. the representative of an entry: the first (rank, value) with the same bytes
    for (uint32_t e = threadIdx.x; e < n; e += blockDim.x)
        if (p.rep[e] >= 0) p.rep[e] = static_cast<int32_t>(p.hash[p.rep[e]] - 1);
    __syncthreads();
    // 3. global ids: ordered compaction of the representatives over (rank, local id)
    uint32_t base = 0;
    for (uint32_t chunk = 0; chunk < n; chunk += blockDim.x) {
        const uint32_t e = chunk + threadIdx.x;
        const bool first = e < n && p.rep[e] == static_cast<int32_t>(e);
        uint32_t total = 0;
        const uint32_t pos = block_excl_scan(first ? 1u : 0u, warp_tot, total);
        if (first) {
            const uint32_t gid = base + pos, r = e / p.cap, v = e % p.cap;
            p.remap[e] = static_cast<int32_t>(gid);
            if (gid < p.cap) {
                const uint8_t *slot = p.slots + static_cast<size_t>(r) * p.slot_bytes;
                const uint32_t len = reinterpret_cast<const uint32_t *>(slot + p.off_lens)[v];
                for (uint32_t i = 0; i < len; ++i) p.g_vals[static_cast<size_t>(gid) * kMaxLit + i] = slot[p.off_vals + static_cast<size_t>(v) * kMaxLit + i];
                p.g_lens[gid] = len;
                p.inv[r * p.cap + gid] = static_cast<int32_t>(v);
            }
        }
        base += total;
        __syncthreads();
    }
    // 4. every other entry takes the id of its representative
    for (uint32_t e = threadIdx.x; e < n; e += blockDim.x) {
        const int32_t rp = p.rep[e];
        if (rp < 0 || rp == static_cast<int32_t>(e)) continue;
        const int32_t gid = p.remap[rp];
        p.remap[e] = gid;
        if (static_cast<uint32_t>(gid) < p.cap) p.inv[(e / p.cap) * p.cap + static_cast<uint32_t>(gid)] = static_cast<int32_t>(e % p.cap);
    }
    if (threadIdx.x == 0) {
        p.ctl[0] = base;
        p.ctl[1] = base > p.cap ? static_cast<uint32_t>(kErrKeyCap) : 0u;
    }
}

void launch_key_union(const KeyUnionParams &p, cudaStream_t s) { key_union_kernel<<<1, 1024, 0, s>>>(p); }

template <class T>
__device__ __forceinline__ const T *rank_ptr(const T *p0, uint32_t r, uint64_t stride) {
    return reinterpret_cast<const T *>(reinterpret_cast<const uint8_t *>(p0) + r * stride);
}

// one thread per (composite group, field) of the Vg x G table
__global__ void key_combine_kernel(const __grid_constant__ KeyCombineParams p) {
    const uint32_t F = p.n_fcols, G = static_cast<uint32_t>(p.n_groups);
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.n_values * G * F) return;
    const uint32_t j = t / F, c = t % F, vg = j / G, g = j % G;
    double sf = 0, mf = 0, nf = 0;
    int64_t si = 0, cn = 0, mi = 0, ni = 0, rows = 0;
    uint64_t fsid = UINT64_MAX;
    int64_t fts = INT64_MAX;
    uint32_t frow = UINT32_MAX;
    int64_t typ = 0, err = 0;
    bool any = false;
    for (uint32_t r = 0; r < p.n_ranks; ++r) {
        const int32_t v = p.inv[r * p.cap + vg];
        if (v < 0) continue;
        const size_t sj = static_cast<size_t>(v) * G + g, so = sj * F + c;
        const double bsf = rank_ptr(p.src.sum_f64, r, p.slot_bytes)[so], bmf = rank_ptr(p.src.max_f64, r, p.slot_bytes)[so],
                     bnf = rank_ptr(p.src.negmin_f64, r, p.slot_bytes)[so];
        const int64_t bsi = rank_ptr(p.src.sum_i64, r, p.slot_bytes)[so], bcn = rank_ptr(p.src.cnt, r, p.slot_bytes)[so],
                      bmi = rank_ptr(p.src.max_i64, r, p.slot_bytes)[so], bni = rank_ptr(p.src.notmin_i64, r, p.slot_bytes)[so];
        if (!any) {
            sf = bsf, mf = bmf, nf = bnf, si = bsi, cn = bcn, mi = bmi, ni = bni;
        } else {  // the rules of combine_tables_kernel
            sf = sf + bsf;
            mf = bmf > mf ? bmf : mf;
            nf = bnf > nf ? bnf : nf;
            si = static_cast<int64_t>(static_cast<uint64_t>(si) + static_cast<uint64_t>(bsi));  // wraps like Go's int64
            cn += bcn;
            mi = bmi > mi ? bmi : mi;
            ni = bni > ni ? bni : ni;
        }
        if (c == 0) {
            rows += rank_ptr(p.src.rows, r, p.slot_bytes)[sj];
            const uint64_t s = rank_ptr(p.src_fsid, r, p.slot_bytes)[sj];
            const int64_t ts = rank_ptr(p.src_fts, r, p.slot_bytes)[sj];
            const uint32_t row = rank_ptr(p.src_frow, r, p.slot_bytes)[sj];
            if (s < fsid || (s == fsid && (ts < fts || (ts == fts && row < frow)))) fsid = s, fts = ts, frow = row;
        }
        if (g == 0) {  // permute_table_kernel's merge of the passes' column types
            const int64_t w = rank_ptr(p.src_ct, r, p.slot_bytes)[static_cast<size_t>(v) * F + c];
            const int64_t wt = w & 0xff, we = w >> 8;
            if (wt != 0 && typ != 0 && wt != typ) err = err > static_cast<int64_t>(kErrTypeMix) ? err : static_cast<int64_t>(kErrTypeMix);
            if (typ == 0) typ = wt;
            err = we > err ? we : err;
        }
        any = true;
    }
    p.dst.sum_f64[t] = sf;
    p.dst.max_f64[t] = mf;
    p.dst.negmin_f64[t] = nf;
    p.dst.sum_i64[t] = si;
    p.dst.cnt[t] = cn;
    p.dst.max_i64[t] = mi;
    p.dst.notmin_i64[t] = ni;
    if (c == 0) {
        p.dst.rows[j] = rows;
        p.fsid[j] = fsid;
        p.fts[j] = fts;
        p.frow[j] = frow;
    }
    if (g == 0) p.dst_ct[static_cast<size_t>(vg) * F + c] = typ | (err << 8);
}

void launch_key_combine(const KeyCombineParams &p, cudaStream_t s) {
    const uint32_t n = p.n_values * static_cast<uint32_t>(p.n_groups) * p.n_fcols;
    if (n) key_combine_kernel<<<(n + 255) / 256, 256, 0, s>>>(p);
}

__global__ void iota_kernel(int32_t *out, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = static_cast<int32_t>(i);
}

struct FirstAppearanceLess {
    const uint64_t *sid;
    const int64_t *ts;
    const uint32_t *row;
    __device__ bool operator()(int32_t a, int32_t b) const {
        if (sid[a] != sid[b]) return sid[a] < sid[b];
        if (ts[a] != ts[b]) return ts[a] < ts[b];
        if (row[a] != row[b]) return row[a] < row[b];
        return a < b;
    }
};

int launch_key_rank(const uint64_t *fsid, const int64_t *fts, const uint32_t *frow, int32_t *perm, uint32_t n, void *temp, size_t *temp_bytes,
                    cudaStream_t s) {
    const FirstAppearanceLess less{fsid, fts, frow};
    if (!temp) return cub::DeviceMergeSort::SortKeys(nullptr, *temp_bytes, perm, n, less, s) == cudaSuccess ? 0 : -1;
    if (n == 0) return 0;
    iota_kernel<<<(n + 255) / 256, 256, 0, s>>>(perm, n);
    return cub::DeviceMergeSort::SortKeys(temp, *temp_bytes, perm, n, less, s) == cudaSuccess ? 0 : -1;
}

void launch_plan_blocks(const ScanParams &p, cudaStream_t s) {
    if (p.total_blocks == 0) return;
    const int threads = 256;
    plan_blocks_kernel<<<(p.total_blocks + threads - 1) / threads, threads, 0, s>>>(p);
}

// cudaFuncSetAttribute applies to the CURRENT device: one flag per device ordinal (several contexts, one per GPU, may
// live in one process), atomics because every entry point is thread-safe
static std::atomic<bool> g_attr_set[64];
static void scan_set_attrs() {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && g_attr_set[dev].load(std::memory_order_acquire)) return;
    const int smem = static_cast<int>(scan_smem_bytes());
    cudaFuncSetAttribute(scan_blocks_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(scan_blocks_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(scan_sum_express_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(dedup_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (dev >= 0 && dev < 64) g_attr_set[dev].store(true, std::memory_order_release);
}
// fast lane over the planned blocks, then the slow lane over whatever the fast lane deferred
void launch_scan_blocks(const ScanParams &p, int grid_fast, int grid_slow, cudaStream_t s) {
    scan_set_attrs();
    const size_t smem = scan_smem_bytes();
    if (p.rest_list) scan_sum_express_kernel<<<grid_fast, kWarpsPerCta * 32, smem, s>>>(p);
    scan_blocks_kernel<true><<<grid_fast, kWarpsPerCta * 32, smem, s>>>(p);
    scan_blocks_kernel<false><<<grid_slow, kWarpsPerCta * 32, smem, s>>>(p);
}

void scan_max_ctas_per_sm(int *fast, int *slow) {
    scan_set_attrs();
    int a = 1, b = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, scan_blocks_kernel<true>, kWarpsPerCta * 32, scan_smem_bytes());
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, scan_blocks_kernel<false>, kWarpsPerCta * 32, scan_smem_bytes());
    *fast = a < 1 ? 1 : a;
    *slow = b < 1 ? 1 : b;
}

void launch_detect_overlap(const ScanParams &p, cudaStream_t s) {
    if (p.n_series == 0) return;
    const int threads = 128;
    detect_overlap_kernel<<<(p.n_series + threads - 1) / threads, threads, 0, s>>>(p);
}
void launch_dedup(const ScanParams &p, int grid, cudaStream_t s) {
    if (p.n_dd_blocks == 0) return;
    const size_t smem = scan_smem_bytes();
    scan_set_attrs();
    dedup_kernel<<<grid, kWarpsPerCta * 32, smem, s>>>(p, 0);
    dedup_kernel<<<grid, kWarpsPerCta * 32, smem, s>>>(p, 1);
}
void launch_series_reduce(const ReduceParams &p, cudaStream_t s) {
    if (p.n_series == 0) return;
    const int threads = 256;  // 8 series (one warp each) per CTA
    series_reduce_kernel<<<(p.n_series + 7) / 8, threads, 0, s>>>(p);
}
void launch_group_reduce(const ReduceParams &p, cudaStream_t s, bool small_groups) {
    if (p.n_groups <= 0) return;
    if (small_groups) group_reduce_small_kernel<<<(p.n_groups + 7) / 8, 256, 0, s>>>(p);
    else group_reduce_kernel<<<p.n_groups, 256, 0, s>>>(p);
}
void launch_combine_tables(uint64_t *tables, uint32_t n_tables, uint64_t words, uint64_t sum_f64_lo, uint64_t sum_f64_hi, uint64_t max_f64_lo,
                           uint64_t max_f64_hi, uint64_t sum_i64_lo, uint64_t sum_i64_hi, uint64_t max_i64_lo, uint64_t max_i64_hi, cudaStream_t s,
                           uint64_t stride_words) {
    if (words == 0 || n_tables < 2) return;
    combine_tables_kernel<<<static_cast<unsigned>((words + 255) / 256), 256, 0, s>>>(tables, n_tables, words, stride_words ? stride_words : words, sum_f64_lo,
                                                                                  sum_f64_hi, max_f64_lo, max_f64_hi, sum_i64_lo, sum_i64_hi, max_i64_lo,
                                                                                  max_i64_hi);
}

// ------------------------------------------------------------------------------------------------
// Multi-GPU reduce without a library collective (SURVEY.md 8e; the liaison reduce of
// pkg/query/logical/measure/measure_plan_aggregation.go:96-124 done by the GPUs themselves): every rank's group_reduce
// writes its partial table straight into ITS slot of the root's mailbox -- peer memory, the stores travel over
// NVLink / NVSwitch -- and then raises its arrival flag there; the root spins on the flags, combines the slots in rank
// order and finalises.  Flags carry the call's epoch (all ranks issue the collective calls in the same order), slots
// alternate between two parities, and a writer first waits until the root has consumed the slot's previous use.
// All waits are bounded: a peer that never arrives becomes an error code, never a hung GPU.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// one warp: lane r waits for word r of `flags` (stride in words) to reach `epoch`
__global__ void comm_wait_kernel(const unsigned long long *flags, uint32_t n, unsigned long long epoch, uint32_t *err, uint32_t err_code) {
    const uint32_t r = threadIdx.x;
    bool ok = true;
    if (r < n) {
        ok = false;
        // bounded by wall time: a peer's first call may spend seconds loading its kernels onto a fresh device
        unsigned long long t0, t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for (uint32_t spins = 0;; ++spins) {
            if (ld_acquire_sys(flags + r) >= epoch) {
                ok = true;
                break;
            }
            __nanosleep(spins < 1024 ? 32 : 1000);
            if ((spins & 1023u) == 1023u) {
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if (t1 - t0 > 60ull * 1000000000ull) break;  // 60 s
            }
        }
    }
    if (!ok && err) atomicCAS(err, 0u, err_code);
}
__global__ void comm_signal_kernel(unsigned long long *flag, unsigned long long epoch) {
    __threadfence_system();  // the table stores of the kernels before this one are visible system-wide first
    st_release_sys(flag, epoch);
}
// The same three steps with the epoch read from DEVICE memory: a captured CUDA graph bakes its kernel arguments in, so a
// replayed collective gets its epoch (and the epoch its slots were last used) from a CommArgs block that a memcpy node at the
// head of the graph refreshes from pinned host memory before every launch.
__global__ void comm_wait_args_kernel(const unsigned long long *flags, uint32_t n, const CommArgs *a, int which, uint32_t *err, uint32_t err_code) {
    const unsigned long long thr = which ? a->prev_use : a->epoch;
    if (thr == 0) return;  // nothing to wait for (the slots were never used before)
    const uint32_t r = threadIdx.x;
    bool ok = true;
    if (r < n) {
        ok = false;
        unsigned long long t0, t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for (uint32_t spins = 0;; ++spins) {
            if (ld_acquire_sys(flags + r) >= thr) {
                ok = true;
                break;
            }
            __nanosleep(spins < 1024 ? 32 : 1000);
            if ((spins & 1023u) == 1023u) {
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if (t1 - t0 > 60ull * 1000000000ull) break;
            }
        }
    }
    if (!ok && err) atomicCAS(err, 0u, err_code);
}
__global__ void comm_signal_args_kernel(unsigned long long *flag, unsigned long long *status, const CommArgs *a) {
    *status = a->epoch << 32;  // no host-side failure can happen inside a replayed graph
    __threadfence_system();
    st_release_sys(flag, a->epoch);
}
__global__ void comm_done_args_kernel(unsigned long long *done, const CommArgs *a) { st_release_sys(done, a->epoch); }
void launch_comm_wait_args(const unsigned long long *flags, uint32_t n, const CommArgs *a, int which, uint32_t *err, uint32_t err_code, cudaStream_t s) {
    comm_wait_args_kernel<<<1, 32, 0, s>>>(flags, n, a, which, err, err_code);
}
void launch_comm_signal_args(unsigned long long *flag, unsigned long long *status, const CommArgs *a, cudaStream_t s) {
    comm_signal_args_kernel<<<1, 1, 0, s>>>(flag, status, a);
}
void launch_comm_done_args(unsigned long long *done, const CommArgs *a, cudaStream_t s) { comm_done_args_kernel<<<1, 1, 0, s>>>(done, a); }

void launch_comm_wait(const unsigned long long *flags, uint32_t n, unsigned long long epoch, uint32_t *err, uint32_t err_code, cudaStream_t s) {
    comm_wait_kernel<<<1, 32, 0, s>>>(flags, n, epoch, err, err_code);
}
void launch_comm_signal(unsigned long long *flag, unsigned long long epoch, cudaStream_t s) { comm_signal_kernel<<<1, 1, 0, s>>>(flag, epoch); }
void launch_select_rows(const SelectParams &p, cudaStream_t s) {
    FinalizeParams none;
    memset(&none, 0, sizeof none);
    select_rows_kernel<false><<<1, 1024, 0, s>>>(p, none);
}
// finalisation + row selection: one launch for up to kFusedFinalizeGroups groups, two beyond
uint32_t launch_finalize_select(const FinalizeParams &fp, const SelectParams &p, cudaStream_t s) {
    if (fp.n_groups <= kFusedFinalizeGroups) {
        select_rows_kernel<true><<<1, 1024, 0, s>>>(p, fp);
        return 1;
    }
    launch_finalize(fp, s);
    launch_select_rows(p, s);
    return 2;
}
void launch_finalize(const FinalizeParams &p, cudaStream_t s) {
    const int threads = 128;
    const int n = p.n_groups > 0 ? p.n_groups : 1;
    finalize_kernel<<<(n + threads - 1) / threads, threads, 0, s>>>(p);
}

// With lazy module loading the first launch of a kernel loads its code, and that may wait for the device to go idle.  A
// collective's wait kernel spins until its peers arrive -- if a peer shares the device (tests, several contexts per GPU) and
// its first-ever launch of some kernel lands behind that spin, both wait for each other until the bounded wait gives up.
// bydb_init therefore touches every kernel of the library once on its device.
void preload_kernels() {
    cudaFuncAttributes ka;
    (void)cudaFuncGetAttributes(&ka, key_values_kernel);
    (void)cudaFuncGetAttributes(&ka, key_pack_kernel);
    (void)cudaFuncGetAttributes(&ka, key_order_kernel);
    (void)cudaFuncGetAttributes(&ka, key_perm_kernel);
    (void)cudaFuncGetAttributes(&ka, permute_table_kernel);
    (void)cudaFuncGetAttributes(&ka, key_first_kernel);
    (void)cudaFuncGetAttributes(&ka, key_union_kernel);
    (void)cudaFuncGetAttributes(&ka, key_combine_kernel);
    (void)cudaFuncGetAttributes(&ka, iota_kernel);
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, plan_blocks_kernel);
    cudaFuncGetAttributes(&a, scan_blocks_kernel<true>);
    cudaFuncGetAttributes(&a, scan_blocks_kernel<false>);
    cudaFuncGetAttributes(&a, scan_sum_express_kernel);
    cudaFuncGetAttributes(&a, detect_overlap_kernel);
    cudaFuncGetAttributes(&a, dedup_kernel);
    cudaFuncGetAttributes(&a, series_reduce_kernel);
    cudaFuncGetAttributes(&a, group_reduce_kernel);
    cudaFuncGetAttributes(&a, group_reduce_small_kernel);
    cudaFuncGetAttributes(&a, finalize_kernel);
    cudaFuncGetAttributes(&a, select_rows_kernel<true>);
    cudaFuncGetAttributes(&a, select_rows_kernel<false>);
    cudaFuncGetAttributes(&a, combine_tables_kernel);
    cudaFuncGetAttributes(&a, comm_wait_kernel);
    cudaFuncGetAttributes(&a, comm_signal_kernel);
    cudaFuncGetAttributes(&a, comm_wait_args_kernel);
    cudaFuncGetAttributes(&a, comm_signal_args_kernel);
    cudaFuncGetAttributes(&a, comm_done_args_kernel);
    cudaGetLastError();
}

// Go math.Pow10 (src/math/pow10.go): pow10postab32[n/32] * pow10tab[n%32].  The product is done
// on the host in IEEE double (no FMA: a single multiply), exactly like the Go runtime.
int upload_pow10_table() {
    static const double tab[32] = {1e00, 1e01, 1e02, 1e03, 1e04, 1e05, 1e06, 1e07, 1e08, 1e09, 1e10,
                                   1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21,
                                   1e22, 1e23, 1e24, 1e25, 1e26, 1e27, 1e28, 1e29, 1e30, 1e31};
    static const double postab32[10] = {1e00, 1e32, 1e64, 1e96, 1e128, 1e160, 1e192, 1e224, 1e256, 1e288};
    double h[309];
    for (int n = 0; n <= 308; ++n) {
        volatile double a = postab32[n / 32], b = tab[n % 32];
        volatile double r = a * b;
        h[n] = r;
    }
    return cudaMemcpyToSymbol(c_pow10, h, sizeof(h)) == cudaSuccess ? 0 : -1;
}

}  // namespace bydb
