// api.cu — host side of libaurora_cuda.so: context, per-device queues and buffers, stream sharding and the
// C ABI declared in include/aurora_cuda.h.  No CPU codec lives here: every Decompress/Compress goes to
// the sm_100a kernels (decode_flaglz.cu, decode_bytelz.cu, encode_lz.cu) and fails with AURORA_CUDA_ERROR
// when no device is usable.
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "api_internal.hpp"
#include "common.cuh"

using namespace aurora;

namespace {

// NVTX ranges of the host scheduler (SURVEY.md §5 "tracing"): one range per device shard and, inside it, one per pipeline
// piece (the enqueue of its H2D copy, kernel and D2H copies) and one for the final wait.  Header-only NVTX v3: no link
// dependency, a no-op unless a profiler injects itself.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    NvtxRange(const char* what, int a, size_t b) {
        char buf[96];
        std::snprintf(buf, sizeof buf, "%s dev %d n %zu", what, a, b);
        nvtxRangePushA(buf);
    }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};


struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = n + n / 8 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

struct HostBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        size_t want = n + n / 8 + 4096;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

struct DeviceCtx {
    int dev = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t s_in = nullptr, s_out = nullptr;   // copy engines of the pipelined host path
    std::vector<cudaEvent_t> ev_in, ev_k;
    DevBuf src, dst, desc, ticket, scratch, order;
    HostBuf hdesc;
    std::mutex mu;   // one batch at a time per device
};

}  // namespace

struct aurora_ctx {
    std::vector<DeviceCtx*> devs;
    std::string last_error;
    std::atomic<uint64_t> launches{0};
    std::mutex err_mu;
    void set_error(const std::string& s) {
        std::lock_guard<std::mutex> g(err_mu);
        last_error = s;
    }
};

namespace {

thread_local std::string g_init_error;

#define CU_TRY(ctx, expr)                                                                           \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            (ctx)->set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                   \
            return AURORA_CUDA_ERROR;                                                               \
        }                                                                                           \
    } while (0)

bool is_flaglz(int f) {
    return f == AURORA_FMT_YAZ0 || f == AURORA_FMT_YAZ1 || f == AURORA_FMT_YAY0 || f == AURORA_FMT_MIO0 ||
           f == AURORA_FMT_LZ10 || f == AURORA_FMT_LZ11 || f == AURORA_FMT_LZSS || f == AURORA_FMT_LZHUDSON ||
           f == AURORA_FMT_LZ40 || f == AURORA_FMT_LZ60 || f == AURORA_FMT_SMSR00;
}
bool is_bytelz(int f) {
    return f == AURORA_FMT_LZ4 || f == AURORA_FMT_LZ4_BLOCK || f == AURORA_FMT_LZ4_LEGACY || f == AURORA_FMT_LZO ||
           f == AURORA_FMT_SNAPPY || f == AURORA_FMT_SNAPPY_BLOCK || f == AURORA_FMT_PRS;
}

int ceil_log2(long long x) {
    int b = 0;
    while ((1LL << b) < x) b++;
    return b;
}

// resolve the option block into kernel parameters; returns a per-batch status override (OK = run)
int fill_decode_params(DecodeParams& p, int format, const aurora_codec_opts* o) {
    p.format = format;
    p.byte_order = o ? o->byte_order : AURORA_ENDIAN_DEFAULT;
    if (p.byte_order != AURORA_ENDIAN_LITTLE && p.byte_order != AURORA_ENDIAN_BIG) p.byte_order = AURORA_ENDIAN_DEFAULT;
    p.size_only = 0;
    p.lz4_verify = o ? o->lz4_verify : 0;
    aurora_lz_props lz;
    if (o && o->lzss.windows_bits != 0) lz = o->lzss;
    else aurora_lz_props_bits(&lz, 12, 4, 2);   // LZSS.DefaultProperties (LZSS.cs:33)
    p.lzss = LzssParams{lz.windows_bits, lz.length_bits, lz.min_length, lz.max_distance, lz.windows_start,
                        o ? o->lzss_initial_fill : 0};
    if (format == AURORA_FMT_LZSS) {
        if (lz.windows_bits < 1 || lz.windows_bits > 12 || lz.length_bits < 1 || lz.length_bits > 8 || lz.max_distance < 2 ||
            lz.max_distance > 4096 || lz.min_length < 1 || lz.min_length > 255)
            return AURORA_NOT_SUPPORTED;
    }
    return AURORA_OK;
}

cudaError_t launch_encode(const EncodeParams& p, int warps, cudaStream_t st) {
    // Flag-byte formats (LZ10 / BLZ, LZ11 / LZ40 / LZ60, Yaz0 / Yaz1, LZSS, MIO0, Yay0, LZHudson, SMSR00): the window search with one lane per
    // position and shared-memory tables (encode_lz_par.cu).  Both encoders write the reference's bytes; which one runs is a
    // speed decision.  Measured on the C2 corpus (64 KiB streams, GB/s raw in, parallel / sequential replay): quality 8 LZ10
    // 14.6 / 8.1, Yaz0 16.1 / 10.4, MIO0 12.6 / 6.5, Yay0 13.3 / 6.4, LZ11 10.8 / 5.9; quality 10-12 LZ10 5.3 / 4.3, LZ11
    // 5.1 / 4.3; quality 15 LZ10 5.1 / 4.2 but LZ11 1.7 / 2.4 — with matches longer than a few words and chains of 256+
    // candidates every lane walks its whole chain, and the warp-cooperative comparison of the sequential replay wins.
    // Default: parallel, except long-match formats from quality 13 on; either can be forced (opts.strategy bits 16 / 17,
    // AURORA_ENCODER).
    static const int forced = [] {
        const char* e = std::getenv("AURORA_ENCODER");
        return !e ? 0 : std::strcmp(e, "serial") == 0 ? 2 : std::strcmp(e, "parallel") == 0 ? 1 : 0;
    }();
    const int want = p.finder_choice ? p.finder_choice : forced;
    const bool par_default = p.max_chain <= 128 || p.max_length <= 32;
    if (encode_lz_par_supported(p) && (want == 1 || (want == 0 && par_default))) return launch_encode_lz_par(p, warps / 48, st);
    if (is_flaglz(p.format) || p.format == AURORA_FMT_BLZ) return launch_encode_lz(p, warps, st);   // BLZ: LZ10's layout
    return launch_encode_bytelz(p, warps, st);
}

cudaError_t launch_decode(const DecodeParams& p, int sm_count, cudaStream_t st) {
    if (p.format == AURORA_FMT_BLZ) return launch_decode_blz(p, sm_count, st);
    if (is_flaglz(p.format)) return launch_decode_flaglz(p, sm_count, st);
    return launch_decode_bytelz(p, sm_count, st);
}

struct Range {
    size_t begin, end;
};

// contiguous ranges of streams with balanced byte counts (streams are independent: SURVEY.md §8e).
// doff (optional): destination offsets — neighbours whose destination windows [doff, doff + b) overlap (the chunks of one
// ChunkLZ10 file) are never cut apart: every device copies its own destination span back to the host, so overlapping
// windows on two devices would let one device's copy overwrite bytes the other one decoded.
std::vector<Range> shard(size_t n, int g, const uint64_t* a, const uint64_t* b, const uint64_t* doff = nullptr) {
    std::vector<Range> r;
    if (g <= 1 || n < size_t(g) * 2) {
        r.push_back(Range{0, n});
        return r;
    }
    long double total = 0;
    for (size_t i = 0; i < n; i++) total += (long double)(a[i] + (b ? b[i] : 0) + 64);
    size_t i = 0;
    long double acc = 0;
    for (int k = 0; k < g; k++) {
        size_t start = i;
        long double target = total * (k + 1) / g;
        while (i < n && (acc < target || k == g - 1)) {
            acc += (long double)(a[i] + (b ? b[i] : 0) + 64);
            i++;
        }
        while (doff && b && i < n && i > start && doff[i] < doff[i - 1] + b[i - 1]) {
            acc += (long double)(a[i] + b[i] + 64);
            i++;
        }
        r.push_back(Range{start, i});
    }
    r.back().end = n;
    return r;
}

inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) & ~(a - 1); }

// Layout of one shard's source or destination bytes on the device: either the host span copied as one
// piece (offsets keep their value relative to the 16-byte aligned span start) or a packed re-layout.
struct Layout {
    bool span = true;
    uint64_t lo = 0;        // host offset of device byte 0 (span mode)
    uint64_t bytes = 0;     // device bytes
    std::vector<uint64_t> dev_off;
};

Layout plan_layout(const uint64_t* off, const uint64_t* len, size_t b, size_t e) {
    Layout L;
    uint64_t lo = ~0ull, hi = 0, sum = 0;
    for (size_t i = b; i < e; i++) {
        lo = std::min(lo, off[i]);
        hi = std::max(hi, off[i] + len[i]);
        sum += len[i];
    }
    if (b == e) { lo = hi = 0; }
    lo &= ~15ull;
    L.dev_off.resize(e - b);
    if (hi - lo <= sum + sum / 4 + (1u << 20) + 64 * (e - b)) {
        L.span = true;
        L.lo = lo;
        L.bytes = align_up(hi - lo, 16);
        for (size_t i = b; i < e; i++) L.dev_off[i - b] = off[i] - lo;
    } else {
        L.span = false;
        uint64_t pos = 0;
        for (size_t i = b; i < e; i++) {
            L.dev_off[i - b] = pos;
            pos += align_up(len[i], 16);
        }
        L.bytes = pos;
    }
    return L;
}


// Device -> host copy of the destination windows [off[i], off[i] + ext(i)) of streams [i0, i1) in span mode.  Windows that
// follow each other in ascending order with a gap of at most `gap_tol` bytes (the alignment padding of a packed batch)
// travel as one copy; anything else starts a new copy, and no copy starts before the first window of its run.  With
// gap_tol = 0 only the windows themselves are written (the wrapper formats run several sub-batches over one destination).
template <typename Ext>
cudaError_t copy_back_windows(uint8_t* dst_base, const uint8_t* ddst, uint64_t dev_lo, const uint64_t* off, size_t i0, size_t i1, Ext ext,
                              uint64_t gap_tol, cudaStream_t st) {
    size_t i = i0;
    while (i < i1) {
        uint64_t lo = off[i], hi = off[i] + ext(i), prev = off[i];
        size_t j = i + 1;
        while (j < i1 && off[j] >= prev && off[j] <= hi + gap_tol) {
            hi = std::max(hi, off[j] + ext(j));
            prev = off[j];
            j++;
        }
        if (hi > lo) {
            cudaError_t e = cudaMemcpyAsync(dst_base + lo, ddst + (lo - dev_lo), hi - lo, cudaMemcpyDeviceToHost, st);
            if (e != cudaSuccess) return e;
        }
        i = j;
    }
    return cudaSuccess;
}

int decode_shard(aurora_ctx* ctx, DeviceCtx* d, int format, const aurora_codec_opts* opts, size_t b, size_t e,
                 const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base,
                 const uint64_t* dst_off, const uint64_t* dst_cap, uint64_t* out_len, uint64_t* consumed, int32_t* status,
                 int size_only, const uint64_t* raw_size = nullptr, const uint32_t* xor_key = nullptr, bool exact = false) {
    NvtxRange nvtx_shard("aurora decode shard", d->dev, e - b);
    const size_t n = e - b;
    if (n == 0) return AURORA_OK;
    // exact (the sub-batches of the wrapper formats): only the bytes a stream produced are written to the host.  Otherwise the
    // whole capacity windows come back, and windows at most 15 bytes apart (alignment padding) travel as one copy.
    const uint64_t gap_tol = exact ? 0 : 15;
    std::lock_guard<std::mutex> guard(d->mu);
    CU_TRY(ctx, cudaSetDevice(d->dev));
    DecodeParams P{};
    const int override_status = fill_decode_params(P, format, opts);
    if (override_status != AURORA_OK) {
        for (size_t i = b; i < e; i++) {
            status[i] = override_status;
            if (out_len) out_len[i] = 0;
            if (consumed) consumed[i] = 0;
        }
        return AURORA_OK;
    }
    P.size_only = size_only;
    P.headerless = raw_size != nullptr;
    const Layout S = plan_layout(src_off, src_len, b, e);
    Layout D;
    if (!size_only) D = plan_layout(dst_off, dst_cap, b, e);
    else D.dev_off.assign(n, 0);

    CU_TRY(ctx, d->src.reserve(S.bytes + 16));
    CU_TRY(ctx, d->dst.reserve(D.bytes + 16));
    // descriptors: src_off, src_len, dst_off, dst_cap | out_len, consumed | status
    // (+ LZ00: one keystream key per stream behind the status array)
    const size_t desc_bytes = n * (6 * sizeof(uint64_t) + 2 * sizeof(int32_t)) + 64;
    CU_TRY(ctx, d->desc.reserve(desc_bytes));
    CU_TRY(ctx, d->hdesc.reserve(desc_bytes));
    CU_TRY(ctx, d->ticket.reserve(256));
    uint64_t* h = static_cast<uint64_t*>(d->hdesc.p);
    uint64_t* dv = static_cast<uint64_t*>(d->desc.p);
    uint32_t* dkey = reinterpret_cast<uint32_t*>(dv + 6 * n) + n;
    if (xor_key) std::memcpy(reinterpret_cast<uint32_t*>(h + 6 * n) + n, xor_key + b, n * sizeof(uint32_t));
    for (size_t i = 0; i < n; i++) {
        h[i] = S.dev_off[i];
        h[n + i] = src_len[b + i];
        h[2 * n + i] = D.dev_off[i];
        h[3 * n + i] = size_only ? 0 : dst_cap[b + i];
        // headerless bodies: the decoded size travels in the upper half of the capacity word (DecodeParams::headerless)
        if (raw_size) h[3 * n + i] = (raw_size[b + i] << 32) | std::min<uint64_t>(dst_cap[b + i], 0xFFFFFFFFull);
    }
    cudaStream_t st = d->stream;
    CU_TRY(ctx, cudaMemcpyAsync(dv, h, 4 * n * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    if (xor_key) CU_TRY(ctx, cudaMemcpyAsync(dkey, reinterpret_cast<uint32_t*>(h + 6 * n) + n, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    uint8_t* dsrc = static_cast<uint8_t*>(d->src.p);
    uint8_t* ddst = static_cast<uint8_t*>(d->dst.p);
    P.src_base = dsrc;
    P.src_limit = align_up(S.bytes, 16);
    P.dst_base = ddst;
    P.order = nullptr;
    P.ticket = static_cast<unsigned int*>(d->ticket.p);
    // wide size spread (max > 2 x mean): hand streams to warps largest first to cut the tail
    bool balance = false;
    if (!size_only && n >= 64 && !(opts && opts->balance == 2)) {
        uint64_t mx = 0, sum = 0;
        for (size_t i = b; i < e; i++) {
            mx = std::max(mx, dst_cap[i]);
            sum += dst_cap[i];
        }
        balance = mx > 2 * (sum / n + 1);
    }
    if (balance) CU_TRY(ctx, d->order.reserve(n * sizeof(uint32_t) + 256));

    // Pipelined host path: the shard is cut into byte-balanced pieces; piece k+1 is uploaded (H2D engine) while piece
    // k decodes and piece k-1 is downloaded (D2H engine), so end-to-end time tends to max(H2D, D2H) instead of their sum.
    uint64_t total_bytes = S.bytes + D.bytes;
    size_t pieces = 1;
    // (not with a keystream pass: piece k+1's upload starts at a 16-byte boundary and may rewrite the tail of piece k's
    //  last stream, harmless only as long as the device copy still equals the host bytes)
    if (S.span && (size_only || D.span) && total_bytes > (64ull << 20) && n >= 64 && !xor_key && !exact) {
        // one piece per 128 MiB, at most 32 (measured on C2 with the short first pieces below: 16 / 24 / 32 / 48 pieces =
        // 48.7 / 49.0 / 49.2 / 48.9 GB/s end to end)
        size_t max_pieces = 32;
        const int shift = 27;
        if (const char* e = std::getenv("AURORA_MAX_PIECES")) max_pieces = std::min<size_t>(48, std::max<size_t>(2, size_t(std::atoi(e))));   // developer knob
        pieces = std::min<size_t>(max_pieces, std::max<size_t>(2, total_bytes >> shift));
    }
    if (pieces > 1) {
        while (d->ev_in.size() < pieces) {
            cudaEvent_t e1, e2;
            CU_TRY(ctx, cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
            CU_TRY(ctx, cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
            d->ev_in.push_back(e1);
            d->ev_k.push_back(e2);
        }
        CU_TRY(ctx, cudaMemsetAsync(d->ticket.p, 0, 256, st));
        CU_TRY(ctx, cudaEventRecord(d->ev_k[0], st));   // descriptors + tickets are in place
        CU_TRY(ctx, cudaStreamWaitEvent(d->s_in, d->ev_k[0], 0));
        // piece boundaries by cumulative bytes.  The first regular piece is cut in three (1/8, 3/8, 1/2 of it): the download
        // engine is the bottleneck of the pipeline and idles until the first kernel has finished, so the first upload is short.
        std::vector<uint64_t> bound;
        bound.push_back(total_bytes / (8 * pieces));
        bound.push_back(total_bytes / (2 * pieces));
        for (size_t k = 1; k < pieces; k++) bound.push_back(total_bytes * k / pieces);
        pieces = bound.size() + 1;
        while (d->ev_in.size() < pieces) {
            cudaEvent_t e1, e2;
            CU_TRY(ctx, cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
            CU_TRY(ctx, cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
            d->ev_in.push_back(e1);
            d->ev_k.push_back(e2);
        }
        std::vector<size_t> cut(pieces + 1, n);
        cut[0] = 0;
        {
            uint64_t acc = 0;
            size_t k = 1;
            for (size_t i = 0; i < n && k < pieces; i++) {
                acc += src_len[b + i] + (size_only ? 0 : dst_cap[b + i]);
                while (k < pieces && acc >= bound[k - 1]) cut[k++] = i + 1;
            }
        }
        for (size_t k = 0; k < pieces; k++) {
            const size_t i0 = cut[k], i1 = cut[k + 1];
            if (i1 <= i0) continue;
            NvtxRange nvtx_piece("decode piece: H2D + kernel + D2H enqueue", int(k), i1 - i0);
            uint64_t lo = ~0ull, hi = 0;
            for (size_t i = i0; i < i1; i++) {
                lo = std::min(lo, src_off[b + i]);
                hi = std::max(hi, src_off[b + i] + src_len[b + i]);
            }
            lo &= ~15ull;
            if (hi > lo) CU_TRY(ctx, cudaMemcpyAsync(dsrc + (lo - S.lo), src_base + lo, hi - lo, cudaMemcpyHostToDevice, d->s_in));
            CU_TRY(ctx, cudaEventRecord(d->ev_in[k], d->s_in));
            CU_TRY(ctx, cudaStreamWaitEvent(st, d->ev_in[k], 0));
            DecodeParams Q = P;
            Q.src_off = dv + i0;
            Q.src_len = dv + n + i0;
            Q.dst_off = dv + 2 * n + i0;
            Q.dst_cap = dv + 3 * n + i0;
            Q.out_len = dv + 4 * n + i0;
            Q.consumed = dv + 5 * n + i0;
            Q.status = reinterpret_cast<int32_t*>(dv + 6 * n) + i0;
            Q.ticket = static_cast<unsigned int*>(d->ticket.p) + k;
            Q.n = uint32_t(i1 - i0);
            if (balance) {
                uint32_t* hist = static_cast<uint32_t*>(d->order.p);
                uint32_t* ord = hist + 64 + i0;
                CU_TRY(ctx, launch_size_order(Q.dst_cap, Q.n, hist, ord, st));
                ctx->launches += 3;
                Q.order = ord;
            }
            if (xor_key) {   // LZ00: lift the keystream off this piece's bodies (device copy, in place)
                CU_TRY(ctx, launch_lcg_xor(dsrc, Q.src_off, Q.src_len, nullptr, dkey + i0, 0, Q.n, st));
                ctx->launches++;
            }
            CU_TRY(ctx, launch_decode(Q, d->sm_count, st));
            ctx->launches++;
            if (!size_only) {
                CU_TRY(ctx, cudaEventRecord(d->ev_k[k], st));
                CU_TRY(ctx, cudaStreamWaitEvent(d->s_out, d->ev_k[k], 0));
                CU_TRY(ctx, copy_back_windows(dst_base, ddst, D.lo, dst_off, b + i0, b + i1, [&](size_t i) { return dst_cap[i]; }, gap_tol, d->s_out));
            }
        }
        CU_TRY(ctx, cudaMemcpyAsync(h + 4 * n, dv + 4 * n, 2 * n * sizeof(uint64_t) + n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        NvtxRange nvtx_wait("decode shard: wait for the pipeline");
        CU_TRY(ctx, cudaStreamSynchronize(st));
        CU_TRY(ctx, cudaStreamSynchronize(d->s_out));
    } else {
        if (S.span) {
            uint64_t hi = 0;
            for (size_t i = b; i < e; i++) hi = std::max(hi, src_off[i] + src_len[i]);
            if (hi > S.lo) CU_TRY(ctx, cudaMemcpyAsync(dsrc, src_base + S.lo, hi - S.lo, cudaMemcpyHostToDevice, st));
        } else {
            for (size_t i = b; i < e; i++)
                if (src_len[i]) CU_TRY(ctx, cudaMemcpyAsync(dsrc + S.dev_off[i - b], src_base + src_off[i], src_len[i], cudaMemcpyHostToDevice, st));
        }
        CU_TRY(ctx, cudaMemsetAsync(d->ticket.p, 0, 64, st));
        P.src_off = dv;
        P.src_len = dv + n;
        P.dst_off = dv + 2 * n;
        P.dst_cap = dv + 3 * n;
        P.out_len = dv + 4 * n;
        P.consumed = dv + 5 * n;
        P.status = reinterpret_cast<int32_t*>(dv + 6 * n);
        P.n = uint32_t(n);
        if (balance) {
            uint32_t* hist = static_cast<uint32_t*>(d->order.p);
            CU_TRY(ctx, launch_size_order(P.dst_cap, P.n, hist, hist + 64, st));
            ctx->launches += 3;
            P.order = hist + 64;
        }
        if (xor_key) {   // LZ00: lift the keystream off the bodies (device copy, in place)
            CU_TRY(ctx, launch_lcg_xor(dsrc, P.src_off, P.src_len, nullptr, dkey, 0, P.n, st));
            ctx->launches++;
        }
        CU_TRY(ctx, launch_decode(P, d->sm_count, st));
        ctx->launches++;
        CU_TRY(ctx, cudaMemcpyAsync(h + 4 * n, dv + 4 * n, 2 * n * sizeof(uint64_t) + n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        if (!size_only) {
            if (D.span && exact) {
                CU_TRY(ctx, cudaStreamSynchronize(st));   // out_len is on the host
                CU_TRY(ctx, copy_back_windows(dst_base, ddst, D.lo, dst_off, b, e,
                                              [&](size_t i) { return std::min<uint64_t>(h[4 * n + (i - b)], dst_cap[i]); }, 0, st));
                CU_TRY(ctx, cudaStreamSynchronize(st));
            } else if (D.span) {
                CU_TRY(ctx, copy_back_windows(dst_base, ddst, D.lo, dst_off, b, e, [&](size_t i) { return dst_cap[i]; }, gap_tol, st));
                CU_TRY(ctx, cudaStreamSynchronize(st));
            } else {
                CU_TRY(ctx, cudaStreamSynchronize(st));
                for (size_t i = b; i < e; i++) {
                    const uint64_t nbytes = std::min<uint64_t>(h[4 * n + (i - b)], dst_cap[i]);
                    if (nbytes) CU_TRY(ctx, cudaMemcpyAsync(dst_base + dst_off[i], ddst + D.dev_off[i - b], nbytes, cudaMemcpyDeviceToHost, st));
                }
                CU_TRY(ctx, cudaStreamSynchronize(st));
            }
        } else {
            CU_TRY(ctx, cudaStreamSynchronize(st));
        }
    }
    const int32_t* hs = reinterpret_cast<const int32_t*>(h + 6 * n);
    for (size_t i = 0; i < n; i++) {
        if (out_len) out_len[b + i] = h[4 * n + i];
        if (consumed) consumed[b + i] = h[5 * n + i];
        if (status) status[b + i] = hs[i];
    }
    return AURORA_OK;
}

template <typename F>
int for_each_shard(aurora_ctx* ctx, const std::vector<Range>& ranges, F&& f) {
    if (ranges.size() == 1) return f(ctx->devs[0], ranges[0]);
    std::vector<int> rc(ranges.size(), AURORA_OK);
    std::vector<std::thread> th;
    for (size_t k = 0; k < ranges.size(); k++) th.emplace_back([&, k] { rc[k] = f(ctx->devs[k], ranges[k]); });
    for (auto& t : th) t.join();
    for (int r : rc)
        if (r != AURORA_OK) return r;
    return AURORA_OK;
}

// CompressionSettings + LzProperties -> LzChainMatchFinder parameters (LzChainMatchFinder.cs:42-119)
int isqrt2q(int q) {
    int r = 0;
    while ((r + 1) * (r + 1) <= 2 * q) r++;
    return r;
}

int fill_encode_params(EncodeParams& p, int format, const aurora_codec_opts* o) {
    int q = (o && o->quality >= 0) ? o->quality : 8;   // default(CompressionSettings) == Balanced
    if (q > 15) return AURORA_INVALID_ARGUMENT;
    const int mwb = o ? o->max_window_bits : 0;
    if (mwb != 0 && (mwb < 7 || mwb > 28)) return AURORA_INVALID_ARGUMENT;
    aurora_lz_props lz;
    switch (format) {
        case AURORA_FMT_LZ10: {
            const bool vram = !o || o->vram_mode != 0;   // LZ10.cs:33 default true (-1 = default)
            aurora_lz_props_window(&lz, 0x1000, 18, 3, 0, vram ? 2 : 1);
            break;
        }
        case AURORA_FMT_BLZ: aurora_lz_props_window(&lz, 0x1000, 18, 3, 0, 3); break;   // BLZ.cs:24: minimum distance 3
        case AURORA_FMT_LZ40:   // LZ40.cs:29-30, :35: the LZ11 properties, GbaVramCompatibilityMode default false
        case AURORA_FMT_LZ60:
        case AURORA_FMT_LZ11: {
            const bool vram = o && o->vram_mode > 0;     // LZ11.cs:29 default false
            aurora_lz_props_window(&lz, 0x1000, 0x4000, 3, 0, vram ? 2 : 1);
            break;
        }
        case AURORA_FMT_YAZ0:
        case AURORA_FMT_YAZ1:
        case AURORA_FMT_LZHUDSON:   // LZHudson.cs:24
        case AURORA_FMT_YAY0: aurora_lz_props_window(&lz, 0x1000, 0xff + 0x12, 3, 0, 1); break;
        case AURORA_FMT_SMSR00:   // SMSR00.cs:30 (and MIO0.CompressHeaderless with MIO0's own properties: the same)
        case AURORA_FMT_MIO0: aurora_lz_props_window(&lz, 0x1000, 18, 3, 0, 1); break;
        case AURORA_FMT_LZSS:
            if (o && o->lzss.windows_bits != 0) lz = o->lzss;
            else aurora_lz_props_bits(&lz, 12, 4, 2);
            if (lz.windows_bits < 1 || lz.windows_bits > 24 || lz.length_bits < 1 || lz.length_bits > 8) return AURORA_INVALID_ARGUMENT;
            break;
        case AURORA_FMT_LZ4:
        case AURORA_FMT_LZ4_LEGACY:
        case AURORA_FMT_LZ4_BLOCK: aurora_lz_props_window(&lz, 0xFFFF, 0x7FFFFFFF, 4, 0, 1); break;   // LZ4.cs:29
        case AURORA_FMT_LZO: aurora_lz_props_window(&lz, 0xBFFF, 0x7FFFFFFF, 3, 0, 1); break;         // LZO.cs:24
        case AURORA_FMT_SNAPPY:
        case AURORA_FMT_SNAPPY_BLOCK: aurora_lz_props_window(&lz, 0x8000, 64, 4, 0, 1); break;        // Snappy.cs:28
        case AURORA_FMT_PRS: aurora_lz_props_window(&lz, 0x1FFF, 0x100, 2, 0, 1); break;              // PRS.cs:21
        default: return AURORA_NOT_SUPPORTED;
    }
    p.format = format;
    p.lz4_block_size = (o && o->lz4_block_size) ? o->lz4_block_size : 0x400000u;
    if (format == AURORA_FMT_LZ4 && p.lz4_block_size != 0x10000 && p.lz4_block_size != 0x40000 && p.lz4_block_size != 0x100000 &&
        p.lz4_block_size != 0x400000)
        return AURORA_INVALID_ARGUMENT;
    p.byte_order = o ? o->byte_order : AURORA_ENDIAN_DEFAULT;
    p.max_chain = q < 6 ? q + 1 : q >= 11 ? 1 << (q - 5) : ((1 << (q >> 1)) | ((1 << (q >> 1)) >> (q & 1)));
    p.lazy_threshold = 3 + q / 3;
    p.hash_bits = 15 + isqrt2q(q);
    int windows_bits = std::max(1, lz.windows_bits);
    p.max_distance = lz.max_distance;
    if (mwb != 0) {
        windows_bits = std::max(windows_bits, mwb);
        p.max_distance = std::max(p.max_distance, 1 << mwb);
    }
    p.chain_bits = std::min(17 + isqrt2q(q), windows_bits);
    p.min_length = lz.min_length;
    p.max_length = lz.max_length;
    p.min_distance = lz.min_distance;
    p.no_self_overlap = o ? (o->strategy & 1) : 0;
    p.finder_choice = !o ? 0 : (o->strategy & AURORA_STRATEGY_PARALLEL_FINDER) ? 1 : (o->strategy & AURORA_STRATEGY_SERIAL_FINDER) ? 2 : 0;
    p.use_min_table = q >= 10;
    p.yaz0_alignment = o ? o->yaz0_alignment : 0;
    p.lzss = LzssParams{lz.windows_bits, lz.length_bits, lz.min_length, lz.max_distance, lz.windows_start, 0};
    return AURORA_OK;
}

int encode_shard(aurora_ctx* ctx, DeviceCtx* d, int format, const aurora_codec_opts* opts, size_t b, size_t e,
                 const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base,
                 const uint64_t* dst_off, const uint64_t* dst_cap, uint64_t* out_len, int32_t* status,
                 const uint32_t* xor_key = nullptr, uint32_t xor_skip = 0) {
    NvtxRange nvtx_shard("aurora encode shard", d->dev, e - b);
    const size_t n = e - b;
    if (n == 0) return AURORA_OK;
    std::lock_guard<std::mutex> guard(d->mu);
    CU_TRY(ctx, cudaSetDevice(d->dev));
    EncodeParams P{};
    if (fill_encode_params(P, format, opts) != AURORA_OK) return AURORA_INVALID_ARGUMENT;
    const Layout S = plan_layout(src_off, src_len, b, e);
    const Layout D = plan_layout(dst_off, dst_cap, b, e);
    uint64_t max_len = 0;
    for (size_t i = b; i < e; i++) max_len = std::max(max_len, src_len[i]);
    const int warps = encode_resident_warps(d->sm_count);
    P.scratch_per_warp = encode_scratch_per_warp(format, P.hash_bits, P.chain_bits, max_len);
    CU_TRY(ctx, d->scratch.reserve(size_t(warps) * P.scratch_per_warp));
    CU_TRY(ctx, d->src.reserve(S.bytes + 16));
    CU_TRY(ctx, d->dst.reserve(D.bytes + 16));
    const size_t desc_bytes = n * (5 * sizeof(uint64_t) + 2 * sizeof(int32_t)) + 64;   // (+ LZ00 keys behind the status array)
    CU_TRY(ctx, d->desc.reserve(desc_bytes));
    CU_TRY(ctx, d->hdesc.reserve(desc_bytes));
    CU_TRY(ctx, d->ticket.reserve(256));
    uint64_t* h = static_cast<uint64_t*>(d->hdesc.p);
    uint64_t* dv = static_cast<uint64_t*>(d->desc.p);
    for (size_t i = 0; i < n; i++) {
        h[i] = S.dev_off[i];
        h[n + i] = src_len[b + i];
        h[2 * n + i] = D.dev_off[i];
        h[3 * n + i] = dst_cap[b + i];
    }
    cudaStream_t st = d->stream;
    CU_TRY(ctx, cudaMemcpyAsync(dv, h, 4 * n * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    uint8_t* dsrc = static_cast<uint8_t*>(d->src.p);
    uint8_t* ddst = static_cast<uint8_t*>(d->dst.p);
    if (S.span) {
        uint64_t hi = 0;
        for (size_t i = b; i < e; i++) hi = std::max(hi, src_off[i] + src_len[i]);
        if (hi > S.lo) CU_TRY(ctx, cudaMemcpyAsync(dsrc, src_base + S.lo, hi - S.lo, cudaMemcpyHostToDevice, st));
    } else {
        for (size_t i = b; i < e; i++)
            if (src_len[i]) CU_TRY(ctx, cudaMemcpyAsync(dsrc + S.dev_off[i - b], src_base + src_off[i], src_len[i], cudaMemcpyHostToDevice, st));
    }
    CU_TRY(ctx, cudaMemsetAsync(d->ticket.p, 0, 64, st));
    if (format == AURORA_FMT_BLZ) {   // the match finder runs over the reversed source (the device copy, in place)
        CU_TRY(ctx, launch_reverse_bytes(dsrc, dv, dv + n, nullptr, uint32_t(n), st));
        ctx->launches++;
    }
    P.scratch = static_cast<uint8_t*>(d->scratch.p);
    P.src_base = dsrc;
    P.src_limit = S.bytes;
    P.src_off = dv;
    P.src_len = dv + n;
    P.dst_base = ddst;
    P.dst_off = dv + 2 * n;
    P.dst_cap = dv + 3 * n;
    P.out_len = dv + 4 * n;
    P.status = reinterpret_cast<int32_t*>(dv + 5 * n);
    P.ticket = static_cast<unsigned int*>(d->ticket.p);
    P.n = uint32_t(n);
    CU_TRY(ctx, launch_encode(P, warps, st));
    ctx->launches++;
    if (format == AURORA_FMT_BLZ) {   // the codes are stored in the order the backwards decoder reads them
        CU_TRY(ctx, launch_reverse_bytes(ddst, P.dst_off, P.out_len, P.dst_cap, P.n, st));
        ctx->launches++;
    }
    if (xor_key) {   // LZ00: the body the encoder just wrote goes under the keystream (bytes [skip, out_len) of every stream)
        uint32_t* hkey = reinterpret_cast<uint32_t*>(h + 5 * n) + n;
        uint32_t* dkey = reinterpret_cast<uint32_t*>(dv + 5 * n) + n;
        std::memcpy(hkey, xor_key + b, n * sizeof(uint32_t));
        CU_TRY(ctx, cudaMemcpyAsync(dkey, hkey, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        CU_TRY(ctx, launch_lcg_xor(ddst, P.dst_off, P.out_len, P.dst_cap, dkey, xor_skip, P.n, st));
        ctx->launches++;
    }
    CU_TRY(ctx, cudaMemcpyAsync(h + 4 * n, dv + 4 * n, n * sizeof(uint64_t) + n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU_TRY(ctx, cudaStreamSynchronize(st));
    const int32_t* hs = reinterpret_cast<const int32_t*>(h + 5 * n);
    if (D.span) {
        // exactly the bytes every stream produced (the capacities of an encode batch are bounds, mostly unused)
        CU_TRY(ctx, copy_back_windows(dst_base, ddst, D.lo, dst_off, b, e,
                                      [&](size_t i) { return std::min<uint64_t>(h[4 * n + (i - b)], dst_cap[i]); }, 0, st));
    } else {
        for (size_t i = b; i < e; i++) {
            const uint64_t nbytes = std::min<uint64_t>(h[4 * n + (i - b)], dst_cap[i]);
            if (nbytes) CU_TRY(ctx, cudaMemcpyAsync(dst_base + dst_off[i], ddst + D.dev_off[i - b], nbytes, cudaMemcpyDeviceToHost, st));
        }
    }
    CU_TRY(ctx, cudaStreamSynchronize(st));
    for (size_t i = 0; i < n; i++) {
        out_len[b + i] = h[4 * n + i];
        status[b + i] = hs[i];
    }
    return AURORA_OK;
}

}  // namespace

extern "C" {

int aurora_abi_version(void) { return AURORA_ABI_VERSION; }

int aurora_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

aurora_ctx* aurora_init(uint32_t device_mask) {
    int n = aurora_device_count();
    if (n <= 0) {
        g_init_error = "no CUDA device visible";
        return nullptr;
    }
    aurora_ctx* ctx = new aurora_ctx();
    for (int i = 0; i < n && i < 32; i++) {
        if (device_mask != 0 && !(device_mask & (1u << i))) continue;
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, i) != cudaSuccess) continue;
        if (prop.major < 10) continue;   // sm_100a code only
        DeviceCtx* d = new DeviceCtx();
        d->dev = i;
        d->sm_count = prop.multiProcessorCount;
        if (cudaSetDevice(i) != cudaSuccess || cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&d->s_in, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&d->s_out, cudaStreamNonBlocking) != cudaSuccess) {
            delete d;
            continue;
        }
        ctx->devs.push_back(d);
    }
    if (ctx->devs.empty()) {
        g_init_error = "no sm_100 device among the visible CUDA devices";
        delete ctx;
        return nullptr;
    }
    return ctx;
}

void aurora_shutdown(aurora_ctx* ctx) {
    if (!ctx) return;
    for (DeviceCtx* d : ctx->devs) {
        cudaSetDevice(d->dev);
        cudaStreamSynchronize(d->stream);
        d->src.release();
        d->dst.release();
        d->desc.release();
        d->ticket.release();
        d->scratch.release();
        d->order.release();
        d->hdesc.release();
        for (cudaEvent_t e : d->ev_in) cudaEventDestroy(e);
        for (cudaEvent_t e : d->ev_k) cudaEventDestroy(e);
        cudaStreamDestroy(d->s_in);
        cudaStreamDestroy(d->s_out);
        cudaStreamDestroy(d->stream);
        delete d;
    }
    delete ctx;
}

int aurora_ctx_device_count(const aurora_ctx* ctx) { return ctx ? int(ctx->devs.size()) : 0; }

const char* aurora_last_error_string(const aurora_ctx* ctx) {
    if (!ctx) return g_init_error.c_str();
    return ctx->last_error.c_str();
}

const char* aurora_status_string(int s) {
    static const char* names[] = {"OK", "END_OF_STREAM", "INVALID_IDENTIFIER", "SIZE_MISMATCH", "DST_TOO_SMALL",
                                  "INVALID_DATA", "NOT_SUPPORTED", "INVALID_ARGUMENT", "CUDA_ERROR"};
    return (s >= 0 && s <= 8) ? names[s] : "UNKNOWN";
}

void* aurora_pinned_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) return nullptr;
    return p;
}
void aurora_pinned_free(void* p) {
    if (p) cudaFreeHost(p);
}

void aurora_lz_props_window(aurora_lz_props* out, int32_t windows_size, int32_t max_length, int32_t min_length,
                            int32_t windows_start, int32_t min_distance) {
    out->windows_bits = ceil_log2(windows_size);
    out->length_bits = ceil_log2((long long)max_length - min_length) & 0xFF;
    out->min_length = min_length;
    out->max_length = max_length;
    out->max_distance = windows_size;
    out->min_distance = min_distance;
    out->windows_start = windows_start;
    out->reserved = 0;
}

void aurora_lz_props_bits(aurora_lz_props* out, int32_t distance_bits, int32_t length_bits, int32_t threshold) {
    out->windows_bits = distance_bits;
    out->length_bits = length_bits;
    out->min_length = threshold + 1;
    out->max_distance = 1 << distance_bits;
    out->max_length = (1 << length_bits) + threshold;
    out->windows_start = out->max_distance - (1 << length_bits) - threshold;
    out->min_distance = 1;
    out->reserved = 0;
}

void aurora_codec_opts_init(aurora_codec_opts* o) {
    std::memset(o, 0, sizeof(*o));
    o->struct_size = sizeof(*o);
    o->byte_order = AURORA_ENDIAN_DEFAULT;
    o->quality = -1;
    o->vram_mode = -1;
}

uint64_t aurora_kernel_launch_count(const aurora_ctx* ctx) { return ctx ? ctx->launches.load() : 0; }

int aurora_decode_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                        const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                        const uint64_t* dst_cap, uint64_t* out_len, uint64_t* consumed, int32_t* status) {
    if (!ctx) return AURORA_INVALID_ARGUMENT;
    if (n == 0) return AURORA_OK;
    if (!src_base || !src_off || !src_len || !dst_base || !dst_off || !dst_cap || !status ||
        !(is_flaglz(format) || is_bytelz(format) || format == AURORA_FMT_BLZ || aurora::is_wrapper_format(format))) {
        ctx->set_error("aurora_decode_batch: null argument or unknown format");
        return AURORA_INVALID_ARGUMENT;
    }
    if (n > 0xFFFFFFF0ull) return AURORA_INVALID_ARGUMENT;
    if (aurora::is_wrapper_format(format))
        return aurora::wrapped_decode_batch(ctx, format, opts, n, src_base, src_off, src_len, dst_base, dst_off, dst_cap, out_len, consumed, status);
    return aurora::decode_core_batch(ctx, format, opts, n, src_base, src_off, src_len, dst_base, dst_off, dst_cap, nullptr, out_len, consumed, status);
}

int aurora_decoded_size_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                              const uint64_t* src_off, const uint64_t* src_len, int size_scan, uint64_t* out_size,
                              int32_t* status) {
    if (!ctx) return AURORA_INVALID_ARGUMENT;
    if (n == 0) return AURORA_OK;
    if (!src_base || !src_off || !src_len || !out_size || !status) return AURORA_INVALID_ARGUMENT;
    // GetDecompressedSize is a header peek (e.g. Yaz0.cs:50-55, LZ10.cs:47-57): a few bytes of host memory
    if (aurora::is_wrapper_format(format) || is_flaglz(format) || format == AURORA_FMT_BLZ) {
        const int bo = opts ? opts->byte_order : AURORA_ENDIAN_DEFAULT;
        for (size_t i = 0; i < n; i++) {
            const uint8_t* p = src_base + src_off[i];
            status[i] = aurora::is_wrapper_format(format) ? aurora::wrapped_decoded_size(format, p, src_len[i], &out_size[i])
                                                          : aurora::core_decoded_size(format, bo, p, src_len[i], &out_size[i]);
        }
        return AURORA_OK;
    }
    if (!is_bytelz(format)) return AURORA_INVALID_ARGUMENT;
    if (!size_scan) {
        for (size_t i = 0; i < n; i++) {
            out_size[i] = 0;
            status[i] = AURORA_NOT_SUPPORTED;   // LZ4/LZO/Snappy/PRS do not implement IProvidesDecompressedSize
        }
        return AURORA_OK;
    }
    // size-only pre-pass on the device: same parser, all stores dropped
    std::vector<uint64_t> zero(n, 0), cons(n);
    uint8_t dummy[16];
    const std::vector<Range> ranges = shard(n, int(ctx->devs.size()), src_len, nullptr);
    int rc = for_each_shard(ctx, ranges, [&](DeviceCtx* d, Range r) {
        return decode_shard(ctx, d, format, opts, r.begin, r.end, src_base, src_off, src_len, dummy, zero.data(), zero.data(),
                            out_size, cons.data(), status, 1);
    });
    if (rc != AURORA_OK) return rc;
    for (size_t i = 0; i < n; i++)
        if (status[i] == AURORA_DST_TOO_SMALL) status[i] = AURORA_OK;
    return AURORA_OK;
}

int aurora_is_match_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                          const uint64_t* src_off, const uint64_t* src_len, uint8_t* match) {
    (void)opts;
    if (!ctx) return AURORA_INVALID_ARGUMENT;
    if (n == 0) return AURORA_OK;
    if (!src_base || !src_off || !src_len || !match) return AURORA_INVALID_ARGUMENT;
    if (aurora::is_wrapper_format(format)) return aurora::wrapped_is_match_batch(ctx, format, opts, n, src_base, src_off, src_len, match);
    if (format == AURORA_FMT_LZ10 || format == AURORA_FMT_LZ11 || format == AURORA_FMT_PRS) {
        // token-walk heuristics run on the device, one thread per candidate stream (csrc/ismatch.cu)
        if (n > 0xFFFFFFF0ull) return AURORA_INVALID_ARGUMENT;
        DeviceCtx* d = ctx->devs[0];
        std::lock_guard<std::mutex> guard(d->mu);
        CU_TRY(ctx, cudaSetDevice(d->dev));
        const Layout S = plan_layout(src_off, src_len, 0, n);
        CU_TRY(ctx, d->src.reserve(S.bytes + 16));
        CU_TRY(ctx, d->desc.reserve(n * 17 + 64));
        CU_TRY(ctx, d->hdesc.reserve(n * 17 + 64));
        uint64_t* h = static_cast<uint64_t*>(d->hdesc.p);
        uint64_t* dv = static_cast<uint64_t*>(d->desc.p);
        for (size_t i = 0; i < n; i++) {
            h[i] = S.dev_off[i];
            h[n + i] = src_len[i];
        }
        cudaStream_t st = d->stream;
        uint8_t* dsrc = static_cast<uint8_t*>(d->src.p);
        CU_TRY(ctx, cudaMemcpyAsync(dv, h, 2 * n * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
        if (S.span) {
            uint64_t hi = 0;
            for (size_t i = 0; i < n; i++) hi = std::max(hi, src_off[i] + src_len[i]);
            if (hi > S.lo) CU_TRY(ctx, cudaMemcpyAsync(dsrc, src_base + S.lo, hi - S.lo, cudaMemcpyHostToDevice, st));
        } else {
            for (size_t i = 0; i < n; i++)
                if (src_len[i]) CU_TRY(ctx, cudaMemcpyAsync(dsrc + S.dev_off[i], src_base + src_off[i], src_len[i], cudaMemcpyHostToDevice, st));
        }
        uint8_t* dm = reinterpret_cast<uint8_t*>(dv + 2 * n);
        CU_TRY(ctx, launch_is_match(dsrc, dv, dv + n, dm, uint32_t(n), format, st));
        ctx->launches++;
        CU_TRY(ctx, cudaMemcpyAsync(match, dm, n, cudaMemcpyDeviceToHost, st));
        CU_TRY(ctx, cudaStreamSynchronize(st));
        return AURORA_OK;
    }
    // the magic and footer rules (csrc/ismatch.cu) on the host: a peek of a few bytes per stream
    for (size_t i = 0; i < n; i++) {
        const int m = aurora::is_match_one(src_base + src_off[i], src_len[i], format);
        if (m < 0) {
            ctx->set_error("aurora_is_match_batch: unknown format");
            return AURORA_INVALID_ARGUMENT;
        }
        match[i] = uint8_t(m);
    }
    return AURORA_OK;
}

int aurora_scan_offsets(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, const uint8_t* image, uint64_t len, uint8_t* match) {
    (void)opts;
    if (!ctx) return AURORA_INVALID_ARGUMENT;
    if (len == 0) return AURORA_OK;
    if (!image || !match || !(is_flaglz(format) || is_bytelz(format)) || format == AURORA_FMT_LZ4_BLOCK || format == AURORA_FMT_SNAPPY_BLOCK ||
        len > 0xFFFFFFFF00ull)
        return AURORA_INVALID_ARGUMENT;
    DeviceCtx* d = ctx->devs[0];
    std::lock_guard<std::mutex> guard(d->mu);
    CU_TRY(ctx, cudaSetDevice(d->dev));
    CU_TRY(ctx, d->src.reserve(len + 16));
    CU_TRY(ctx, d->dst.reserve(len + 16));
    cudaStream_t st = d->stream;
    CU_TRY(ctx, cudaMemcpyAsync(d->src.p, image, len, cudaMemcpyHostToDevice, st));
    CU_TRY(ctx, launch_scan(static_cast<const uint8_t*>(d->src.p), len, static_cast<uint8_t*>(d->dst.p), format, st));
    ctx->launches++;
    CU_TRY(ctx, cudaMemcpyAsync(match, d->dst.p, len, cudaMemcpyDeviceToHost, st));
    CU_TRY(ctx, cudaStreamSynchronize(st));
    return AURORA_OK;
}

int aurora_decode_batch_device(aurora_ctx* ctx, int device, int format, const aurora_codec_opts* opts, size_t n,
                               const uint8_t* d_src_base, uint64_t src_total, const uint64_t* d_src_off,
                               const uint64_t* d_src_len, uint8_t* d_dst_base, const uint64_t* d_dst_off,
                               const uint64_t* d_dst_cap, uint64_t* d_out_len, uint64_t* d_consumed, int32_t* d_status,
                               void* stream) {
    if (!ctx || device < 0 || device >= int(ctx->devs.size())) return AURORA_INVALID_ARGUMENT;
    if (n == 0) return AURORA_OK;
    if (!(is_flaglz(format) || is_bytelz(format) || format == AURORA_FMT_BLZ) || n > 0xFFFFFFF0ull) return AURORA_INVALID_ARGUMENT;
    if ((reinterpret_cast<uintptr_t>(d_src_base) & 15) != 0) {
        ctx->set_error("aurora_decode_batch_device: d_src_base must be 16-byte aligned");
        return AURORA_INVALID_ARGUMENT;
    }
    DeviceCtx* d = ctx->devs[device];
    std::lock_guard<std::mutex> guard(d->mu);
    CU_TRY(ctx, cudaSetDevice(d->dev));
    DecodeParams P{};
    if (fill_decode_params(P, format, opts) != AURORA_OK) {
        ctx->set_error("aurora_decode_batch_device: unsupported LZSS properties");
        return AURORA_INVALID_ARGUMENT;
    }
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : d->stream;
    CU_TRY(ctx, d->ticket.reserve(256));
    CU_TRY(ctx, cudaMemsetAsync(d->ticket.p, 0, 64, st));
    P.src_base = d_src_base;
    P.src_limit = align_up(src_total, 16);   // the allocation must be readable up to the next multiple of 16
    P.src_off = d_src_off;
    P.src_len = d_src_len;
    P.dst_base = d_dst_base;
    P.dst_off = d_dst_off;
    P.dst_cap = d_dst_cap;
    P.out_len = d_out_len;
    P.consumed = d_consumed;
    P.status = d_status;
    P.order = nullptr;
    if (opts && opts->balance == 1 && n > 1) {
        // largest-first hand-out (streams with a wide size spread, config C3): three tiny kernels, no host sync
        CU_TRY(ctx, d->order.reserve(n * sizeof(uint32_t) + 256));
        uint32_t* hist = static_cast<uint32_t*>(d->order.p);
        uint32_t* ord = hist + 64;
        CU_TRY(ctx, launch_size_order(d_dst_cap, uint32_t(n), hist, ord, st));
        ctx->launches += 3;
        P.order = ord;
    }
    P.ticket = static_cast<unsigned int*>(d->ticket.p);
    P.n = uint32_t(n);
    CU_TRY(ctx, launch_decode(P, d->sm_count, st));
    ctx->launches++;
    return AURORA_OK;
}

}  // extern "C"

extern "C" {

uint64_t aurora_encode_bound(int format, uint64_t raw_len) {
    if (aurora::is_wrapper_format(format)) return aurora::wrapped_encode_bound(format, raw_len, nullptr);
    // worst case of every token writer on the hot path: all literals + flag bits + headers / chunk framing
    switch (format) {
        case AURORA_FMT_LZ4:
        case AURORA_FMT_LZ4_LEGACY:
        case AURORA_FMT_LZ4_BLOCK: return raw_len + raw_len / 255 + 64 + 8 * (raw_len / 0x400000 + 1);
        case AURORA_FMT_SNAPPY:
        case AURORA_FMT_SNAPPY_BLOCK: return raw_len + raw_len / 60 + 32 + 16 * (raw_len / 0x10000 + 1);
        // LZO: a far 3-byte match costs 3 bytes and splits the literal run around it (4 literals + 1 match = 7 bytes in, 8 out)
        case AURORA_FMT_LZO: return raw_len + raw_len / 6 + 64;
        default: return raw_len + raw_len / 8 + 64;
    }
}

int aurora_encode_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                        const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                        const uint64_t* dst_cap, uint64_t* out_len, int32_t* status) {
    if (!ctx) return AURORA_INVALID_ARGUMENT;
    if (n == 0) return AURORA_OK;
    if (!src_base || !src_off || !src_len || !dst_base || !dst_off || !dst_cap || !out_len || !status || n > 0xFFFFFFF0ull) {
        ctx->set_error("aurora_encode_batch: null argument");
        return AURORA_INVALID_ARGUMENT;
    }
    if (aurora::is_wrapper_format(format))
        return aurora::wrapped_encode_batch(ctx, format, opts, n, src_base, src_off, src_len, dst_base, dst_off, dst_cap, out_len, status);
    const int rc = aurora::encode_core_batch(ctx, format, opts, n, src_base, src_off, src_len, dst_base, dst_off, dst_cap, out_len, status);
    if (rc == AURORA_OK && format == AURORA_FMT_BLZ) {
        // BLZ.Compress (BLZ.cs:78-92): behind the codes 0xFF padding to a multiple of 16, then the footer — u24 LE total size,
        // u8 footer-and-padding size, i32 LE (decoded size - total size)
        for (size_t i = 0; i < n; i++) {
            if (status[i] != AURORA_OK) continue;
            const uint64_t total0 = out_len[i] + 8, padding = (16 - total0 % 16) % 16, total = total0 + padding;
            if (total > dst_cap[i]) { status[i] = AURORA_DST_TOO_SMALL; continue; }
            uint8_t* d = dst_base + dst_off[i] + out_len[i];
            std::memset(d, 0xFF, size_t(padding));
            d += padding;
            d[0] = uint8_t(total); d[1] = uint8_t(total >> 8); d[2] = uint8_t(total >> 16);
            d[3] = uint8_t(8 + padding);
            const uint32_t delta = uint32_t(src_len[i]) - uint32_t(total);
            d[4] = uint8_t(delta); d[5] = uint8_t(delta >> 8); d[6] = uint8_t(delta >> 16); d[7] = uint8_t(delta >> 24);
            out_len[i] = total;
        }
    }
    return rc;
}

}  // extern "C"

namespace aurora {

int decode_core_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                      const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                      const uint64_t* dst_cap, const uint64_t* raw_size, uint64_t* out_len, uint64_t* consumed, int32_t* status,
                      const uint32_t* xor_key, bool exact) {
    if (n == 0) return AURORA_OK;
    const std::vector<Range> ranges = shard(n, int(ctx->devs.size()), src_len, dst_cap, dst_off);
    return for_each_shard(ctx, ranges, [&](DeviceCtx* d, Range r) {
        return decode_shard(ctx, d, format, opts, r.begin, r.end, src_base, src_off, src_len, dst_base, dst_off, dst_cap,
                            out_len, consumed, status, 0, raw_size, xor_key, exact);
    });
}

int encode_core_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                      const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                      const uint64_t* dst_cap, uint64_t* out_len, int32_t* status, const uint32_t* xor_key, uint32_t xor_skip) {
    if (n == 0) return AURORA_OK;
    EncodeParams probe{};
    const int rc = fill_encode_params(probe, format, opts);
    if (rc != AURORA_OK) {
        ctx->set_error("aurora_encode_batch: unknown format or invalid settings");
        return rc;
    }
    const std::vector<Range> ranges = shard(n, int(ctx->devs.size()), src_len, nullptr);
    return for_each_shard(ctx, ranges, [&](DeviceCtx* d, Range r) {
        return encode_shard(ctx, d, format, opts, r.begin, r.end, src_base, src_off, src_len, dst_base, dst_off, dst_cap, out_len, status,
                            xor_key, xor_skip);
    });
}

}  // namespace aurora

extern "C" {

int aurora_encode_batch_device(aurora_ctx* ctx, int device, int format, const aurora_codec_opts* opts, size_t n,
                               const uint8_t* d_src_base, uint64_t src_total, const uint64_t* d_src_off,
                               const uint64_t* d_src_len, uint8_t* d_dst_base, const uint64_t* d_dst_off,
                               const uint64_t* d_dst_cap, uint64_t* d_out_len, int32_t* d_status, void* stream) {
    if (!ctx || device < 0 || device >= int(ctx->devs.size())) return AURORA_INVALID_ARGUMENT;
    if (n == 0) return AURORA_OK;
    if (n > 0xFFFFFFF0ull) return AURORA_INVALID_ARGUMENT;
    DeviceCtx* d = ctx->devs[device];
    std::lock_guard<std::mutex> guard(d->mu);
    CU_TRY(ctx, cudaSetDevice(d->dev));
    EncodeParams P{};
    const int rc = format == AURORA_FMT_BLZ ? AURORA_NOT_SUPPORTED   // needs the reversal passes and the host-written footer
                                             : fill_encode_params(P, format, opts);
    if (rc != AURORA_OK) {
        ctx->set_error("aurora_encode_batch_device: unknown format or invalid settings");
        return rc;
    }
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : d->stream;
    // MIO0/Yay0 stage their code and literal sections per warp, sized by the largest stream of the batch
    uint64_t max_len = 0;
    if (format == AURORA_FMT_MIO0 || format == AURORA_FMT_YAY0 || format == AURORA_FMT_SMSR00) {
        CU_TRY(ctx, d->hdesc.reserve(n * sizeof(uint64_t)));
        CU_TRY(ctx, cudaMemcpyAsync(d->hdesc.p, d_src_len, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        CU_TRY(ctx, cudaStreamSynchronize(st));
        const uint64_t* hl = static_cast<const uint64_t*>(d->hdesc.p);
        for (size_t i = 0; i < n; i++) max_len = std::max(max_len, hl[i]);
    }
    const int warps = encode_resident_warps(d->sm_count);
    P.scratch_per_warp = encode_scratch_per_warp(format, P.hash_bits, P.chain_bits, max_len);
    CU_TRY(ctx, d->scratch.reserve(size_t(warps) * P.scratch_per_warp));
    CU_TRY(ctx, d->ticket.reserve(256));
    CU_TRY(ctx, cudaMemsetAsync(d->ticket.p, 0, 64, st));
    P.scratch = static_cast<uint8_t*>(d->scratch.p);
    P.src_base = d_src_base;
    P.src_limit = src_total;
    P.src_off = d_src_off;
    P.src_len = d_src_len;
    P.dst_base = d_dst_base;
    P.dst_off = d_dst_off;
    P.dst_cap = d_dst_cap;
    P.out_len = d_out_len;
    P.status = d_status;
    P.ticket = static_cast<unsigned int*>(d->ticket.p);
    P.n = uint32_t(n);
    CU_TRY(ctx, launch_encode(P, warps, st));
    ctx->launches++;
    return AURORA_OK;
}

}  // extern "C"
