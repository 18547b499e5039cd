// scan_decode.cu — aurora_scan_decode_device: the CLI's `-scan` walk (Commands/ScanDecompressCommand.cs:23-39) on the device.
// The walk tests IsMatch at a position, decodes there when it hits, resumes after the consumed bytes of an OK stream and steps
// by one byte otherwise.  It runs in rounds from the current position p (DESIGN.md §4.5):
//   1. the hits of the window [p, p + W), ascending, at most kRoundHits of them (launch_window_hits, ismatch.cu);
//   2. a capacity per hit that gives the decode at max_size's answer (hit_prep_kernel; the byte-LZ formats first run the
//      decode kernel's size-only parse), 16-byte aligned slots for them by an exclusive scan, cut at the round's slot budget;
//   3. the decode kernel on the windows [h, len) of all the round's hits, into the slots;
//   4. one warp follows the walk through the round's hits (walk_round) and writes the entries' descriptors;
//   5. the entries' bytes go from their slots to the caller's packed destination.
// Everything above the "// ---- kernel" line is the walk's rule, which tests/test_scan_walk_simt.py compiles for the CPU.
#include "api_internal.hpp"
#include "common.cuh"

namespace aurora {

__host__ __device__ inline uint64_t scan_align16(uint64_t v) { return (v + 15) & ~uint64_t(15); }

// The walk's successor rule: where the walk goes on from a hit at `start` whose decode gave `status` and `consumed`.
__host__ __device__ inline uint64_t walk_target(uint64_t start, int32_t status, uint64_t consumed) {
    return start + (status == AURORA_OK && consumed > 1 ? consumed : 1);
}

// The walk's state between rounds and calls: the position, the entries written and the bytes they take.
struct WalkState {
    uint64_t p;          // the walk position (W(p) continues the walk)
    uint64_t found;      // entries written
    uint64_t dst_pos;    // destination offset of the next entry (16-byte aligned)
    uint64_t round_first;   // the first entry of the current round
    uint32_t nsel;       // hits of the current round's window (all of them; at most kRoundHits are kept)
    uint32_t cut;        // the first hit of the round without a slot (0xFFFFFFFF: none)
    uint32_t stopped;    // the walk met an entry past max_found or dst_bytes; p is its start
    uint32_t pad;
};

// One round's hits: every hit in [first position, end) is among hit[0 .. n), ascending, with its decode's outcome.
struct WalkRound {
    const uint64_t* hit;
    const int32_t* status;
    const uint64_t* consumed;
    const uint64_t* out_len;
    uint32_t n;
    uint64_t end;   // where this round's knowledge of the hits ends (<= len)
    uint64_t len;
};

// The walk through one round from s.p, the emission rule included.  first_ok(k, t): the first index j >= k with hit[j] >= t
// and status[j] OK, or n — the hits in between are not OK, so the walk steps over them one byte at a time.  emit(k, entry,
// dst_off): hit k becomes entry `entry` at destination offset dst_off.  The walk stops before an entry that would be the
// max_found + 1-th or whose bytes would pass dst_bytes, with s.p at its start; it leaves the round at the first position the
// round does not know.
template <typename FirstOk, typename Emit>
__host__ __device__ void walk_round(const WalkRound& r, WalkState& s, uint64_t max_found, uint64_t dst_bytes, FirstOk first_ok, Emit emit) {
    uint32_t k = first_ok(0u, s.p);
    while (k < r.n) {
        const uint64_t h = r.hit[k], ol = r.out_len[k];
        if (s.found >= max_found || ol > dst_bytes || s.dst_pos > dst_bytes - ol) {
            s.p = h;
            s.stopped = 1;
            return;
        }
        emit(k, s.found, s.dst_pos);
        s.found++;
        s.dst_pos += scan_align16(ol);
        const uint64_t t = walk_target(h, AURORA_OK, r.consumed[k]);
        if (t >= r.end) {
            s.p = t < r.len ? t : r.len;
            return;
        }
        k = first_ok(k + 1, t);
    }
    s.p = r.end;
}

// ---- kernel
}  // namespace aurora

#include <cub/device/device_scan.cuh>
#include <thrust/iterator/transform_iterator.h>

#include "size_peek.cuh"

namespace aurora {

namespace {

constexpr uint32_t kRoundHits = 1u << 16;     // hits kept per round
constexpr uint32_t kWindowMin = 1u << 17;     // window bounds (bytes of the image tested per round)
constexpr uint32_t kWindowMax = 1u << 30;
constexpr uint32_t kWindowStart = 1u << 24;
constexpr uint64_t kSlotBudget = 256ull << 20;   // decoded bytes per round, at least max_size
constexpr int kGatherBlocks = 1024;

// the round's per-hit arrays, carved out of ScanScratch::hits
struct HitArrays {
    uint64_t *hit, *src_len, *cap, *off, *out_len, *consumed;
    int32_t* status;
    uint32_t *rel, *entry_hit;
};

HitArrays carve(void* base) {
    HitArrays a;
    uint64_t* q = static_cast<uint64_t*>(base);
    a.hit = q;
    a.src_len = q + kRoundHits;
    a.cap = q + 2 * kRoundHits;
    a.off = q + 3 * kRoundHits;
    a.out_len = q + 4 * kRoundHits;
    a.consumed = q + 5 * kRoundHits;
    a.status = reinterpret_cast<int32_t*>(q + 6 * kRoundHits);
    a.rel = reinterpret_cast<uint32_t*>(a.status + kRoundHits);
    a.entry_hit = a.rel + kRoundHits;
    return a;
}
constexpr size_t kHitArrayBytes = size_t(kRoundHits) * (6 * 8 + 3 * 4);

// The capacity at which a flag-LZ hit's decode answers as the decode at max_size does: the decode kernel refuses a header size
// above its capacity up front and otherwise stays below it unless it fails (written > size is SIZE_MISMATCH), so any capacity
// at least the largest size it may try that fits max_size, and at most max_size, gives the same outcome and bytes.  Yaz0 /
// Yaz1 retry with the byte-swapped size, MIO0 and Yay0 pick an order from the header: both orders of the u32 at 4 count for
// them.  A header the peek cannot read fails the decode at every capacity.
__device__ uint64_t flaglz_capacity(int format, int byte_order, const uint8_t* p, uint64_t len, uint64_t max_size) {
    if (format == AURORA_FMT_YAZ0 || format == AURORA_FMT_YAZ1 || format == AURORA_FMT_YAY0 || format == AURORA_FMT_MIO0) {
        if (len < 8) return 0;
        const uint64_t be = (uint32_t(p[4]) << 24) | (uint32_t(p[5]) << 16) | (uint32_t(p[6]) << 8) | p[7];
        const uint64_t le = uint32_t(p[4]) | (uint32_t(p[5]) << 8) | (uint32_t(p[6]) << 16) | (uint32_t(p[7]) << 24);
        uint64_t c = be <= max_size ? be : 0;
        if (le <= max_size && le > c) c = le;
        return c;
    }
    uint64_t s;
    if (core_decoded_size(format, byte_order, p, len, &s) != AURORA_OK) return 0;
    return s <= max_size ? s : 0;
}

// hit k: its absolute position, its window's length and (flag-LZ) its capacity; the byte-LZ formats get 0 for the size-only
// parse (zero destination offsets and capacities)
__global__ void hit_prep_kernel(const uint8_t* image, uint64_t len, const WalkState* s, HitArrays a, uint32_t n, int format,
                                int byte_order, uint64_t max_size, int flaglz) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint64_t h = s->p + a.rel[k];
    a.hit[k] = h;
    a.src_len[k] = len - h;
    a.cap[k] = flaglz ? flaglz_capacity(format, byte_order, image + h, len - h, max_size) : 0;
    a.off[k] = 0;
}

// byte-LZ: the size-only parse's length is the capacity when the parse reached the end (OK, or DST_TOO_SMALL against its zero
// capacity, as size_scan_status) and fits max_size; a parse that fails fails the decode at every capacity
__global__ void bytelz_cap_kernel(HitArrays a, uint32_t n, uint64_t max_size) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int32_t st = a.status[k];
    a.cap[k] = (st == AURORA_OK || st == AURORA_DST_TOO_SMALL) && a.out_len[k] <= max_size ? a.out_len[k] : 0;
}

// hits whose slot passes the budget get no slot (capacity 0, offset 0: nothing written); slot offsets rise with k, so they are a
// suffix, and the walk of this round ends at the first of them
__global__ void slot_cut_kernel(HitArrays a, uint32_t n, uint64_t budget, WalkState* s) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    if (a.off[k] + a.cap[k] > budget) {
        atomicMin(&s->cut, k);
        a.cap[k] = 0;
        a.off[k] = 0;
    }
}

struct Align16 {
    __host__ __device__ uint64_t operator()(uint64_t v) const { return scan_align16(v); }
};

// one warp: the walk through the round (all lanes run walk_round in step; first_ok is a ballot over 32 hits at a time)
__global__ void walk_kernel(HitArrays a, uint32_t n, uint32_t items, uint64_t len, WalkState* s, uint64_t max_found, uint64_t dst_bytes,
                            uint64_t* d_start, uint64_t* d_consumed, uint64_t* d_out_len, uint64_t* d_dst_off) {
    const uint32_t lane = threadIdx.x & 31;
    WalkState w = *s;
    const uint32_t known = min(n, w.cut);
    WalkRound r;
    r.hit = a.hit;
    r.status = a.status;
    r.consumed = a.consumed;
    r.out_len = a.out_len;
    r.n = known;
    r.len = len;
    // the hits of [p, end) are all known: up to the first hit without a slot, or past the last hit kept of a window with more
    r.end = known < n ? a.hit[known] : n < w.nsel ? a.hit[n - 1] + 1 : min(w.p + items, len);
    w.round_first = w.found;
    auto first_ok = [&](uint32_t k, uint64_t t) -> uint32_t {
        for (; k < known; k += 32) {
            const uint32_t j = k + lane;
            const uint32_t m = __ballot_sync(kFull, j < known && a.status[j] == AURORA_OK && a.hit[j] >= t);
            if (m) return k + __ffs(m) - 1;
        }
        return known;
    };
    auto emit = [&](uint32_t k, uint64_t e, uint64_t dst_off) {
        if (lane == 0) {
            d_start[e] = a.hit[k];
            d_consumed[e] = a.consumed[k];
            d_out_len[e] = a.out_len[k];
            d_dst_off[e] = dst_off;
            a.entry_hit[e - w.round_first] = k;
        }
    };
    walk_round(r, w, max_found, dst_bytes, first_ok, emit);
    if (lane == 0) {
        w.cut = 0xFFFFFFFFu;
        *s = w;
    }
}

// the round's entries: their bytes from the slots to the caller's destination, one block per entry
__global__ void gather_kernel(const uint8_t* slots, HitArrays a, const WalkState* s, const uint64_t* d_out_len, const uint64_t* d_dst_off,
                              uint8_t* dst_base) {
    const uint64_t first = s->round_first, count = s->found - first;
    for (uint64_t e = blockIdx.x; e < count; e += gridDim.x) {
        const uint32_t k = a.entry_hit[e];
        const uint8_t* from = slots + a.off[k];
        uint8_t* to = dst_base + d_dst_off[first + e];
        const uint64_t nb = d_out_len[first + e];
        uint64_t done = 0;
        if ((reinterpret_cast<uintptr_t>(to) & 15) == 0) {   // slots and destination offsets are 16-byte aligned
            const uint64_t words = nb / 16;
            for (uint64_t i = threadIdx.x; i < words; i += blockDim.x)
                reinterpret_cast<uint4*>(to)[i] = reinterpret_cast<const uint4*>(from)[i];
            done = words * 16;
        }
        for (uint64_t i = done + threadIdx.x; i < nb; i += blockDim.x) to[i] = from[i];
    }
}

}  // namespace

cudaError_t scan_decode_rounds(int format, const aurora_codec_opts* opts, const uint8_t* d_image, uint64_t len, uint64_t begin,
                               uint64_t max_size, uint64_t max_found, uint64_t* d_start, uint64_t* d_consumed, uint64_t* d_out_len,
                               uint8_t* d_dst_base, uint64_t dst_bytes, uint64_t* d_dst_off, uint64_t* found, uint64_t* next,
                               ScanScratch& scr, unsigned int* ticket, int sm_count, cudaStream_t st, uint64_t* launches) {
    DecodeParams P{};
    fill_decode_params(P, format, opts);   // (the caller has checked its LZSS properties)
    const bool flag = is_flaglz(format);
    const uint64_t budget = max_size > kSlotBudget ? max_size : kSlotBudget;

    size_t sel_bytes = 0, scan_bytes = 0;
    cudaError_t e = launch_window_hits(nullptr, 0, nullptr, kWindowMax, format, nullptr, 0, nullptr, nullptr, &sel_bytes, st);
    if (e != cudaSuccess) return e;
    e = cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, thrust::make_transform_iterator(static_cast<const uint64_t*>(nullptr), Align16{}),
                                      static_cast<uint64_t*>(nullptr), int(kRoundHits), st);
    if (e != cudaSuccess) return e;
    const size_t temp_bytes = sel_bytes > scan_bytes ? sel_bytes : scan_bytes;
    if ((e = scr.state.reserve(sizeof(WalkState))) != cudaSuccess || (e = scr.hits.reserve(kHitArrayBytes)) != cudaSuccess ||
        (e = scr.temp.reserve(temp_bytes)) != cudaSuccess || (e = scr.slots.reserve(budget + 16)) != cudaSuccess)
        return e;
    WalkState* ds = static_cast<WalkState*>(scr.state.p);
    const HitArrays a = carve(scr.hits.p);
    uint8_t* slots = static_cast<uint8_t*>(scr.slots.p);

    WalkState hs{};
    hs.p = begin;
    hs.cut = 0xFFFFFFFFu;
    if ((e = cudaMemcpyAsync(ds, &hs, sizeof hs, cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
    uint64_t p_known = begin;   // a lower bound of the device's walk position
    uint32_t window = kWindowStart;
    for (;;) {
        const uint32_t items = uint32_t(window < len - p_known ? window : len - p_known);
        size_t tb = temp_bytes;
        if ((e = launch_window_hits(d_image, len, &ds->p, items, format, a.rel, kRoundHits, &ds->nsel, scr.temp.p, &tb, st)) != cudaSuccess)
            return e;
        *launches += 2;
        // the round's one host read: the walk position and the window's hit count
        if ((e = cudaMemcpyAsync(&hs, ds, sizeof hs, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
        if (hs.stopped || hs.p >= len) break;
        const uint32_t n = hs.nsel < kRoundHits ? hs.nsel : kRoundHits;
        if (n > 0) {
            const uint32_t grid = (n + 255) / 256;
            hit_prep_kernel<<<grid, 256, 0, st>>>(d_image, len, ds, a, n, format, P.byte_order, max_size, flag ? 1 : 0);
            *launches += 1;
            P.src_base = d_image;
            P.src_limit = scan_align16(len);
            P.src_off = a.hit;
            P.src_len = a.src_len;
            P.dst_base = slots;
            P.out_len = a.out_len;
            P.consumed = a.consumed;
            P.status = a.status;
            P.order = nullptr;
            P.ticket = ticket;
            P.n = n;
            if (!flag) {   // the size-only parse (no stores) against zero offsets and capacities
                P.size_only = 1;
                P.dst_off = a.off;
                P.dst_cap = a.cap;
                if ((e = cudaMemsetAsync(ticket, 0, 64, st)) != cudaSuccess || (e = launch_decode(P, sm_count, st)) != cudaSuccess) return e;
                bytelz_cap_kernel<<<grid, 256, 0, st>>>(a, n, max_size);
                *launches += 2;
                P.size_only = 0;
            }
            size_t sb = temp_bytes;
            if ((e = cub::DeviceScan::ExclusiveSum(scr.temp.p, sb, thrust::make_transform_iterator(static_cast<const uint64_t*>(a.cap), Align16{}),
                                                   a.off, int(n), st)) != cudaSuccess)
                return e;
            slot_cut_kernel<<<grid, 256, 0, st>>>(a, n, budget, ds);
            *launches += 3;
            P.dst_off = a.off;
            P.dst_cap = a.cap;
            if ((e = cudaMemsetAsync(ticket, 0, 64, st)) != cudaSuccess || (e = launch_decode(P, sm_count, st)) != cudaSuccess) return e;
            *launches += 1;
        }
        walk_kernel<<<1, 32, 0, st>>>(a, n, items, len, ds, max_found, dst_bytes, d_start, d_consumed, d_out_len, d_dst_off);
        *launches += 1;
        if (n > 0) {
            gather_kernel<<<kGatherBlocks, 256, 0, st>>>(slots, a, ds, d_out_len, d_dst_off, d_dst_base);
            *launches += 1;
        }
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        // a window with more hits than a round keeps is tested again from where the round stopped: narrow it
        if (hs.nsel > kRoundHits) window = window / 2 > kWindowMin ? window / 2 : kWindowMin;
        else window = window < kWindowMax / 2 ? window * 2 : kWindowMax;
        p_known = hs.p;
    }
    *found = hs.found;
    *next = hs.p < len ? hs.p : len;
    return cudaSuccess;
}

}  // namespace aurora
