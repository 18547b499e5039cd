// tests/simt/scan_walk_harness.cpp — the offset walk of aurora_scan_decode_device (walk_round in csrc/scan_decode.cu,
// everything above its "// ---- kernel" line, cut out of the real file by tests/test_scan_walk_simt.py), compiled for the CPU
// and driven through rounds the way scan_decode_rounds drives it: a window of the hit table from the walk position, at most
// `keep` hits kept, slots cut at `budget` bytes of capacity.  TEST INFRASTRUCTURE.
#include "common.cuh"
#include SCAN_WALK_INC   // leaves `namespace aurora {` open
}  // namespace aurora

#include <algorithm>
#include <vector>

// hit[0 .. nhits): ascending hit positions with their decode outcome; cap: each hit's slot size.  Writes the entries, *found,
// *next and the number of rounds.
extern "C" void simt_scan_walk(uint64_t len, uint64_t begin, const uint64_t* hit, const int32_t* status, const uint64_t* consumed,
                               const uint64_t* out_len, const uint64_t* cap, uint32_t nhits, uint64_t window, uint32_t keep,
                               uint64_t budget, uint64_t max_found, uint64_t dst_bytes, uint64_t* e_start, uint64_t* e_consumed,
                               uint64_t* e_len, uint64_t* e_off, uint64_t* found, uint64_t* next, uint64_t* rounds) {
    aurora::WalkState s{};
    s.p = begin;
    *rounds = 0;
    while (!s.stopped && s.p < len) {
        ++*rounds;
        const uint64_t wend = std::min(s.p + window, len);
        const uint32_t b = uint32_t(std::lower_bound(hit, hit + nhits, s.p) - hit);
        const uint32_t nsel = uint32_t(std::lower_bound(hit, hit + nhits, wend) - hit) - b;
        const uint32_t n = std::min(nsel, keep);
        uint32_t known = n;
        uint64_t off = 0;
        for (uint32_t k = 0; k < n; k++) {   // the slot cut
            if (off + cap[b + k] > budget) {
                known = k;
                break;
            }
            off += aurora::scan_align16(cap[b + k]);
        }
        aurora::WalkRound r;
        r.hit = hit + b;
        r.status = status + b;
        r.consumed = consumed + b;
        r.out_len = out_len + b;
        r.n = known;
        r.len = len;
        r.end = known < n ? r.hit[known] : n < nsel ? r.hit[n - 1] + 1 : wend;
        auto first_ok = [&](uint32_t k, uint64_t t) {
            while (k < r.n && !(r.status[k] == AURORA_OK && r.hit[k] >= t)) k++;
            return k;
        };
        auto emit = [&](uint32_t k, uint64_t e, uint64_t dst_off) {
            e_start[e] = r.hit[k];
            e_consumed[e] = r.consumed[k];
            e_len[e] = r.out_len[k];
            e_off[e] = dst_off;
        };
        aurora::walk_round(r, s, max_found, dst_bytes, first_ok, emit);
    }
    *found = s.found;
    *next = std::min(s.p, len);
}

extern "C" uint64_t simt_walk_target(uint64_t start, int32_t status, uint64_t consumed) { return aurora::walk_target(start, status, consumed); }
