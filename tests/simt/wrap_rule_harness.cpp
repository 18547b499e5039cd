// tests/simt/wrap_rule_harness.cpp — the wrapper rules as both aurora_decode_batch and the device's wrapper kernels run them
// (wrap_resolve, wrap_chunk, wrap_merge and wrap_redo_chunk in csrc/wrappers.cu, everything above its "// ---- kernel" line,
// cut out of the real file by tests/test_wrap_rule_simt.py), compiled for the CPU.  Plans and sub-streams travel as u64
// arrays in field order.  TEST INFRASTRUCTURE.
#include "common.cuh"
#include WRAPPERS_DEVICE_INC   // leaves `namespace aurora {` open
}  // namespace aurora

using aurora::WrapPlan;
using aurora::WrapSub;

static void put_plan(const WrapPlan& p, uint64_t* o) {
    const uint64_t v[10] = {uint64_t(p.status), p.consumed, p.out_len, p.expect, p.end_consumed, p.chunks, p.table, p.copy_off, p.copy_len, p.fill_len};
    for (int k = 0; k < 10; k++) o[k] = v[k];
}
static WrapPlan get_plan(const uint64_t* o) { return WrapPlan{int(o[0]), o[1], o[2], o[3], o[4], o[5], o[6], o[7], o[8], o[9]}; }
static void put_sub(const WrapSub& s, uint64_t* o) {
    const uint64_t v[6] = {uint64_t(s.core), s.off, s.len, s.doff, s.raw, s.key};
    for (int k = 0; k < 6; k++) o[k] = v[k];
}
static WrapSub get_sub(const uint64_t* o) { return WrapSub{int(o[0]), o[1], o[2], o[3], o[4], uint32_t(o[5])}; }

// plan (10 words) and sub-streams (6 words each: the one sub-stream, or every ChunkLZ10 chunk); returns the number of
// sub-streams written (at most max_sub), or -1 when there are more
extern "C" int64_t simt_wrap_resolve(int format, const uint8_t* p, uint64_t len, uint64_t cap, uint64_t* plan, uint64_t* subs, uint64_t max_sub) {
    WrapPlan pl;
    WrapSub s;
    aurora::wrap_resolve(format, p, len, cap, pl, s);
    put_plan(pl, plan);
    if (!pl.chunks) {
        put_sub(s, subs);
        return s.core ? 1 : 0;
    }
    if (pl.chunks > max_sub) return -1;
    uint64_t doff = 0;
    for (uint64_t k = 0; k < pl.chunks; k++) {
        const WrapSub c = aurora::wrap_chunk(p, len, pl, k, doff);
        put_sub(c, subs + 6 * k);
        doff += aurora::wrap_chunk_size(p, c);
    }
    return int64_t(pl.chunks);
}

// out: out_len, consumed, status
extern "C" void simt_wrap_merge(int format, const uint64_t* plan, const uint64_t* subs, uint64_t n_sub, const uint64_t* r_out,
                                const uint64_t* r_cons, const int32_t* r_st, uint64_t* out) {
    const WrapPlan pl = get_plan(plan);
    std::vector<WrapSub> s(n_sub ? n_sub : 1, WrapSub{0, 0, 0, 0, 0, 0u});
    for (uint64_t k = 0; k < n_sub; k++) s[k] = get_sub(subs + 6 * k);
    uint64_t ol, cs;
    int st;
    aurora::wrap_merge(format, pl, s.data(), r_out, r_cons, r_st, ol, cs, st);
    out[0] = ol;
    out[1] = cs;
    out[2] = uint64_t(int64_t(st));
}

extern "C" int64_t simt_wrap_redo_chunk(const uint64_t* plan, const int32_t* r_st) { return aurora::wrap_redo_chunk(get_plan(plan), r_st); }
