// tests/simt/wrap_encode_rule_harness.cpp — the wrapper encode rules as aurora_encode_batch and the device's wrapper encode
// kernels run them (wrap_encode_opts, wrap_encode_plan, wrap_encode_piece, wrap_encode_finish, wrap_encode_chunk_move,
// wrap_encode_table and wrap_encode_header in csrc/wrappers.cu, everything above its "// ---- kernel" line, cut out of the real
// file by tests/test_wrap_encode_rule_simt.py), compiled for the CPU.  The finish rule is applied to a caller's window with
// memcpy / memmove in the order aurora_encode_batch applies it.  TEST INFRASTRUCTURE.
#include <cstring>

#include "common.cuh"
#include WRAPPERS_DEVICE_INC   // leaves `namespace aurora {` open
}  // namespace aurora

using namespace aurora;

// info: status, stored, chunked, pieces, core, head; pieces: soff, slen, doff, dcap per piece.  Returns the number of pieces
// written, -1 when there are more than max_pieces, -2 for a format that is not a wrapper.
extern "C" int64_t simt_wrap_encode_plan(int format, const aurora_codec_opts* o, uint64_t len, uint64_t cap, int64_t* info, uint64_t* pieces,
                                         uint64_t max_pieces) {
    WrapEnc e;
    if (!wrap_encode_opts(format, *o, e)) return -2;
    const WrapEncPlan pl = wrap_encode_plan(e, len, cap);
    const int64_t v[6] = {pl.status, pl.stored, pl.chunked, int64_t(pl.pieces), e.core, int64_t(e.head)};
    for (int k = 0; k < 6; k++) info[k] = v[k];
    if (pl.pieces > max_pieces) return -1;
    for (uint64_t k = 0; k < pl.pieces; k++) {
        const WrapEncPiece pc = wrap_encode_piece(e, pl, k);
        const uint64_t w[4] = {pc.soff, pc.slen, pc.doff, pc.dcap};
        for (int q = 0; q < 4; q++) pieces[4 * k + q] = w[q];
    }
    return int64_t(pl.pieces);
}

// d: the stream's destination window with the pieces' core outputs in place; src: its raw bytes.  out: out_len, status.
extern "C" void simt_wrap_encode_finish(int format, const aurora_codec_opts* o, uint64_t len, uint64_t cap, const uint64_t* r_out,
                                        const int32_t* r_st, const uint8_t* src, uint8_t* d, int64_t* out) {
    WrapEnc e;
    wrap_encode_opts(format, *o, e);
    const WrapEncPlan pl = wrap_encode_plan(e, len, cap);
    const WrapEncFin f = wrap_encode_finish(e, pl, r_out, r_st);
    if (f.copy_len) std::memcpy(d + f.copy_dst, src + f.copy_src, size_t(f.copy_len));
    if (f.move_len) std::memmove(d + f.move_dst, d + f.move_src, size_t(f.move_len));
    uint64_t end = 0;
    for (uint64_t k = 0; k < f.chunks; k++) {
        const WrapMove mv = wrap_encode_chunk_move(e, pl, k, r_out[k], end);
        std::memmove(d + mv.dst, d + mv.src, size_t(mv.len));
        wrap_encode_table(d, k, end);
    }
    wrap_encode_header(e, pl, f, d);
    out[0] = int64_t(f.out_len);
    out[1] = f.status;
}
