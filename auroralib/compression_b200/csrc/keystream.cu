// keystream.cu — LZ00's StreamTransformer (AuroraLib.Compression.Sega/Sega/LZ00.cs:112-139) as a data-parallel pass.
//
// The reference wraps the compressed stream in a Stream that XORs every byte with a value derived from a 32-bit key and
// steps the key once per byte (GenerateNextKey :125-131: the shift / subtract ladder multiplies by 1103515245, then adds
// 12345 — an affine map K' = A*K + C mod 2^32).  An affine map composes in closed form, so byte i's key
// K_(i+1) = A^(i+1)*K0 + C*(A^i + ... + 1) is reachable by square-and-multiply from any position: every thread jumps to
// its first byte and then strides with the 256-step map.  Decode lifts the keystream off the LZSS body before the LZSS kernel
// reads it (the host entry point in place on its own device copy, the device entry point out of place from the caller's
// bytes into per-stream scratch slots); encode runs it in place over the body the LZSS encoder just wrote.
#include "common.cuh"

namespace aurora {

namespace {

struct Affine {
    uint32_t a, c;   // x -> a * x + c
};
__device__ __forceinline__ Affine compose(Affine f, Affine g) { return Affine{f.a * g.a, f.a * g.c + f.c}; }   // f after g
__device__ __forceinline__ Affine affine_pow(Affine f, uint64_t k) {
    Affine r{1u, 0u};
    while (k) {
        if (k & 1) r = compose(f, r);
        f = compose(f, f);
        k >>= 1;
    }
    return r;
}

constexpr int kThreads = 256;

// bytes [skip, min(len[i], cap[i])) of stream i under key[i], read at in + in_off[i] and written at out + out_off[i] (the same
// bytes when in == out and in_off == out_off); blockIdx.y cuts every stream into gridDim.y segments
__global__ void __launch_bounds__(kThreads) lcg_xor_kernel(const uint8_t* in, const uint64_t* in_off, uint8_t* out, const uint64_t* out_off,
                                                           const uint64_t* len, const uint64_t* cap, const uint32_t* key, uint32_t skip,
                                                           uint32_t n) {
    const Affine step{1103515245u, 12345u};
    const Affine stride = affine_pow(step, kThreads);
    for (uint32_t s = blockIdx.x; s < n; s += gridDim.x) {
        uint64_t end = len[s];
        if (cap && cap[s] < end) end = cap[s];   // an encoder that ran out of room reports the length it would have needed
        const uint64_t total = end > skip ? end - skip : 0;
        const uint64_t seg = ((total + gridDim.y - 1) / gridDim.y + kThreads - 1) / kThreads * kThreads;
        const uint64_t lo = seg * blockIdx.y, hi = lo + seg < total ? lo + seg : total;
        uint64_t i = lo + threadIdx.x;
        if (i >= hi) continue;
        const uint8_t* p = in + in_off[s] + skip;
        uint8_t* q = out + out_off[s] + skip;
        const Affine jump = affine_pow(step, i + 1);   // Transform steps the key BEFORE it uses it
        uint32_t k = jump.a * key[s] + jump.c;
        for (; i < hi; i += kThreads) {
            const uint32_t t = (k >> 16) & 0x7FFFu;
            q[i] = uint8_t(p[i] ^ (((t << 8) - t) >> 15));
            k = stride.a * k + stride.c;
        }
    }
}

}  // namespace

cudaError_t launch_lcg_xor(const uint8_t* in, const uint64_t* d_in_off, uint8_t* out, const uint64_t* d_out_off, const uint64_t* d_len,
                           const uint64_t* d_cap, const uint32_t* d_key, uint32_t skip, uint32_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const dim3 grid(n < 4736u ? n : 4736u, n >= 1184u ? 1u : n >= 148u ? 8u : 32u);
    lcg_xor_kernel<<<grid, kThreads, 0, st>>>(in, d_in_off, out, d_out_off, d_len, d_cap, d_key, skip, n);
    return cudaGetLastError();
}

}  // namespace aurora
