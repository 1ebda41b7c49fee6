// png.cu — PNG files on the device (DESIGN.md §4, "PNG files on the device").
//
// k_png_filter   one warp per row: libpng's minimum-sum-of-absolute-differences choice of the row filter, then the
//                filtered row (filter-type byte first) into the image's filtered stream.
// k_png_deflate  one CTA per 32 KiB segment of a filtered stream, the segment in shared memory: a hash chain over
//                its positions, a greedy LZ77 parse (each thread parses its own 128 bytes, matches reach back
//                anywhere in the segment), one dynamic Huffman block with codes of at most 15 bits, bit-packed with
//                shared-memory atomicOr, or stored when that would be larger than the segment.  Every segment ends
//                with an empty stored block, byte-aligned; the last one's is BFINAL.  Also the segment's Adler sums.
// k_png_layout   one CTA: where each segment's IDAT chunk starts, every file's Adler-32 and size, and the running
//                file offsets.
// k_png_emit     one CTA per segment: its IDAT chunk (the zlib header in the first, the Adler-32 in the last) and its
//                CRC-32, which the threads compute piecewise and combine; signature and IHDR before the first
//                segment, IEND after the last.
//
// Every value that lands in a file is built from counts, prefix sums and order-independent atomics (max, add, or),
// never from the order in which threads run, so a file's bytes do not depend on the run, the batch or its place in it.
#include "png.cuh"

namespace mcskin {
namespace png {
namespace {

constexpr int kFilterWarps = 8;
constexpr int kDeflateThreads = 256;
constexpr int kSubBytes = static_cast<int>(kSegBytes) / kDeflateThreads;  // what one thread parses
constexpr int kHashBits = 12;
constexpr int kMaxChain = 4;       // hash-chain candidates tried per position (zlib level 1 tries 4)
constexpr int kNiceLength = 128;   // a match this long ends the search
constexpr uint16_t kNoPos = 0xffff;
constexpr uint32_t kAdlerMod = 65521;
constexpr int kLitLen = 286, kDist = 30, kCodeLen = 19;
constexpr int kEmitThreads = 256;
constexpr int kCrcPieceLog = 8;    // each emit thread folds 256 bytes; 256 * 256 covers the largest chunk
static_assert(kEmitThreads << kCrcPieceLog >= kSlotBytes + 16, "CRC pieces must cover an IDAT chunk");

// x^(2^k) mod the CRC-32 polynomial, reflected (zlib's x2n_table)
__constant__ uint32_t c_x2n[32] = {
    0x40000000u, 0x20000000u, 0x08000000u, 0x00800000u, 0x00008000u, 0xedb88320u, 0xb1e6b092u, 0xa06a2517u,
    0xed627daeu, 0x88d14467u, 0xd7bbfe6au, 0xec447f11u, 0x8e7ea170u, 0x6427800eu, 0x4d47bae0u, 0x09fe548fu,
    0x83852d0fu, 0x30362f1au, 0x7b5a9cc3u, 0x31fec169u, 0x9fec022au, 0x6c8dedc4u, 0x15d6874du, 0x5fde7a4eu,
    0xbad90e37u, 0x2e4e5eefu, 0x4eaba214u, 0xa8a472c0u, 0x429a969eu, 0x148d302au, 0xc40ba6d0u, 0xc4e22c3cu};

// ---------------------------------------------------------------- filters
__device__ __forceinline__ int paeth(int a, int b, int c) {
    const int p = a + b - c, pa = abs(p - a), pb = abs(p - b), pc = abs(p - c);
    return (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
}
__device__ __forceinline__ uint32_t filter_byte(int type, int x, int a, int b, int c) {
    const int pred = type == 0 ? 0 : type == 1 ? a : type == 2 ? b : type == 3 ? ((a + b) >> 1) : paeth(a, b, c);
    return static_cast<uint32_t>(x - pred) & 0xffu;
}
__device__ __forceinline__ int byte_of(uchar4 v, int k) { return k == 0 ? v.x : k == 1 ? v.y : k == 2 ? v.z : v.w; }

__global__ void __launch_bounds__(kFilterWarps * 32) k_png_filter(const uchar4* __restrict__ img, int w, int h, long long rows,
                                                                  uint8_t* __restrict__ out, unsigned long long stride) {
    const long long row = static_cast<long long>(blockIdx.x) * kFilterWarps + threadIdx.x / 32;
    if (row >= rows) return;  // (whole warps)
    const int lane = threadIdx.x & 31;
    const long long image = row / h;
    const int y = static_cast<int>(row - image * h);
    const uchar4* cur = img + row * w;
    const uchar4* up = cur - w;
    uint8_t* dst = out + image * stride + static_cast<unsigned long long>(y) * (4ull * w + 1);
    const uchar4 zero = make_uchar4(0, 0, 0, 0);
    unsigned sum[5] = {0, 0, 0, 0, 0};
    for (int x = lane; x < w; x += 32) {
        const uchar4 X = cur[x], A = x ? cur[x - 1] : zero, B = y ? up[x] : zero, Cc = (x && y) ? up[x - 1] : zero;
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int t = 0; t < 5; ++t)
                sum[t] += abs(static_cast<int>(static_cast<int8_t>(filter_byte(t, byte_of(X, k), byte_of(A, k), byte_of(B, k), byte_of(Cc, k)))));
    }
#pragma unroll
    for (int t = 0; t < 5; ++t)
        for (int o = 16; o; o >>= 1) sum[t] += __shfl_xor_sync(0xffffffffu, sum[t], o);
    int best = 0;
#pragma unroll
    for (int t = 1; t < 5; ++t)
        if (sum[t] < sum[best]) best = t;
    if (lane == 0) dst[0] = static_cast<uint8_t>(best);
    for (int x = lane; x < w; x += 32) {
        const uchar4 X = cur[x], A = x ? cur[x - 1] : zero, B = y ? up[x] : zero, Cc = (x && y) ? up[x - 1] : zero;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            dst[1 + 4 * x + k] = static_cast<uint8_t>(filter_byte(best, byte_of(X, k), byte_of(A, k), byte_of(B, k), byte_of(Cc, k)));
    }
}

// ---------------------------------------------------------------- deflate symbols (RFC 1951 §3.2.5)
// length 3..258 -> code 0..28 (symbol 257 + code), extra bits and their value
__device__ __forceinline__ void length_code(int len, int* code, int* nExtra, int* extra) {
    const int l = len - 3;
    if (l == 255) { *code = 28; *nExtra = 0; *extra = 0; return; }
    if (l < 8) { *code = l; *nExtra = 0; *extra = 0; return; }
    const int e = 31 - __clz(l) - 2;
    *code = 4 * (e + 1) + ((l >> e) & 3);
    *nExtra = e;
    *extra = l - ((4 + (*code & 3)) << e);
}
// distance 1..32768 -> code 0..29, extra bits and their value
__device__ __forceinline__ void dist_code(int dist, int* code, int* nExtra, int* extra) {
    const int x = dist - 1;
    if (x < 4) { *code = x; *nExtra = 0; *extra = 0; return; }
    const int e = 31 - __clz(x) - 1;
    *code = 2 * (e + 1) + ((x >> e) & 1);
    *nExtra = e;
    *extra = x - ((2 + (*code & 1)) << e);
}

// LSB-first bits into shared words that other threads write too (atomicOr: the result does not depend on the order)
struct BitWriter {
    uint32_t* words;
    unsigned w;
    unsigned long long acc;
    int n;
    __device__ BitWriter(uint32_t* buf, unsigned long long bitPos) : words(buf), w(static_cast<unsigned>(bitPos >> 5)), acc(0), n(bitPos & 31) {}
    __device__ void put(uint32_t v, int bits) {
        acc |= static_cast<unsigned long long>(v) << n;
        n += bits;
        while (n >= 32) {
            atomicOr(&words[w++], static_cast<uint32_t>(acc));
            acc >>= 32;
            n -= 32;
        }
    }
    __device__ void flush() {
        if (n > 0) atomicOr(&words[w], static_cast<uint32_t>(acc));
    }
};

struct DeflateSmem {
    uint32_t data[kSegBytes / 4];  // the segment; then its deflate bytes
    uint16_t prev[kSegBytes];      // the previous position of the same hash, or kNoPos
    union {
        int head[1 << kHashBits];  // while the chain is built
        struct {
            uint32_t lfreq[kLitLen], dfreq[kDist], cfreq[kCodeLen];
            uint32_t work[kLitLen];
            uint16_t lcode[kLitLen], dcode[kDist], ccode[kCodeLen];
            uint16_t sorted[kLitLen + kDist];
            uint8_t llen[kLitLen], dlen[kDist], clen[kCodeLen];
            uint8_t rleSym[kLitLen + kDist], rleExtra[kLitLen + kDist];
            uint32_t s1[kDeflateThreads], s2[kDeflateThreads];  // Adler partials, then the bit counts' scan
            uint32_t warpSum[kDeflateThreads / 32];
            int nRle, hlit, hdist, hclen;
            uint32_t hdrBits;
        } b;
    } u;
};

// Code lengths of at most maxLen bits for the symbols of `sorted` (n of them, ascending (frequency, symbol)):
// Moffat and Katajainen's in-place minimum-redundancy lengths, then lengths over maxLen folded back by
// rebalancing the length counts (the Kraft sum restored), the shortest lengths to the most frequent symbols.
__device__ void huffman_lengths(const uint32_t* freq, const uint16_t* sorted, int n, int nSym, int maxLen, uint8_t* lens,
                                uint32_t* A) {
    for (int s = 0; s < nSym; ++s) lens[s] = 0;
    if (n == 0) return;
    if (n == 1) {
        lens[sorted[0]] = 1;
        return;
    }
    for (int i = 0; i < n; ++i) A[i] = freq[sorted[i]];
    A[0] += A[1];
    int root = 0, leaf = 2;
    for (int next = 1; next < n - 1; ++next) {
        if (leaf >= n || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = next; }
        else A[next] = A[leaf++];
        if (leaf >= n || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = next; }
        else A[next] += A[leaf++];
    }
    A[n - 2] = 0;
    for (int next = n - 3; next >= 0; --next) A[next] = A[A[next]] + 1;
    int avail = 1, used = 0, depth = 0;
    root = n - 2;
    int next = n - 1;
    while (avail > 0) {
        while (root >= 0 && static_cast<int>(A[root]) == depth) { ++used; --root; }
        while (avail > used) { A[next--] = depth; --avail; }
        avail = 2 * used;
        ++depth;
        used = 0;
    }
    int count[33] = {0};
    for (int i = 0; i < n; ++i) ++count[min(static_cast<int>(A[i]), 32)];
    for (int l = maxLen + 1; l <= 32; ++l) { count[maxLen] += count[l]; count[l] = 0; }
    uint32_t total = 0;
    for (int l = maxLen; l > 0; --l) total += static_cast<uint32_t>(count[l]) << (maxLen - l);
    while (total != (1u << maxLen)) {
        --count[maxLen];
        for (int l = maxLen - 1; l > 0; --l)
            if (count[l]) {
                --count[l];
                count[l + 1] += 2;
                break;
            }
        --total;
    }
    int j = n;
    for (int l = 1; l <= maxLen; ++l)
        for (int c = count[l]; c > 0; --c) lens[sorted[--j]] = static_cast<uint8_t>(l);
}

// canonical codes (RFC 1951 §3.2.2), bit-reversed for LSB-first output
__device__ void canonical_codes(const uint8_t* lens, int nSym, uint16_t* codes) {
    int count[16] = {0}, next[16];
    for (int s = 0; s < nSym; ++s) ++count[lens[s]];
    count[0] = 0;
    int code = 0;
    for (int b = 1; b < 16; ++b) {
        code = (code + count[b - 1]) << 1;
        next[b] = code;
    }
    for (int s = 0; s < nSym; ++s)
        codes[s] = lens[s] ? static_cast<uint16_t>(__brev(static_cast<unsigned>(next[lens[s]]++)) >> (32 - lens[s])) : 0;
}

__device__ __forceinline__ uint32_t hash3(const uint8_t* d, int p) {
    const uint32_t v = (static_cast<uint32_t>(d[p]) << 16) | (static_cast<uint32_t>(d[p + 1]) << 8) | d[p + 2];
    return (v * 2654435761u) >> (32 - kHashBits);
}

__global__ void __launch_bounds__(kDeflateThreads, 2) k_png_deflate(const uint8_t* __restrict__ filtered, unsigned long long stride,
                                                                    unsigned long long L, int nSeg, uint32_t* __restrict__ tokens,
                                                                    uint8_t* __restrict__ slots, uint32_t* __restrict__ segBytes,
                                                                    uint2* __restrict__ segAdler) {
    extern __shared__ __align__(16) unsigned char smemRaw[];
    DeflateSmem& sm = *reinterpret_cast<DeflateSmem*>(smemRaw);
    const int tid = threadIdx.x;
    const long long seg = blockIdx.x;
    const long long image = seg / nSeg;
    const int k = static_cast<int>(seg - image * nSeg);
    const bool last = k == nSeg - 1;
    const int segLen = static_cast<int>(min(static_cast<unsigned long long>(kSegBytes), L - static_cast<unsigned long long>(k) * kSegBytes));
    const uint4* src = reinterpret_cast<const uint4*>(filtered + image * stride + static_cast<unsigned long long>(k) * kSegBytes);
    for (int j = tid; j < (segLen + 15) / 16; j += kDeflateThreads) reinterpret_cast<uint4*>(sm.data)[j] = src[j];
    for (int j = tid; j < (1 << kHashBits); j += kDeflateThreads) sm.u.head[j] = -1;
    __syncthreads();
    const uint8_t* d = reinterpret_cast<const uint8_t*>(sm.data);

    // hash chain, a block of positions at a time: the nearest earlier lane of the warp with the same hash, else
    // the latest position of an earlier block (atomicMax)
    const int lane = tid & 31;
    for (int base = 0; base < segLen; base += kDeflateThreads) {
        const int p = base + tid;
        const bool hashed = p + 2 < segLen;
        const uint32_t h = hashed ? hash3(d, p) : (1u << kHashBits) + lane;
        const unsigned same = __match_any_sync(0xffffffffu, h);
        if (hashed) {
            const unsigned lower = same & ((1u << lane) - 1);
            const int q = lower ? p - lane + (31 - __clz(lower)) : sm.u.head[h];
            sm.prev[p] = q < 0 ? kNoPos : static_cast<uint16_t>(q);
        } else if (p < segLen) {
            sm.prev[p] = kNoPos;
        }
        __syncthreads();
        if (hashed && (same >> lane) == 1u) atomicMax(&sm.u.head[h], p);
        __syncthreads();
    }
    for (int j = tid; j < kLitLen; j += kDeflateThreads) sm.u.b.lfreq[j] = j == 256 ? 1 : 0;
    if (tid < kDist) sm.u.b.dfreq[tid] = 0;
    if (tid < kCodeLen) sm.u.b.cfreq[tid] = 0;
    __syncthreads();

    // greedy parse of this thread's bytes; tokens: literal byte, or (distance << 16 | length)
    const int begin = min(tid * kSubBytes, segLen), end = min(begin + kSubBytes, segLen);
    uint32_t* tok = tokens + seg * kSegBytes + tid * kSubBytes;
    int nTok = 0;
    {
        uint32_t s1 = 0, s2 = 0;
        for (int p = begin; p < end; ++p) {
            s1 += d[p];
            s2 += static_cast<uint32_t>(end - p) * d[p];
        }
        sm.u.b.s1[tid] = s1 % kAdlerMod;
        sm.u.b.s2[tid] = s2 % kAdlerMod;
    }
    for (int p = begin; p < end;) {
        const int limit = min(258, end - p);
        int bestLen = 0, bestDist = 0;
        if (limit >= 3) {
            int q = sm.prev[p];
            for (int c = 0; c < kMaxChain && q != kNoPos; ++c) {
                if (d[q + bestLen] == d[p + bestLen]) {
                    int l = 0;
                    while (l < limit && d[q + l] == d[p + l]) ++l;
                    if (l > bestLen) {
                        bestLen = l;
                        bestDist = p - q;
                        if (l >= limit || l >= kNiceLength) break;
                    }
                }
                q = sm.prev[q];
            }
        }
        if (bestLen >= 3) {
            tok[nTok++] = (static_cast<uint32_t>(bestDist) << 16) | static_cast<uint32_t>(bestLen);
            int lc, ne, ev;
            length_code(bestLen, &lc, &ne, &ev);
            atomicAdd(&sm.u.b.lfreq[257 + lc], 1u);
            dist_code(bestDist, &lc, &ne, &ev);
            atomicAdd(&sm.u.b.dfreq[lc], 1u);
            p += bestLen;
        } else {
            tok[nTok++] = d[p];
            atomicAdd(&sm.u.b.lfreq[d[p]], 1u);
            ++p;
        }
    }
    __syncthreads();

    // code lengths: rank every used symbol by (frequency, symbol), then one thread builds the codes
    for (int j = tid; j < kLitLen + kDist; j += kDeflateThreads) {
        const bool lit = j < kLitLen;
        const uint32_t* f = lit ? sm.u.b.lfreq : sm.u.b.dfreq;
        const int s = lit ? j : j - kLitLen, n = lit ? kLitLen : kDist;
        if (f[s]) {
            int rank = 0;
            for (int o = 0; o < n; ++o) rank += f[o] && (f[o] < f[s] || (f[o] == f[s] && o < s));
            sm.u.b.sorted[(lit ? 0 : kLitLen) + rank] = static_cast<uint16_t>(s);
        }
    }
    __syncthreads();
    if (tid == 32) {
        // the segment's Adler sums: S1(AB) = S1(A) + S1(B), S2(AB) = S2(A) + |B| S1(A) + S2(B)
        unsigned long long S1 = 0, S2 = 0;
        for (int t = 0; t < kDeflateThreads; ++t) {
            const int len = min((t + 1) * kSubBytes, segLen) - min(t * kSubBytes, segLen);
            S2 = (S2 + static_cast<unsigned long long>(len) * S1 + sm.u.b.s2[t]) % kAdlerMod;
            S1 = (S1 + sm.u.b.s1[t]) % kAdlerMod;
        }
        segAdler[seg] = make_uint2(static_cast<uint32_t>(S1), static_cast<uint32_t>(S2));
    }
    if (tid == 0) {
        auto& b = sm.u.b;
        int nL = 0, nD = 0;
        for (int s = 0; s < kLitLen; ++s) nL += b.lfreq[s] != 0;
        for (int s = 0; s < kDist; ++s) nD += b.dfreq[s] != 0;
        huffman_lengths(b.lfreq, b.sorted, nL, kLitLen, 15, b.llen, b.work);
        huffman_lengths(b.dfreq, b.sorted + kLitLen, nD, kDist, 15, b.dlen, b.work);
        if (nD == 0) b.dlen[0] = 1;  // one distance code of one bit: no match in the block
        canonical_codes(b.llen, kLitLen, b.lcode);
        canonical_codes(b.dlen, kDist, b.dcode);
        int hlit = kLitLen, hdist = kDist;
        while (hlit > 257 && !b.llen[hlit - 1]) --hlit;
        while (hdist > 1 && !b.dlen[hdist - 1]) --hdist;
        // run-length code of the code lengths (16: repeat the previous 3-6 times, 17: 3-10 zeros, 18: 11-138 zeros)
        int nRle = 0;
        auto emit = [&](int sym, int extra) {
            b.rleSym[nRle] = static_cast<uint8_t>(sym);
            b.rleExtra[nRle++] = static_cast<uint8_t>(extra);
            ++b.cfreq[sym];
        };
        const int nLens = hlit + hdist;
        for (int i = 0; i < nLens;) {
            const int v = i < hlit ? b.llen[i] : b.dlen[i - hlit];
            int r = 1;
            while (i + r < nLens && (i + r < hlit ? b.llen[i + r] : b.dlen[i + r - hlit]) == v) ++r;
            i += r;
            if (v == 0) {
                while (r >= 11) { const int m = min(r, 138); emit(18, m - 11); r -= m; }
                if (r >= 3) { emit(17, r - 3); r = 0; }
            } else {
                emit(v, 0);
                --r;
                while (r >= 3) { const int m = min(r, 6); emit(16, m - 3); r -= m; }
            }
            while (r-- > 0) emit(v, 0);
        }
        // code-length code: at most 7 bits, complete (a lone symbol gets a partner)
        int nC = 0;
        for (int s = 0; s < kCodeLen; ++s)
            if (b.cfreq[s]) {
                int j = nC++;
                while (j > 0 && b.cfreq[b.sorted[j - 1]] > b.cfreq[s]) { b.sorted[j] = b.sorted[j - 1]; --j; }
                b.sorted[j] = static_cast<uint16_t>(s);
            }
        huffman_lengths(b.cfreq, b.sorted, nC, kCodeLen, 7, b.clen, b.work);
        if (nC == 1) b.clen[b.sorted[0] == 0 ? 1 : 0] = 1;
        canonical_codes(b.clen, kCodeLen, b.ccode);
        constexpr uint8_t kOrder[kCodeLen] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        int hclen = kCodeLen;
        while (hclen > 4 && !b.clen[kOrder[hclen - 1]]) --hclen;
        uint32_t bits = 3 + 5 + 5 + 4 + 3 * hclen;
        for (int i = 0; i < nRle; ++i) {
            const int s = b.rleSym[i];
            bits += b.clen[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
        }
        b.nRle = nRle;
        b.hlit = hlit;
        b.hdist = hdist;
        b.hclen = hclen;
        b.hdrBits = bits;
    }
    __syncthreads();

    // this thread's bits, and where they start: an exclusive scan over the threads
    uint32_t myBits = 0;
    for (int i = 0; i < nTok; ++i) {
        const uint32_t t = tok[i];
        if (t < 256) {
            myBits += sm.u.b.llen[t];
        } else {
            int lc, ne, ev, dc, de, dv;
            length_code(t & 0xffff, &lc, &ne, &ev);
            dist_code(t >> 16, &dc, &de, &dv);
            myBits += sm.u.b.llen[257 + lc] + ne + sm.u.b.dlen[dc] + de;
        }
    }
    uint32_t incl = myBits;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) sm.u.b.warpSum[tid / 32] = incl;
    __syncthreads();
    uint32_t before = 0, body = 0;
    for (int w = 0; w < kDeflateThreads / 32; ++w) {
        if (w < tid / 32) before += sm.u.b.warpSum[w];
        body += sm.u.b.warpSum[w];
    }
    const unsigned long long start = sm.u.b.hdrBits + before + (incl - myBits);
    const unsigned long long eobAt = sm.u.b.hdrBits + static_cast<unsigned long long>(body);
    const unsigned long long dynBits = eobAt + sm.u.b.llen[256] + 3;  // + the empty stored block's header
    const uint32_t dynBytes = static_cast<uint32_t>((dynBits + 7) / 8 + 4);
    uint8_t* slot = slots + seg * kSlotBytes;
    if (dynBytes > static_cast<uint32_t>(segLen)) {
        // stored: [BFINAL 0, BTYPE 00] LEN NLEN data, then the empty stored block
        const uint32_t len = segLen, nlen = ~len & 0xffffu;
        for (int j = tid; j < segLen; j += kDeflateThreads) slot[5 + j] = d[j];
        if (tid == 0) {
            const uint8_t head[5] = {0, static_cast<uint8_t>(len), static_cast<uint8_t>(len >> 8), static_cast<uint8_t>(nlen),
                                     static_cast<uint8_t>(nlen >> 8)};
            for (int j = 0; j < 5; ++j) slot[j] = head[j];
            const uint8_t tail[5] = {static_cast<uint8_t>(last ? 1 : 0), 0, 0, 0xff, 0xff};
            for (int j = 0; j < 5; ++j) slot[5 + segLen + j] = tail[j];
            segBytes[seg] = segLen + 10;
        }
        return;
    }
    __syncthreads();  // every read of the segment's bytes is done: the buffer takes the bits
    for (int j = tid; j < static_cast<int>((dynBytes + 3) / 4); j += kDeflateThreads) sm.data[j] = 0;
    __syncthreads();
    {
        const auto& b = sm.u.b;
        if (tid == 0) {
            BitWriter bw(sm.data, 0);
            bw.put(2u << 1, 3);  // BFINAL 0, BTYPE 10 (dynamic)
            bw.put(b.hlit - 257, 5);
            bw.put(b.hdist - 1, 5);
            bw.put(b.hclen - 4, 4);
            constexpr uint8_t kOrder[kCodeLen] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
            for (int i = 0; i < b.hclen; ++i) bw.put(b.clen[kOrder[i]], 3);
            for (int i = 0; i < b.nRle; ++i) {
                const int s = b.rleSym[i];
                bw.put(b.ccode[s], b.clen[s]);
                if (s >= 16) bw.put(b.rleExtra[i], s == 16 ? 2 : s == 17 ? 3 : 7);
            }
            bw.flush();
        }
        BitWriter bw(sm.data, start);
        for (int i = 0; i < nTok; ++i) {
            const uint32_t t = tok[i];
            if (t < 256) {
                bw.put(b.lcode[t], b.llen[t]);
            } else {
                int lc, ne, ev, dc, de, dv;
                length_code(t & 0xffff, &lc, &ne, &ev);
                dist_code(t >> 16, &dc, &de, &dv);
                bw.put(b.lcode[257 + lc], b.llen[257 + lc]);
                if (ne) bw.put(ev, ne);
                bw.put(b.dcode[dc], b.dlen[dc]);
                if (de) bw.put(dv, de);
            }
        }
        bw.flush();
        if (tid == kDeflateThreads - 1) {
            BitWriter eob(sm.data, eobAt);
            eob.put(b.lcode[256], b.llen[256]);
            eob.put(last ? 1 : 0, 3);  // the empty stored block: BFINAL on the last segment, BTYPE 00
            eob.flush();
        }
    }
    __syncthreads();
    if (tid == 0) {
        uint8_t* bytes = reinterpret_cast<uint8_t*>(sm.data);
        bytes[dynBytes - 4] = 0;
        bytes[dynBytes - 3] = 0;
        bytes[dynBytes - 2] = 0xff;
        bytes[dynBytes - 1] = 0xff;
        segBytes[seg] = dynBytes;
    }
    __syncthreads();
    for (int j = tid; j < static_cast<int>((dynBytes + 3) / 4); j += kDeflateThreads) reinterpret_cast<uint32_t*>(slot)[j] = sm.data[j];
}

// ---------------------------------------------------------------- layout
constexpr int kLayoutThreads = 1024;

__global__ void __launch_bounds__(kLayoutThreads) k_png_layout(const uint32_t* __restrict__ segBytes, const uint2* __restrict__ segAdler,
                                                               int n, int nSeg, unsigned long long L,
                                                               unsigned long long* __restrict__ segOff, uint32_t* __restrict__ imgAdler,
                                                               unsigned long long* __restrict__ offsets, bool first) {
    __shared__ unsigned long long scan[kLayoutThreads];
    unsigned long long base = first ? 0 : offsets[0];
    if (first && threadIdx.x == 0) offsets[0] = 0;
    for (int c0 = 0; c0 < n; c0 += kLayoutThreads) {
        const int i = c0 + threadIdx.x;
        unsigned long long size = 0;
        if (i < n) {
            unsigned long long off = 8 + 25, S1 = 0, S2 = 0;
            for (int k = 0; k < nSeg; ++k) {
                const long long s = static_cast<long long>(i) * nSeg + k;
                segOff[s] = off;
                off += 12 + segBytes[s] + (k == 0 ? 2 : 0) + (k == nSeg - 1 ? 4 : 0);
                const unsigned long long len = min(static_cast<unsigned long long>(kSegBytes), L - static_cast<unsigned long long>(k) * kSegBytes);
                S2 = (S2 + len % kAdlerMod * S1 + segAdler[s].y) % kAdlerMod;
                S1 = (S1 + segAdler[s].x) % kAdlerMod;
            }
            const uint32_t a = static_cast<uint32_t>((1 + S1) % kAdlerMod), b = static_cast<uint32_t>((L % kAdlerMod + S2) % kAdlerMod);
            imgAdler[i] = (b << 16) | a;
            size = off + 12;
        }
        scan[threadIdx.x] = size;
        __syncthreads();
        for (int o = 1; o < kLayoutThreads; o <<= 1) {
            const unsigned long long v = threadIdx.x >= o ? scan[threadIdx.x - o] : 0;
            __syncthreads();
            scan[threadIdx.x] += v;
            __syncthreads();
        }
        if (i < n) offsets[1 + i] = base + scan[threadIdx.x];
        base += scan[kLayoutThreads - 1];
        __syncthreads();
    }
}

// ---------------------------------------------------------------- chunks and CRC-32
// a * b modulo the CRC-32 polynomial (reflected; zlib's multmodp)
__device__ uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}
// x^(n * 2^k) modulo the polynomial
__device__ uint32_t x2nmodp(unsigned long long n, int k) {
    uint32_t p = 1u << 31;
    for (; n; n >>= 1, ++k)
        if (n & 1) p = multmodp(c_x2n[k & 31], p);
    return p;
}

__device__ __forceinline__ void put_be32(uint8_t* p, uint32_t v) {
    p[0] = static_cast<uint8_t>(v >> 24);
    p[1] = static_cast<uint8_t>(v >> 16);
    p[2] = static_cast<uint8_t>(v >> 8);
    p[3] = static_cast<uint8_t>(v);
}

__global__ void __launch_bounds__(kEmitThreads) k_png_emit(const uint8_t* __restrict__ slots, const uint32_t* __restrict__ segBytes,
                                                           const unsigned long long* __restrict__ segOff, const uint32_t* __restrict__ imgAdler,
                                                           int nSeg, int w, int h, const unsigned long long* __restrict__ offsets,
                                                           uint8_t* __restrict__ png) {
    __shared__ uint32_t table[256];
    __shared__ uint32_t warpCrc[kEmitThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31;
    {
        uint32_t c = tid;
        for (int j = 0; j < 8; ++j) c = c & 1 ? (c >> 1) ^ 0xedb88320u : c >> 1;
        table[tid] = c;
    }
    const long long seg = blockIdx.x;
    const long long image = seg / nSeg;
    const int k = static_cast<int>(seg - image * nSeg);
    uint8_t* file = png + offsets[image];
    uint8_t* chunk = file + segOff[seg];
    const uint8_t* slot = slots + seg * kSlotBytes;
    const int zh = k == 0 ? 2 : 0, sb = static_cast<int>(segBytes[seg]), ad = k == nSeg - 1 ? 4 : 0;
    const int plen = zh + sb + ad, nMsg = 4 + plen;  // the CRC covers the chunk type and data
    const uint32_t adler = ad ? imgAdler[image] : 0;
    auto byte_at = [&](int j) -> uint32_t {
        if (j < 4) return "IDAT"[j];
        j -= 4;
        if (j < zh) return j == 0 ? 0x78 : 0x01;  // deflate, 32 KiB window, no dictionary, "fastest"
        j -= zh;
        if (j < sb) return slot[j];
        j -= sb;
        return (adler >> (24 - 8 * j)) & 0xff;
    };
    for (int j = tid; j < nMsg; j += kEmitThreads) chunk[4 + j] = static_cast<uint8_t>(byte_at(j));
    __syncthreads();  // (the table)
    // the message, zero-padded at the front to kEmitThreads equal pieces: leading zeros leave a CRC register of 0 at
    // 0, so every piece's register can be combined with fixed shifts
    constexpr int kPiece = 1 << kCrcPieceLog;
    const int pad = (kEmitThreads << kCrcPieceLog) - nMsg;
    uint32_t crc = 0;
    for (int v = max(tid * kPiece, pad); v < (tid + 1) * kPiece; ++v) crc = table[(crc ^ byte_at(v - pad)) & 0xff] ^ (crc >> 8);
    for (int o = 1, lg = 0; o < 32; o <<= 1, ++lg) {
        const uint32_t right = __shfl_down_sync(0xffffffffu, crc, o);
        if ((lane & (2 * o - 1)) == 0) crc = multmodp(c_x2n[3 + kCrcPieceLog + lg], crc) ^ right;
    }
    if (lane == 0) warpCrc[tid / 32] = crc;
    __syncthreads();
    if (tid == 0) {
        crc = warpCrc[0];
        for (int wi = 1; wi < kEmitThreads / 32; ++wi) crc = multmodp(c_x2n[3 + kCrcPieceLog + 5], crc) ^ warpCrc[wi];
        // from the register of the whole message to the CRC with its all-ones start and final inversion
        crc = ~(multmodp(x2nmodp(static_cast<unsigned long long>(nMsg), 3), 0xffffffffu) ^ crc);
        put_be32(chunk, static_cast<uint32_t>(plen));
        put_be32(chunk + 8 + plen, crc);
        if (k == 0) {
            const uint8_t sig[8] = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1a, '\n'};
            for (int j = 0; j < 8; ++j) file[j] = sig[j];
            uint8_t ihdr[4 + 4 + 13];
            put_be32(ihdr, 13);
            ihdr[4] = 'I'; ihdr[5] = 'H'; ihdr[6] = 'D'; ihdr[7] = 'R';
            put_be32(ihdr + 8, static_cast<uint32_t>(w));
            put_be32(ihdr + 12, static_cast<uint32_t>(h));
            ihdr[16] = 8;   // bit depth
            ihdr[17] = 6;   // RGBA
            ihdr[18] = 0;   // deflate
            ihdr[19] = 0;   // adaptive filtering
            ihdr[20] = 0;   // no interlace
            uint32_t c = 0xffffffffu;
            for (int j = 4; j < 21; ++j) c = table[(c ^ ihdr[j]) & 0xff] ^ (c >> 8);
            for (int j = 0; j < 21; ++j) file[8 + j] = ihdr[j];
            put_be32(file + 8 + 21, ~c);
        }
        if (k == nSeg - 1) {
            const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xae, 0x42, 0x60, 0x82};
            uint8_t* at = png + offsets[image + 1] - 12;
            for (int j = 0; j < 12; ++j) at[j] = iend[j];
        }
    }
}

}  // namespace

cudaError_t encode(const uint8_t* rgba, int32_t w, int32_t h, int32_t n, const Scratch& s, uint8_t* png,
                   unsigned long long* offsets, bool first, cudaStream_t stream) {
    const long long rows = static_cast<long long>(n) * h;
    const unsigned long long L = filtered_bytes(w, h), stride = filtered_stride(w, h);
    const int nSeg = static_cast<int>(segments(w, h));
    const long long nTotal = static_cast<long long>(n) * nSeg;
    k_png_filter<<<static_cast<unsigned>((rows + kFilterWarps - 1) / kFilterWarps), kFilterWarps * 32, 0, stream>>>(
        reinterpret_cast<const uchar4*>(rgba), w, h, rows, s.filtered, stride);
    constexpr int smem = sizeof(DeflateSmem);
    static_assert(smem <= 113 * 1024, "two deflate CTAs per SM");
    cudaError_t e = cudaFuncSetAttribute(k_png_deflate, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    k_png_deflate<<<static_cast<unsigned>(nTotal), kDeflateThreads, smem, stream>>>(s.filtered, stride, L, nSeg, s.tokens, s.slots,
                                                                                  s.segBytes, s.segAdler);
    k_png_layout<<<1, kLayoutThreads, 0, stream>>>(s.segBytes, s.segAdler, n, nSeg, L, s.segOff, s.imgAdler, offsets, first);
    k_png_emit<<<static_cast<unsigned>(nTotal), kEmitThreads, 0, stream>>>(s.slots, s.segBytes, s.segOff, s.imgAdler, nSeg, w, h,
                                                                         offsets, png);
    return cudaGetLastError();
}

}  // namespace png
}  // namespace mcskin
