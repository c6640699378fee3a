// scl_lut_warp: the specialised kernel for the LUT SC / SCL / CRC-aided SCL decoders
// and their Fast-SSC variants (SCLUTDecoder, SCLLUTDecoder, CASCLLUTDecoder, FastSCLUTDecoder, FastSCLLUTDecoder,
// CAFastSCLLUTDecoder -- SURVEY.md 8a rows a10, a12, a14, a16, a18, a19; a14 is the north-star shape).
//
// Mapping: one warp decodes 32/L codewords at once, ONE LANE PER LIST PATH (L in {1,2,4,8}); the tree walk is
// the same for every frame, so the whole warp runs one uniform instruction stream and never diverges.
//   * symbols are 4-bit (table dims <= 16) and packed 8 per 32-bit word; level d of a path lives in shared
//     memory at V[(voff[d]+w)*32 + slot_lane]  (lane-interleaved: conflict-free for any slot permutation);
//   * partial sums are bits, stored IN PLACE in an N-bit array per slot: X[w*32 + slot_lane];
//   * list permutations copy nothing: two 4-bit-per-level pointer words per lane say which physical slot
//     holds level d of this logical path (values) / the left-child partial sums of level d; every f/g/combine
//     writes the lane's OWN slot and re-points that level to itself (lazy copy-on-write);
//   * f / g lookups: the 16x16 nibble table of the node is ONE 32-bit register per lane (128 B per warp) and a
//     lookup is a warp shuffle + shift (no bank conflicts, no shared memory);
//   * every table / LLR row is consumed exactly once per pass and in a fixed order, so the host lays them out
//     as one linear stream of 128-byte lines, which every warp brings on chip through a private 4-chunk ring that
//     its lanes fill with cp.async;
//   * fork: 2L path metrics ranked with a stable (key,index) count -- identical to libstdc++'s insertion sort
//     for 2L <= 16 (PD/src/SCLLUTDecoder.cpp:8-22, SURVEY App. B1);
//   * schedule: persistent CTAs of 4 warps that take frame groups from a counter in the workspace (dynamic);
//   * code size matters as much as instruction count: an SM's warps sit all over the walk, the instruction cache
//     sees the whole kernel (DESIGN.md 4.1).
// Output: the root partial sums x of the selected path are turned back into u = x F^{(x)n} and gathered.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <type_traits>
#include <vector>

#include "pb_generic.cuh"
#include "pb_internal.h"

namespace pb {

constexpr int kMaxWarps = 4;                         // decoding warps per CTA
constexpr unsigned kFull = 0xffffffffu;
constexpr int kWsHeadWords = 64;                     // launch state at the head of the workspace (256 bytes)

enum FastOp : uint32_t {
    FOP_UF = 0, FOP_UG, FOP_UC,          // f / g / combine at depth <= top-1 (levels in memory; plain walks: depth <= top-2)
    FOP_SUB8,                            // a plain 8-leaf subtree (registers; Fast-SSC walks)
    FOP_SBEGIN, FOP_SF3, FOP_SG3, FOP_SF2, FOP_SG2, FOP_SPAIR, FOP_SC2, FOP_SC3, FOP_SEND,   // a subtree with special nodes inside
    FOP_SP,                              // Fast-SSC special node: arg = 0 R0, 1 R1, 2 REP, 3 SPC
    FOP_SUB16                            // the depth top-1 node with its two 8-leaf subtrees (registers; plain walks)
};

// Plain walks: the constants of an upper f / g / combine step, packed into its op entry by plan_fast_lut.  Byte 0 of
// x is the type and byte 1 the depth, as in every entry; the rest:
//   UF / UG  x >> 16 = source level's word offset * 32 (kOpOffMask) | kOpInWs if that level is in the workspace
//            y       = destination level's word offset * 32 | kOpInWs | kOpLeftmost (an f step on the leftmost chain)
//                      | first leaf of the node << kOpLeafShift (its partial-sum word * 32 and bit shift)
//   UC       y       = kOpOwnLeft (a left child at depth >= 1: the combine re-points its partial sums) | first leaf << kOpLeafShift
constexpr uint32_t kOpOffMask = 0x7fffu, kOpInWs = 0x8000u, kOpLeftmost = 0x10000u, kOpOwnLeft = 0x10000u;
constexpr int kOpLeafShift = 17;

struct FastParams {
    const uint32_t *stream;        // table stream in consumption order: [chunk][lane][4 lines' word of that lane]
    int n_chunks;
    const uint32_t *frozen_words;  // frozen mask, 32 leaves per word
    int n_ops;                     // compiled tree walk; the ops travel inside the stream (one line per 16 ops):
                                   // x = type | depth<<8 | arg<<16, y = node
    int r1_words;                  // shared-memory words for the R1 scratch (0 when the code has no R1 node)
    const uint32_t *crc_rem;       // [A] CRC remainder of each unit message bit (CA kinds)
    uint32_t crc_checkmask;
    int warps;                     // decoding warps per CTA
    int dbg;                       // POLAR_B200_KDEBUG bits (A/B measurements): 1 = never take the sorted-keeps shortcut
                                   // in fork (and so its identity exit), 2 = never take the identity exit in fork
    int reserved[2];               // unused: keeps the offsets of the fields below, which the kernels' register allocation
                                   // (and so the occupancy and pd_wave_frames) follows -- without it the L=1 kernel of
                                   // SCLUTDecoder drops from 61 to 56 registers and gets a different wave size
    int warp_words;                // shared-memory words of one decoding warp (its V, X, scratch, fork cells)
    int vwords, xwords, scrwords;  // shared-memory words per lane: value levels gl+1..top (top-1: plain walks), X; scratch words per warp
    int scr_off;                   // word offset of the epilogue scratch: its own region, or 0 = on top of the (then dead) value levels
    int gl;                        // value levels 1..gl live in the global (L2-resident) workspace, the rest in shared memory
    int gwords;                    // workspace words per lane
    int voff[kMaxLog + 2];         // word offset of level d inside its home (workspace for d<=gl, shared memory above)
};

struct FastPlan {
    bool ok = false;
    const char *why = "";  // when !ok for a LUT class: which shape rule sent it to the slower kernels
    int logL = 0;
    bool ca = false;
    bool fastk = false;   // the walk contains Fast-SSC special nodes
    FastParams p{};
    size_t smem = 0;
    size_t ws_bytes_per_cta = 0;
    int ctas_per_sm = 0;
    std::vector<void *> allocs;
    std::vector<uint2> ops;   // host copy of the compiled walk (x = type | depth<<8 | arg<<16, y = node), for inspection
};

// shared-memory address of the asynchronous-copy primitives: a 32-bit shared-window address on the device, a plain
// pointer value in the host emulation (tools/emu)
#ifdef PB_HOST_EMU
using smaddr_t = size_t;   // (lds128: with the emulated cp.async below)
#else
using smaddr_t = unsigned;
__device__ __forceinline__ uint4 lds128(smaddr_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];\n" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
#endif

// Table ring: every lane copies ITS 16 bytes of a chunk (512 bytes = 4 table lines, lane-transposed) with cp.async into a
// ring owned by its warp -- no barrier, nothing shared between warps; kRingChunks - 1 chunks in flight per lane.
constexpr int kRingChunks = 4;
#ifdef PB_HOST_EMU
// The emulator copies at once, so by itself it would miss a wait that is too shallow or a refill of a slot whose chunk
// has not been read yet.  This bookkeeping aborts on either: per thread the copies issued and waited for (one commit
// group per copy), per ring address the group that filled it and whether it has been read since.
namespace emu_ring {
struct Slot { unsigned long long grp = 0; bool unread = false; };
inline std::map<size_t, Slot> &slots() { static std::map<size_t, Slot> m; return m; }
inline unsigned long long *counts() { static unsigned long long c[2 * 1024] = {}; return c + 2 * pb_emu::st().cur; }   // issued, waited
inline void forget(smaddr_t lane_slot0) { for (int k = 0; k < kRingChunks; ++k) slots().erase(lane_slot0 + k * 512u); }
}  // namespace emu_ring
// forks seen and identity exits taken (see fork), counted once per warp
namespace emu_fork {
inline unsigned long long &seen() { static unsigned long long n = 0; return n; }
inline unsigned long long &taken() { static unsigned long long n = 0; return n; }
}  // namespace emu_fork
__device__ __forceinline__ void cp_async16(smaddr_t dst, const void *gsrc) {
    emu_ring::Slot &s = emu_ring::slots()[dst];
    if (s.unread) { fprintf(stderr, "scl_lut_warp: ring slot refilled before its chunk was read\n"); abort(); }
    s.grp = ++emu_ring::counts()[0];
    s.unread = true;
    memcpy(reinterpret_cast<void *>(dst), gsrc, 16);
}
template <int NPEND> __device__ __forceinline__ void cp_async_wait() {
    unsigned long long *c = emu_ring::counts();
    if (c[0] >= (unsigned long long)NPEND && c[0] - NPEND > c[1]) c[1] = c[0] - NPEND;
}
__device__ __forceinline__ uint4 lds128(smaddr_t a) {
    auto it = emu_ring::slots().find(a);
    if (it == emu_ring::slots().end() || it->second.grp > emu_ring::counts()[1]) { fprintf(stderr, "scl_lut_warp: ring slot read before its copy was waited for\n"); abort(); }
    it->second.unread = false;
    uint4 v;
    memcpy(&v, reinterpret_cast<const void *>(a), 16);
    return v;
}
#else
__device__ __forceinline__ void cp_async16(smaddr_t dst, const void *gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n cp.async.commit_group;\n" ::"r"(dst), "l"(gsrc) : "memory");
}
template <int NPEND> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(NPEND) : "memory"); }
#endif
// `fetch` = byte offset (inside the lane's column of the stream) of the next chunk to request; wraps at the end of the stream
__device__ __forceinline__ uint4 ring_next_chunk(uint32_t &cc, uint32_t &fetch, smaddr_t ring_lane, const char *stream_lane, uint32_t stream_bytes) {
    const uint32_t slot = cc & (kRingChunks - 1);
    cp_async16(ring_lane + ((slot + kRingChunks - 1) & (kRingChunks - 1)) * 512u, stream_lane + fetch);   // refill the slot consumed before
    fetch += 512u;
    if (fetch == stream_bytes) fetch = 0u;
    cp_async_wait<kRingChunks - 1>();                                                                     // ... and make sure this chunk has landed
    ++cc;
    return lds128(ring_lane + slot * 512u);
}
// out-of-line form for the Fast-SSC kernels (~40 consumption sites); the caller advances cc and fetch
static __device__ __noinline__ uint4 ring_fetch_outlined(uint32_t cc, uint32_t fetch, smaddr_t ring_lane, const char *stream_lane) {
    const uint32_t slot = cc & (kRingChunks - 1);
    cp_async16(ring_lane + ((slot + kRingChunks - 1) & (kRingChunks - 1)) * 512u, stream_lane + fetch);
    cp_async_wait<kRingChunks - 1>();
    return lds128(ring_lane + slot * 512u);
}
// Plain walks: the stream is followed by copies of its first kRingChunks - 1 chunks (plan_fast_lut), so the prefetch
// runs straight through the end of a pass and the kernel sets `fetch` back once per pass: no wrap test per chunk.
__device__ __forceinline__ uint4 ring_next_chunk_lin(uint32_t &cc, uint32_t &fetch, smaddr_t ring_lane, const char *stream_lane) {
    const uint32_t slot = cc & (kRingChunks - 1);
    cp_async16(ring_lane + ((slot + kRingChunks - 1) & (kRingChunks - 1)) * 512u, stream_lane + fetch);
    fetch += 512u;
    cp_async_wait<kRingChunks - 1>();
    ++cc;
    return lds128(ring_lane + slot * 512u);
}
// The two chunks of a SUB8 leaf pair in one go: chunk cc+3 goes into the slot consumed before, one wait covers chunks cc
// and cc+1, and chunk cc+4 goes into the slot of chunk cc once that has been read.  Afterwards kRingChunks - 1 chunks
// are requested ahead again, as after ring_next_chunk_lin, so the two accessors mix freely.
__device__ __forceinline__ void ring_next_pair(uint32_t &cc, uint32_t &fetch, smaddr_t ring_lane, const char *stream_lane,
                                               uint4 &c0, uint4 &c1) {
    constexpr uint32_t kMask = (kRingChunks - 1) * 512u;
    const uint32_t s0 = (cc * 512u) & kMask;
    cp_async16(ring_lane + ((s0 - 512u) & kMask), stream_lane + fetch);
    cp_async_wait<kRingChunks - 2>();
    c0 = lds128(ring_lane + s0);
    c1 = lds128(ring_lane + ((s0 + 512u) & kMask));
    cp_async16(ring_lane + s0, stream_lane + fetch + 512u);
    fetch += 1024u;
    cc += 2u;
}

// R1 nodes of the list Fast decoders: elements packed as rank<<5 | index, one column of a [element][32 lanes] array of
// 16-bit words; std::sort order under "rank < rank" (equal ranks = equal |llr|: libstdc++'s introsort order)
struct R1Acc {
    using V = unsigned short;
    unsigned short *p;   // element i at p[i * 32]
    __device__ __forceinline__ V get(int i) const { return p[i * 32]; }
    __device__ __forceinline__ void set(int i, V v) const { p[i * 32] = v; }
};
struct R1Less {
    __device__ __forceinline__ bool operator()(unsigned short x, unsigned short y) const { return (x >> 5) < (y >> 5); }
};
static __device__ __noinline__ void sort_r1_packed(unsigned short *col, int n) { std_sort_acc<16>(R1Acc{col}, n, R1Less{}); }

struct LineState {
    uint32_t cc;   // chunks consumed so far
    uint32_t fetch;   // stream offset of the next chunk to request
    uint4 cur;     // the chunk lines are currently taken from
    int q;         // next line inside `cur` (4 = exhausted)
};

// 4 symbol bytes -> 4 nibbles (16 bits)
__device__ __forceinline__ uint32_t pack4(uint32_t x) {
    return (x & 0xfu) | ((x >> 4) & 0xf0u) | ((x >> 8) & 0xf00u) | ((x >> 12) & 0xf000u);
}

// One CTA = fp.warps decoding warps, each working on its own frame groups (7 CTAs of 4 warps per SM at N=1024, L=8 =
// 28 decoding warps, 72 registers per thread at most; the Fast variants, which run best with 12 resident warps, may take
// 100).
template <int LOGL, bool CA, bool FAST>
__global__ void __launch_bounds__(kMaxWarps * 32, FAST ? 5 : 7)
scl_lut_warp_kernel(const __grid_constant__ Dev d, const __grid_constant__ FastParams fp, const void *__restrict__ in, int in_dtype,
                    uint8_t *__restrict__ out, long long B, uint32_t *__restrict__ ws, int *err_flag, double *dbg_pm, int *dbg_win) {
    constexpr int L = 1 << LOGL;
    constexpr int FPW = 32 / L;
    PB_DYN_SMEM(uint32_t, sm);
    const int lane = threadIdx.x & 31, W = fp.warps;
    const int wid = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);   // (read through a shuffle: the compiler then treats it as warp-uniform)
    const int grp = lane >> LOGL, me = lane & (L - 1), gbase = lane & ~(L - 1);
    const int N = d.N, n = d.n;
    const int top = n - 3;          // depth of the subtree roots = deepest value level kept in memory (Fast-SSC walks)

    // ---- table stream.  Every f/g table (one 128-byte line = 16x16 nibbles) and every leaf LLR row (16 doubles) is
    //      consumed exactly once per pass, in a fixed order, the same for every warp, and lane l only ever needs word l of
    //      a line.  The host lays the lines out in consumption order, 4 lines per lane-transposed 512-byte chunk; each
    //      warp keeps a private ring of kRingChunks chunks that its lanes fill with cp.async and read with one LDS.128
    //      per chunk (ring_next_chunk). ----
    uint32_t *RINGB = sm + (size_t)W * fp.warp_words + (size_t)wid * (kRingChunks * 128);
    const smaddr_t ring0 = (smaddr_t)__cvta_generic_to_shared(RINGB);
    const long long n_groups = (B + FPW - 1) / FPW;

    uint32_t *V = sm + (size_t)wid * fp.warp_words;    // value levels gl+1..top, [word][lane]
    uint32_t *X = V + fp.vwords * 32;                  // partial sums, in place, [word][lane]
    uint32_t *SCR = V + fp.scr_off;                    // epilogue scratch [word][frame in warp] (L > 1)
    double *KS = reinterpret_cast<double *>(X + fp.xwords * 32 + fp.scrwords);   // key pairs (keep, flip), [path][frame in warp][2]: the FPW groups read adjacent 16-byte cells
    uint32_t *SEL = reinterpret_cast<uint32_t *>(KS + 64);               // [32]
    double *R1S = reinterpret_cast<double *>(SEL + 32);                  // [7][32] smallest |llr| of an R1 node (Fast kinds)
    uint32_t *R1Q = reinterpret_cast<uint32_t *>(R1S + 7 * 32);          // [7][32] their positions
    unsigned short *R1P = reinterpret_cast<unsigned short *>(R1S);       // [32][32] packed sort keys of an R1 node (dead before R1S/R1Q are written)
    // workspace: kWsHeadWords of launch state (word 0 = next frame group), then one region per resident warp
    uint32_t *G = ws + kWsHeadWords + ((size_t)blockIdx.x * W + wid) * fp.gwords * 32;  // value levels 1..gl, [word][lane], L2-resident

    LineState ls;
    ls.cc = 0u; ls.fetch = 0u; ls.cur = make_uint4(0, 0, 0, 0); ls.q = 4;
    const smaddr_t ring_lane = ring0 + (unsigned)lane * 16u;   // this lane's 16 bytes of slot 0
    const char *stream_lane = reinterpret_cast<const char *>(fp.stream) + lane * 16;
    const uint32_t stream_bytes = (uint32_t)fp.n_chunks * 512u;
#ifdef PB_HOST_EMU
    emu_ring::forget(ring_lane);   // (the previous block's last prefetches, never read, went into the same shared memory)
#endif
    for (int i = 0; i < kRingChunks - 1; ++i) { cp_async16(ring_lane + i * 512u, stream_lane + ls.fetch); ls.fetch += 512u; if (FAST && ls.fetch == stream_bytes) ls.fetch = 0u; }
    // the Fast-SSC variant has ~40 consumption sites: there the stream accessors are real (out-of-line) functions so
    // that the hot code stays inside the instruction cache; the plain variant inlines them.  The Fast-SSC variant wraps
    // `fetch` at the end of the stream; the plain one reads on into the copy of the stream's head (ring_next_chunk_lin).
    auto next_chunk = [&]() -> uint4 {
        if (FAST && L > 1) {
            const uint4 v = ring_fetch_outlined(ls.cc, ls.fetch, ring_lane, stream_lane);
            ++ls.cc;
            ls.fetch += 512u;
            if (ls.fetch == stream_bytes) ls.fetch = 0u;
            return v;
        }
        if (!FAST) return ring_next_chunk_lin(ls.cc, ls.fetch, ring_lane, stream_lane);
        return ring_next_chunk(ls.cc, ls.fetch, ring_lane, stream_lane, stream_bytes);
    };
    // upper-level steps and special nodes take their lines one at a time out of the current chunk.  In the Fast-SSC
    // variant `cur` is a queue with the next line in .x (no selects at the many call sites)
    auto next_line = [&]() -> uint32_t {
        if (FAST && L > 1) {
            if (ls.q == 4) { ls.cur = next_chunk(); ls.q = 0; }
            const uint32_t v = ls.cur.x;
            ls.cur.x = ls.cur.y; ls.cur.y = ls.cur.z; ls.cur.z = ls.cur.w;
            ++ls.q;
            return v;
        }
        if (ls.q == 4) { ls.cur = next_chunk(); ls.q = 0; }
        const uint32_t v = ls.q == 0 ? ls.cur.x : ls.q == 1 ? ls.cur.y : ls.q == 2 ? ls.cur.z : ls.cur.w;
        ++ls.q;
        return v;
    };
    // eight f (or g) lookups for one word of symbols: out nibble k = T[u_k][a_k][b_k] with a_k / b_k nibble k of A / Bv.
    // Even and odd nibbles are split into byte lanes so that shuffle sources (a*2 + b>>3) and nibble shifts ((b&7)*4)
    // of four elements come out of a handful of word-wide ops; SHFL only looks at the low 5 bits of its source lane
    // and the funnel shift at the low 5 bits of its amount, so a plain >>8i isolates element i.
    auto lookup8 = [&](uint32_t A, uint32_t Bv, uint32_t ub, uint32_t t0, uint32_t t1, auto isg_c) -> uint32_t {
        constexpr bool ISG = decltype(isg_c)::value;
        const uint32_t m4 = 0x0f0f0f0fu;
        const uint32_t Ae = A & m4, Ao = (A >> 4) & m4, Be = Bv & m4, Bo = (Bv >> 4) & m4;
        const uint32_t Se = (Ae << 1) | ((Be >> 3) & 0x01010101u), So = (Ao << 1) | ((Bo >> 3) & 0x01010101u);
        const uint32_t He = (Be & 0x07070707u) << 2, Ho = (Bo & 0x07070707u) << 2;
        uint32_t accE = 0, accO = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t sel = i == 0 ? 0x3214u : i == 1 ? 0x3240u : i == 2 ? 0x3410u : 0x4210u;
            uint32_t we = __shfl_sync(kFull, t0, (int)(Se >> (8 * i)));
            uint32_t wo = __shfl_sync(kFull, t0, (int)(So >> (8 * i)));
            if (ISG) {
                const uint32_t we1 = __shfl_sync(kFull, t1, (int)(Se >> (8 * i)));
                const uint32_t wo1 = __shfl_sync(kFull, t1, (int)(So >> (8 * i)));
                const uint32_t me_ = (uint32_t)((int)(ub << (31 - 2 * i)) >> 31);
                const uint32_t mo_ = (uint32_t)((int)(ub << (30 - 2 * i)) >> 31);
                we = (we & ~me_) | (we1 & me_);
                wo = (wo & ~mo_) | (wo1 & mo_);
            }
            accE = __byte_perm(accE, __funnelshift_r(we, 0u, He >> (8 * i)), sel);
            accO = __byte_perm(accO, __funnelshift_r(wo, 0u, Ho >> (8 * i)), sel);
        }
        return (accE & m4) | ((accO & m4) << 4);
    };
    auto lut16 = [&](uint32_t treg, uint32_t a, uint32_t b) -> uint32_t {
        const uint32_t w = __shfl_sync(kFull, treg, a * 2 + (b >> 3));
        return (w >> ((b & 7u) * 4)) & 15u;
    };
    auto nib = [](uint32_t w, int k) -> uint32_t { return (w >> (4 * k)) & 15u; };

    for (;;) {
        // the warps take their frame groups from a counter (zeroed by the host before the launch), so a warp that runs
        // ahead -- they do, by a few per cent -- takes more of them and the launch ends without a tail
        unsigned t = 0;
        if (lane == 0) t = atomicAdd(ws, 1u);
        const long long g = (long long)__shfl_sync(kFull, t, 0);
        if (g >= n_groups) break;
        const uint32_t cc_pass = ls.cc;
        long long my_frame = g * FPW + grp;
        if (my_frame >= B) my_frame = B - 1;
        // 8 channel symbols (one output word's worth of the a- or b-half) -> 8 nibbles, with the range check the
        // reference does not have (an out-of-range symbol indexes past the root table there)
        auto in8 = [&](int sym0) -> uint32_t {
            uint32_t x0, x1;
            bool bad = false;
            if (in_dtype == 0) {
                const uint2 v = __ldcs(reinterpret_cast<const uint2 *>(reinterpret_cast<const uint8_t *>(in) + (size_t)my_frame * N + sym0));   // streamed: keep L2 for the workspace
                x0 = v.x; x1 = v.y;
            } else {
                const uint4 *p = reinterpret_cast<const uint4 *>(reinterpret_cast<const int32_t *>(in) + (size_t)my_frame * N + sym0);
                const uint4 v0 = __ldcs(p), v1 = __ldcs(p + 1);
                bad = ((v0.x | v0.y | v0.z | v0.w | v1.x | v1.y | v1.z | v1.w) & 0xffffff00u) != 0;
                x0 = (v0.x & 0xff) | ((v0.y & 0xff) << 8) | ((v0.z & 0xff) << 16) | ((v0.w & 0xff) << 24);
                x1 = (v1.x & 0xff) | ((v1.y & 0xff) << 8) | ((v1.z & 0xff) << 16) | ((v1.w & 0xff) << 24);
            }
            const uint32_t bound = (sym0 < N / 2) ? (uint32_t)d.root_qa : (uint32_t)d.root_qb;
            // every byte < bound  <=>  no byte of (x + (128-bound)) has its top bit set, given x < 128 per byte
            const uint32_t addc = 0x01010101u * (128u - bound);
            bad |= (((x0 | x1) & 0x80808080u) != 0) || ((((x0 & 0x7f7f7f7fu) + addc) | ((x1 & 0x7f7f7f7fu) + addc)) & 0x80808080u) != 0;
            if (bad) { *err_flag = 1; x0 = x1 = 0; }
            return pack4(x0) | (pack4(x1) << 16);
        };

        // level 0: the frame's channel symbols, range-checked and packed 8 per word ONCE, into the group's slot-0 column
        // of the workspace (every path of the frame reads the same words; the root f and g steps then look like any
        // other level).  Lane `me` packs words me, me+L, ...
        {
            uint32_t *g0 = G + grp;                       // level 0 is stored compactly: [word][frame in warp]
            for (int w = me; w < (N >> 3); w += L) g0[w * FPW] = in8(8 * w);
            __syncwarp();
        }

        double PM = (me == 0) ? 0.0 : d.pm_init;
        bool srt = !(fp.dbg & 1) && d.pm_init >= 0.0;   // the path metrics are in non-decreasing slot order (see fork)
        // 3-bit-per-level slot pointers for levels 1..top: values (pv) and left-child partial sums (pu)
        uint32_t pv = 0x09249249u * (uint32_t)me, pu = pv;
        auto getp = [&](uint32_t pw, int lev) -> int { return (int)((pw >> (3 * (lev - 1))) & 7u); };
        auto setown = [&](uint32_t &pw, int lev) { pw = (pw & ~(7u << (3 * (lev - 1)))) | ((uint32_t)me << (3 * (lev - 1))); };
        auto vslot = [&](int lev) -> int { return L == 1 ? lane : (gbase | getp(pv, lev)); };
        auto uslot = [&](int lev) -> int { return L == 1 ? lane : (gbase | getp(pu, lev)); };
        // home of value level `lev` (1..top) for slot lane `sl`: word w is at ptr[w*32]
        auto level_ptr = [&](int lev, int sl) -> uint32_t * {
            return (lev <= fp.gl ? G : V) + fp.voff[lev] * 32 + sl;
        };

        // f / g step at depth dd (<= top-1): level dd -> level dd+1 (>= 8 symbols), written to the lane's own slot.
        // Plain walks take the step's constants from its op entry, where plan_fast_lut packed them (see there):
        // hi = opx >> 16 and node = the entry's second word.  Only the slot lanes are looked up at run time.
        auto fg_step = [&](int dd, uint32_t node, uint32_t hi, bool isg) {
            const int ct = N >> (dd + 1);
            const uint32_t t0 = next_line();
            uint32_t t1 = t0;
            if (isg) t1 = next_line();
            const int sstride = (dd == 0) ? FPW : 32;
            const int nw = ct >> 3;
            int so, dof, xo_, ush;
            bool sg, dg;   // source / destination in the workspace (dd == 0: the packed channel words live there too)
            if (FAST) {
                const uint32_t ub0 = (2u * node) * (uint32_t)ct;
                so = (dd == 0) ? grp : fp.voff[dd] * 32 + vslot(dd);
                dof = fp.voff[dd + 1] * 32 + lane;
                xo_ = (int)(ub0 >> 5) * 32 + uslot(dd + 1);
                ush = (int)(ub0 & 31u);
                sg = dd <= fp.gl;
                dg = dd + 1 <= fp.gl;
            } else {
                so = (int)(hi & kOpOffMask) + ((dd == 0) ? grp : vslot(dd));
                sg = (hi & kOpInWs) != 0u;
                dg = (node & kOpInWs) != 0u;
                const uint32_t ub0 = node >> kOpLeafShift;
                xo_ = (int)(ub0 & ~31u) + uslot(dd + 1);
                ush = (int)(ub0 & 31u);
                if (L > 1 && !isg && (node & kOpLeftmost)) {   // (not in the Fast variant: it is instruction-fetch bound, the extra code costs 10 % there)
                    // leftmost chain of the tree: f outputs of f outputs of the channel symbols depend on no decision, so all
                    // L paths of a frame hold the same words.  Computed once per frame -- the lanes split the words -- into
                    // slot 0 of the group, which every path then points to (the source is shared the same way, by induction).
                    const uint32_t *src = (sg ? G : V) + so;
                    uint32_t *dst0 = (dg ? G : V) + (node & kOpOffMask) + gbase;
                    for (int w0 = 0; w0 < nw; w0 += L) {   // (every lane takes part in the lookup shuffles, also when nw < L)
                        const bool act = w0 + me < nw;
                        const int w = act ? w0 + me : 0;
                        const uint32_t o = lookup8(src[w * sstride], src[(nw + w) * sstride], 0u, t0, t0, std::false_type{});
                        if (act) dst0[w * 32] = o;
                    }
                    pv &= ~(7u << (3 * dd));            // level dd+1 -> slot 0
                    __syncwarp();
                    return;
                }
                dof = (int)(node & kOpOffMask) + lane;
            }
            // ONE word loop per step kind (f / g), source and destination space (workspace or shared memory) chosen at run
            // time through generic pointers.  Round 2 had one instance per (source, destination) space -- plain LDG/LDS with
            // running offsets, 1 % fewer instructions -- but six copies of the hottest loop: the kernel's code grew to 51 KB
            // and, with the warps of an SM spread over the whole walk, instruction fetch became the limit (the same launch
            // was 8 % faster as a sequence of fresh one-wave launches whose warps start in step).  Two copies: 41 KB, and the
            // persistent launch runs 12 % faster (profiles/r2/README.md).  Operands of word w+1 are fetched while word w is
            // looked up; the u bits of a g step come 32 at a time out of the partial-sum column.
            auto body = [&](auto isg_c) {
                constexpr bool ISG = decltype(isg_c)::value;
                const uint32_t *pa = (sg ? G : V) + so;
                uint32_t *pd = (dg ? G : V) + dof;
                const uint32_t *pb = pa + nw * sstride;
                const uint32_t *px = X + xo_;
                uint32_t A = *pa, Bv = *pb, xw = 0;
                if (ISG) xw = *px >> ush;
                for (int w = 0; w < nw; ++w) {
                    uint32_t An = 0, Bn = 0;
                    if (w + 1 < nw) { pa += sstride; pb += sstride; An = *pa; Bn = *pb; }
                    const uint32_t o = lookup8(A, Bv, xw, t0, t1, isg_c);
                    *pd = o;
                    pd += 32;
                    A = An; Bv = Bn;
                    if (ISG) {
                        xw >>= 8;
                        if ((w & 3) == 3 && w + 1 < nw) { px += 32; xw = *px; }
                    }
                }
            };
            if (isg) body(std::true_type{});
            else body(std::false_type{});
            if (L > 1) setown(pv, dd + 1);
            __syncwarp();
        };

        // combine at depth dc (<= top-1): own[left range] = ptr-slot[left range] ^ own[right range]  (u(), utils.cpp:62-67)
        auto combine = [&](int dc, uint32_t node) {
            const int ct = N >> (dc + 1);
            const uint32_t lo = FAST ? node * 2u * (uint32_t)ct : node >> kOpLeafShift;
            const uint32_t *xl = X + uslot(dc + 1);
            uint32_t *xo = X + lane;
            if (ct >= 32) {
                const int nw = ct >> 5, lw = (int)(lo >> 5);
                for (int w = 0; w < nw; ++w) {
                    const uint32_t v = xl[(lw + w) * 32] ^ xo[(lw + nw + w) * 32];
                    __syncwarp();
                    xo[(lw + w) * 32] = v;
                }
            } else {
                const int W = (int)(lo >> 5), sh = (int)(lo & 31u);
                const uint32_t lwv = xl[W * 32];
                uint32_t ow = xo[W * 32];
                const uint32_t mask = ((1u << ct) - 1u) << sh;
                ow = (ow & ~mask) | ((lwv ^ (ow >> ct)) & mask);
                __syncwarp();
                xo[W * 32] = ow;
            }
            if (L > 1 && (FAST ? dc >= 1 && (node & 1u) == 0 : (node & kOpOwnLeft) != 0u)) setown(pu, dc);
            __syncwarp();
        };

        // ---- by-value state of the 8-leaf subtree being decoded (shuffled wholesale on a fork) ----
        uint32_t w3 = 0;     // 8 symbols entering the subtree root (depth top)
        uint32_t w21 = 0;    // [15:0] 4 symbols of the depth top+1 node, [23:16] 2 symbols of the depth top+2 node
        uint32_t xb = 0;     // partial sums of the subtree, in place (bit i = leaf i)

        // mink + list permutation (PD/src/SCLLUTDecoder.cpp:8-22,106-145): every path offers the keys K0 (index
        // me, "keep") and K1 (index L+me, "flip"); the L smallest of the group's 2L keys in std::sort order survive.
        // For 2L <= 16 libstdc++ is an insertion sort, i.e. a stable rank of (key, index).  Returns the lane of the
        // parent path and the flip flag; PM, the pointer words and the subtree registers follow the parent.
        // `keeps_sorted`: the caller offers K0 = PM and no path metric has changed since the previous fork.  A fork leaves
        // the metrics in rank order (slot r = r-th smallest key, equal keys in index order), so (keep_j, j) < (K0, me) is
        // exactly j < me: that part of the rank is `me`, and a third of the compares goes away.  Uniform over the warp
        // (it follows the frozen pattern, not the data).
        // Identity exit: with the keeps sorted, every flip key that is >= the largest keep K0[L-1] ranks after all keeps
        // (on a tie its index L+j is larger), so when that holds on every lane the survivors are the keeps in their slots:
        // p = lane, fl = 0, and PM, the pointer words and the subtree registers stay.  Exact, the same fp64 compares
        // as the rank; most forks of a frame's later leaves take it.
        auto fork = [&](double K0, double K1, int &p, uint32_t &fl, bool keeps_sorted) {
#ifdef PB_HOST_EMU
            if (lane == 0) emu_fork::seen()++;
#endif
            if (!FAST && L > 1 && keeps_sorted && !(fp.dbg & 2)) {
                const double Klast = __shfl_sync(kFull, K0, gbase | (L - 1));
                if (__all_sync(kFull, K1 >= Klast)) {
#ifdef PB_HOST_EMU
                    if (lane == 0) emu_fork::taken()++;
                    if (!(__shfl_sync(kFull, K0, me > 0 ? lane - 1 : lane) <= K0)) { fprintf(stderr, "scl_lut_warp: identity exit on unsorted metrics\n"); abort(); }
#endif
                    p = lane;
                    fl = 0;
                    return;
                }
            }
            __syncwarp();
            *reinterpret_cast<double2 *>(&KS[(me * FPW + grp) * 2]) = make_double2(K0, K1);
            __syncwarp();
            int r0 = 0, r1 = 0;
            if (!FAST && keeps_sorted) {     // (not in the Fast variants: code size, see fg_step)
                r0 = me;
#pragma unroll
                for (int j = 0; j < L; ++j) {
                    const double2 kf = *reinterpret_cast<const double2 *>(&KS[(j * FPW + grp) * 2]);
                    // r0 += flip_j < K0 ;  r1 += keep_j <= K1  +  (flip_j,j) < (K1,me)
#ifdef PB_HOST_EMU
                    if (j < me && !(kf.x <= K0)) { fprintf(stderr, "scl_lut_warp: fork called with keeps_sorted on unsorted metrics\n"); abort(); }
                    r0 += (int)(kf.y < K0);
                    r1 += (int)(kf.x <= K1) + (int)((kf.y < K1) || (kf.y <= K1 && j < me));
#else
                    asm("{\n"
                        " .reg .pred f0, le1, lt1, lf1, jb, t1;\n"
                        " setp.lt.s32 jb, %6, %7;\n"
                        " setp.lt.f64 f0, %3, %4;\n"
                        " setp.le.f64 le1, %2, %5;\n"
                        " setp.lt.f64 lt1, %3, %5;\n"
                        " setp.le.f64 lf1, %3, %5;\n"
                        " and.pred t1, jb, lf1;\n"
                        " or.pred t1, t1, lt1;\n"
                        " @f0 add.s32 %0, %0, 1;\n"
                        " @le1 add.s32 %1, %1, 1;\n"
                        " @t1 add.s32 %1, %1, 1;\n"
                        "}\n"
                        : "+r"(r0), "+r"(r1)
                        : "d"(kf.x), "d"(kf.y), "d"(K0), "d"(K1), "r"(j), "r"(me));
#endif
                }
            } else {
#pragma unroll
            for (int j = 0; j < L; ++j) {
                const double2 kf = *reinterpret_cast<const double2 *>(&KS[(j * FPW + grp) * 2]);
                // r0 += (keep_j,j) < (K0,me)  +  flip_j < K0 ;  r1 += keep_j <= K1  +  (flip_j,j) < (K1,me)
                // (predicated adds: the compiler's bool->int lowering of the same expression costs 40 % more issue slots)
#ifdef PB_HOST_EMU
                r0 += (int)((kf.x < K0) || (kf.x <= K0 && j < me)) + (int)(kf.y < K0);
                r1 += (int)(kf.x <= K1) + (int)((kf.y < K1) || (kf.y <= K1 && j < me));
#else
                asm("{\n"
                    " .reg .pred lt0, le0, f0, le1, lt1, lf1, jb, t0, t1;\n"
                    " setp.lt.s32 jb, %6, %7;\n"
                    " setp.lt.f64 lt0, %2, %4;\n"
                    " setp.le.f64 le0, %2, %4;\n"
                    " setp.lt.f64 f0, %3, %4;\n"
                    " setp.le.f64 le1, %2, %5;\n"
                    " setp.lt.f64 lt1, %3, %5;\n"
                    " setp.le.f64 lf1, %3, %5;\n"
                    " and.pred t0, jb, le0;\n"
                    " or.pred t0, t0, lt0;\n"
                    " and.pred t1, jb, lf1;\n"
                    " or.pred t1, t1, lt1;\n"
                    " @t0 add.s32 %0, %0, 1;\n"
                    " @f0 add.s32 %0, %0, 1;\n"
                    " @le1 add.s32 %1, %1, 1;\n"
                    " @t1 add.s32 %1, %1, 1;\n"
                    "}\n"
                    : "+r"(r0), "+r"(r1)
                    : "d"(kf.x), "d"(kf.y), "d"(K0), "d"(K1), "r"(j), "r"(me));
#endif
            }
            }
            if (r0 < L) SEL[gbase + r0] = (uint32_t)me;
            if (r1 < L) SEL[gbase + r1] = (uint32_t)me | 16u;
            __syncwarp();
            const uint32_t sv = SEL[lane];
            p = gbase | (int)(sv & 15u);
            fl = sv >> 4;
            PM = KS[(((int)(sv & 15u)) * FPW + grp) * 2 + fl];
            w3 = __shfl_sync(kFull, w3, p);
            w21 = __shfl_sync(kFull, w21, p);
            xb = __shfl_sync(kFull, xb, p);
            pv = __shfl_sync(kFull, pv, p);
            pu = __shfl_sync(kFull, pu, p);
            srt = !(fp.dbg & 1);
        };
        // LLR line: lane s holds the low word of entry s, lane 16+s its high word (sym < 16)
        auto llr_of = [&](uint32_t lr, uint32_t sym) -> double {
            const int lo_ = __shfl_sync(kFull, (int)lr, (int)sym), hi_ = __shfl_sync(kFull, (int)lr, (int)(sym + 16u));
            return __hiloint2double(hi_, lo_);
        };
        // result bits of a node at (dd,node) with `temp` <= 32 leaves -> in place (subtree register or own X slot)
        auto put_bits = [&](int dd, uint32_t node, int temp, uint32_t bits) {
            const uint32_t base = node * (uint32_t)temp;
            if (dd > top) {
                const int pos = (int)(base & 7u);
                const uint32_t mask = ((1u << temp) - 1u) << pos;
                xb = (xb & ~mask) | ((bits << pos) & mask);
            } else {
                uint32_t *xo = X + (base >> 5) * 32 + lane;
                if (temp == 32) {
                    *xo = bits;
                } else {
                    const int sh = (int)(base & 31u);
                    const uint32_t mask = ((1u << temp) - 1u) << sh;
                    *xo = (*xo & ~mask) | ((bits << sh) & mask);
                }
                if (L > 1 && (node & 1u) == 0) setown(pu, dd);
                __syncwarp();
            }
        };
        // symbols of the special node at depth dd: word w (8 symbols) of its region
        auto node_word = [&](int dd, int w) -> uint32_t {
            if (dd == top + 2) return w21 >> 16;
            if (dd == top + 1) return w21 & 0xffffu;
            return level_ptr(dd, vslot(dd))[w * 32];
        };

        // Fast-SSC special node (R0 / R1 / REP, plus SPC for the non-list decoder): the LLR of element j is
        // virtual_channel_llrs[dd-1][pos][symbol] (PD/src/FastSCLLUTDecoder.cpp:89,112,179), one stream line per element
        auto special = [&](int spt, int dd, uint32_t node) {
            srt = false;      // special nodes add penalties to the path metrics
            const int temp = N >> dd;
            // the node's LLR lines start on a chunk boundary: four elements per chunk, no per-line bookkeeping
            // (the non-list R0 has no lines; the list R1 takes its rank lines one by one like the upper-level steps)
            if (!(L == 1 && spt == 0) && !(L > 1 && spt == 1)) ls.q = 4;
            uint4 ech = make_uint4(0, 0, 0, 0);
            auto elem_line = [&](int j) -> uint32_t {
                if ((j & 3) == 0) ech = next_chunk();
                return (j & 3) == 0 ? ech.x : (j & 3) == 1 ? ech.y : (j & 3) == 2 ? ech.z : ech.w;
            };
            // a node of 2 elements leaves half a chunk: the following ops' lines continue there
            auto elem_done = [&]() {
                if ((temp & 3) == 0) return;
                ls.q = 2;                                                  // temp == 2
                if (FAST && L > 1) { ls.cur.x = ech.z; ls.cur.y = ech.w; }  // queue form: next line in .x
                else ls.cur = ech;
            };
            const uint32_t full = temp >= 32 ? 0xffffffffu : ((1u << temp) - 1u);
            if (L == 1) {
                // PD/src/FastSCLUT.cpp:43-106
                if (spt == 0) {                                   // R0
                    if (temp <= 32) put_bits(dd, node, temp, 0u);
                    else for (int w = 0; w < (temp >> 5); ++w) X[((node * (uint32_t)temp >> 5) + w) * 32 + lane] = 0u;
                    return;
                }
                double S = 0, best = 0;
                int parity = 0, amin = 0;
                uint32_t bits = 0, sw = 0;
                for (int j = 0; j < temp; ++j) {
                    if ((j & 7) == 0) sw = node_word(dd, j >> 3);
                    const double DM = llr_of(elem_line(j), nib(sw, j & 7));
                    const uint32_t hd = DM <= 0 ? 1u : 0u;
                    S += DM;
                    parity ^= (int)hd;
                    if (j == 0 || fabs(DM) < best) { best = fabs(DM); amin = j; }   // first minimum
                    bits |= hd << (j & 31);
                    if (temp > 32 && (j & 31) == 31) {            // R1 / SPC wider than a word: spill per word
                        X[((node * (uint32_t)temp >> 5) + (j >> 5)) * 32 + lane] = (spt == 2) ? 0u : bits;
                        bits = 0;
                    }
                }
                elem_done();
                if (temp <= 32) {
                    if (spt == 2) bits = (S <= 0) ? full : 0u;   // REP
                    if (spt == 3 && parity) bits ^= 1u << amin;  // SPC: Wagner flip
                    put_bits(dd, node, temp, bits);
                } else {
                    const uint32_t w0 = node * (uint32_t)temp >> 5;
                    if (spt == 2) { const uint32_t v = (S <= 0) ? 0xffffffffu : 0u; for (int w = 0; w < (temp >> 5); ++w) X[(w0 + w) * 32 + lane] = v; }
                    if (spt == 3 && parity) X[(w0 + (amin >> 5)) * 32 + lane] ^= 1u << (amin & 31);
                }
                return;
            }
            int rounds = 1;
            uint32_t dec = 0, rowp = (uint32_t)me;
            double a0 = PM, a1 = PM;
            if (spt != 1) {
                // one pass over the node's elements, in position order (the fp64 sums are serial in the reference):
                //   R0  (PD/src/FastSCLLUTDecoder.cpp:83-93)   PM += (l<0)|l|
                //   REP (:169-184)                             candidates all-0 / all-1: a0 += (l<0)|l|, a1 += (l>=0)|l|
                uint32_t sw = 0;
                for (int j = 0; j < temp; ++j) {
                    if ((j & 7) == 0) sw = node_word(dd, j >> 3);
                    const double l = llr_of(elem_line(j), nib(sw, j & 7));
                    const double al = fabs(l);
                    if (spt == 0) {
                        if (l < 0) PM += al;
                    } else {
                        a0 += (double)(l < 0) * al;
                        a1 += (double)(l >= 0) * al;
                    }
                }
                elem_done();
                if (spt == 0) rounds = 0;
            } else {
                // R1 (:98-121, temp <= 32): hard decisions and argsort(|l|), of which only the first min(L-1,temp)
                // entries are used.  The order of the |l| of a node depends only on how the <= 32*16 table values
                // compare, so the host ships their dense ranks (equal values share a rank) and the sign bits, 16 bits
                // per (element, symbol), four elements per line: the sort runs on small integers in shared memory,
                // [element][lane] (conflict free), packed as rank<<5 | element.
                rounds = (L - 1 < temp) ? L - 1 : temp;
                __syncwarp();
                uint32_t sw = 0, line = 0;
                for (int j = 0; j < temp; ++j) {
                    if ((j & 3) == 0) line = next_line();
                    if ((j & 7) == 0) sw = node_word(dd, j >> 3);
                    const uint32_t sym = nib(sw, j & 7);
                    const uint32_t w = __shfl_sync(kFull, line, (j & 3) * 8 + (int)(sym >> 1));
                    const uint32_t e = (sym & 1u) ? (w >> 16) : (w & 0xffffu);
                    dec |= (e & 1u) << j;
                    R1P[j * 32 + lane] = (unsigned short)(((e >> 1) << 5) | (uint32_t)j);
                }
                unsigned long long qs = 0;   // the `rounds` least reliable positions, 5 bits each
                if (temp <= 16) {
                    // <= 16 elements: std::sort is an insertion sort = stable, i.e. ascending (rank, element) = ascending
                    // packed value: repeated extraction of the next larger one
                    int prev = -1;
                    for (int k = 0; k < rounds; ++k) {
                        int best = 0x7fffffff;
                        for (int j = 0; j < temp; ++j) {
                            const int v = (int)R1P[j * 32 + lane];
                            if (v > prev && v < best) best = v;
                        }
                        prev = best;
                        qs |= (unsigned long long)(best & 31) << (5 * k);
                    }
                } else {
                    sort_r1_packed(R1P + lane, temp);     // libstdc++'s introsort order of equal ranks
                    for (int k = 0; k < rounds; ++k) qs |= (unsigned long long)(R1P[k * 32 + lane] & 31u) << (5 * k);
                }
                __syncwarp();                             // R1P shares its storage with R1S / R1Q
                for (int k = 0; k < rounds; ++k) {
                    const int qk = (int)((qs >> (5 * k)) & 31ull);
                    const uint32_t sym = nib(node_word(dd, qk >> 3), qk & 7);
                    const uint32_t row = __ldg(d.llr_off + (size_t)(dd - 1) * N + node * (uint32_t)temp + qk);
                    R1S[k * 32 + lane] = fabs(__ldg(d.llr + row + sym));
                    R1Q[k * 32 + lane] = (uint32_t)qk;
                }
                __syncwarp();
            }
            for (int layer = 0; layer < rounds; ++layer) {
                uint32_t q = 0;
                if (spt == 1) {
                    const int rl = gbase | (int)rowp;
                    q = R1Q[layer * 32 + rl];
                    a0 = PM;
                    a1 = PM + R1S[layer * 32 + rl];
                }
                int p;
                uint32_t fl;
                fork(a0, a1, p, fl, false);
                if (spt == 1) {      // the flipped position is the slot's OWN pre-permutation ordering (SURVEY App. B4)
                    dec = __shfl_sync(kFull, dec, p);
                    if (fl) dec ^= 1u << q;
                    rowp = __shfl_sync(kFull, rowp, p);
                } else {
                    dec = fl ? full : 0u;
                }
            }
            if (temp <= 32) put_bits(dd, node, temp, dec);
            else {                   // REP wider than a word
                for (int w = 0; w < (temp >> 5); ++w) X[((node * (uint32_t)temp >> 5) + w) * 32 + lane] = dec;
                if ((node & 1u) == 0) setown(pu, dd);
                __syncwarp();
            }
        };

        // ---- the compiled tree walk ----
        ls.q = 4;           // every pass starts on a fresh chunk (the stream is padded to a chunk boundary at its end)
        uint32_t opl = 0;   // this lane's word of the current op line (16 ops)
        for (int oi = 0; oi < fp.n_ops; ++oi) {
            if ((oi & 15) == 0) opl = next_line();
            const uint32_t opx = __shfl_sync(kFull, opl, 2 * (oi & 15)), onode = __shfl_sync(kFull, opl, 2 * (oi & 15) + 1);
            const int ot = (int)(opx & 0xffu), od = (int)((opx >> 8) & 0xffu), oa = (int)((opx >> 16) & 0xffu);
            switch (ot) {
            case FOP_UF: fg_step(od, onode, opx >> 16, false); break;
            case FOP_UG: fg_step(od, onode, opx >> 16, true); break;
            case FOP_UC: combine(od, onode); break;
            case FOP_SP: if (FAST) special(oa, od, onode); break;
            case FOP_SBEGIN: if (FAST) { w3 = *level_ptr(top, vslot(top)); xb = 0; w21 = 0; } break;
            case FOP_SF3: if (FAST) {      // A.f : 8 -> 4 symbols
                const uint32_t t = next_line();
                uint32_t w2 = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) w2 |= lut16(t, nib(w3, k), nib(w3, k + 4)) << (4 * k);
                w21 = w2;
                break;
            }
            case FOP_SG3: if (FAST) {      // A.g : u = the 4 partial sums of the left half
                const uint32_t t0 = next_line(), t1 = next_line();
                uint32_t w2 = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint32_t a = nib(w3, k), b = nib(w3, k + 4);
                    const uint32_t s0 = lut16(t0, a, b), s1 = lut16(t1, a, b);
                    w2 |= (((xb >> k) & 1u) ? s1 : s0) << (4 * k);
                }
                w21 = w2;
                break;
            }
            case FOP_SF2: if (FAST) {      // B.f : 4 -> 2 symbols
                const uint32_t t = next_line();
                const uint32_t c2 = w21 & 0xffffu;
                const uint32_t w1 = lut16(t, nib(c2, 0), nib(c2, 2)) | (lut16(t, nib(c2, 1), nib(c2, 3)) << 4);
                w21 = c2 | (w1 << 16);
                break;
            }
            case FOP_SG2: if (FAST) {      // B.g : u = the 2 partial sums of the left pair (oa = which half of the subtree)
                const uint32_t t0 = next_line(), t1 = next_line();
                const uint32_t c2 = w21 & 0xffffu;
                uint32_t w1 = 0;
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const uint32_t a = nib(c2, k), b = nib(c2, k + 2);
                    const uint32_t s0 = lut16(t0, a, b), s1 = lut16(t1, a, b);
                    w1 |= (((xb >> (4 * oa + k)) & 1u) ? s1 : s0) << (4 * k);
                }
                w21 = c2 | (w1 << 16);
                break;
            }
            case FOP_SC2: if (FAST) xb ^= ((xb >> (4 * oa + 2)) & 3u) << (4 * oa); break;
            case FOP_SC3: if (FAST) xb ^= (xb >> 4) & 15u; break;
            case FOP_SEND: if (FAST) {     // publish the subtree's 8 partial sums in the lane's own slot
                uint32_t *xo = X + ((8u * onode) >> 5) * 32 + lane;
                const int sh = (int)((8u * onode) & 31u);
                *xo = (*xo & ~(0xffu << sh)) | ((xb & 0xffu) << sh);
                if (L > 1 && (onode & 1u) == 0) setown(pu, top);
                __syncwarp();
                break;
            }
            case FAST ? FOP_SUB8 : FOP_SUB16: {   // (Fast-SSC walks have SUB8 ops only, plain walks SUB16 ops only)
                // SUB8: a whole plain 8-leaf subtree, 8 chunk-aligned chunks (see plan_fast_lut), entered through level top
                // in memory.  SUB16: the depth top-1 node and its two 8-leaf subtrees, one SUB8 body per half: the node's f
                // (left) or g (right, u = the left subtree's partial sums) lookup goes straight into w3, so level top never
                // reaches memory, and the left subtree's partial sums wait in xb[15:8] while the right one is decoded.
                // Symbols travel as PAIR BYTES p = a | b << 4 (the two operands of one lookup): the table word is lane
                // a*2 + (b>>3) = ((p&15)<<1) | (p>>7), the nibble shift (b&7)*4 = (p>>2) & 0x1c -- for four pairs at once with
                // byte-lane arithmetic.  w3 = 4 pair bytes of the subtree root, w21 = [15:0] 2 pair bytes of the depth
                // top+1 node, [23:16] the pair byte of the depth top+2 node, xb = partial sums in place.
                // SUB16 arg bit h: the half's 8 leaves are all frozen (plan_fast_lut).  Every decision and so every u of
                // such a half is 0: at L = 1 nothing of it is read (no lines in the stream), at L > 1 it is a
                // feed-forward map from w3 to 8 leaf LLRs and only the path-metric updates stay serial.
                xb = 0;
#pragma unroll 1
                for (int h = 0; h < (FAST ? 1 : 2); ++h) {
                    const bool rate0 = !FAST && ((oa >> h) & 1);
                    if (L == 1 && rate0) { xb <<= 8; continue; }
                    const int s = FAST ? (int)onode : 2 * (int)onode + h;
                    const uint32_t fz = (__ldg(fp.frozen_words + (s >> 2)) >> ((s & 3) * 8)) & 0xffu;
                    {
                        uint32_t w;   // nibbles a0..a3 b0..b3
                        if (FAST) {
                            w = *level_ptr(top, vslot(top));
                        } else {
                            // the node's lines end the chunk before each SUB8 part: [.. f] (left half; the chunk may be
                            // the current one) and [- - g0 g1] (right half; it is the current chunk when the left half
                            // left lines in it).  f is g with t1 = t0 and u = 0.
                            if (ls.q > 3 - h) ls.cur = next_chunk();
                            const uint32_t t1 = ls.cur.w, t0 = h ? ls.cur.z : t1;
                            const uint32_t *src = level_ptr(top - 1, vslot(top - 1));
                            w = lookup8(src[0], src[32], xb, t0, t1, std::true_type{});
                            xb <<= 8;
                        }
                        uint32_t lo = w & 0xffffu, hi = w >> 16;
                        lo = (lo | (lo << 8)) & 0x00ff00ffu; lo = (lo | (lo << 4)) & 0x0f0f0f0fu;
                        hi = (hi | (hi << 8)) & 0x00ff00ffu; hi = (hi | (hi << 4)) & 0x0f0f0f0fu;
                        w3 = lo | (hi << 4);
                    }
                    auto pb_lane = [](uint32_t P) -> uint32_t { return ((P & 0x0f0f0f0fu) << 1) | ((P >> 7) & 0x01010101u); };
                    auto pb_amt = [](uint32_t P) -> uint32_t { return (P >> 2) & 0x1c1c1c1cu; };
                    if (!FAST && L > 1 && rate0) {
                        // all-frozen half: node A (depth top), B0 B1, C0..C3 (depth top+2), each through its f and g0
                        // tables; pair byte k of P goes through table t_k.  Six chunks [A.f A.g0 B0.f B0.g0]
                        // [B1.f B1.g0 C0.f C0.g0] [C1.f C1.g0 C2.f C2.g0] [C3.f C3.g0 llr0 llr1] [llr2 .. llr5]
                        // [llr6 llr7 . .]: the last one stays `cur`, its .z .w are the next lines of the stream.
                        auto look4 = [&](uint32_t P, uint32_t t0, uint32_t t1, uint32_t t2, uint32_t t3) -> uint32_t {
                            const uint32_t S = pb_lane(P), H = pb_amt(P);
                            uint32_t R = 0;
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const uint32_t sel = k == 0 ? 0x3214u : k == 1 ? 0x3240u : k == 2 ? 0x3410u : 0x4210u;
                                const uint32_t wv = __shfl_sync(kFull, k == 0 ? t0 : k == 1 ? t1 : k == 2 ? t2 : t3, (int)(S >> (8 * k)));
                                R = __byte_perm(R, __funnelshift_r(wv, 0u, H >> (8 * k)), sel);
                            }
                            return R & 0x0f0f0f0fu;    // output k in byte k
                        };
                        auto leaf = [&](uint32_t lr, uint32_t sym) {   // (PD/src/SCLLUTDecoder.cpp:92-145, frozen leaf)
                            const double DM = llr_of(lr, sym & 15u);
                            if (DM < 0) PM += fabs(DM);
                        };
                        uint4 c0, c1;
                        ring_next_pair(ls.cc, ls.fetch, ring_lane, stream_lane, c0, c1);
                        const uint32_t fa = look4(w3, c0.x, c0.x, c0.x, c0.x), ga = look4(w3, c0.y, c0.y, c0.y, c0.y);
                        const uint32_t pb = ((fa | (fa >> 12)) & 0xffffu) | (((ga | (ga >> 12)) & 0xffffu) << 16);   // B0 B0 B1 B1
                        const uint32_t fb = look4(pb, c0.z, c0.z, c1.x, c1.x), gb = look4(pb, c0.w, c0.w, c1.y, c1.y);
                        const uint32_t pc = ((fb | (fb >> 4)) & 0x00ff00ffu) | (((gb | (gb >> 4)) & 0x00ff00ffu) << 8);   // C0 C1 C2 C3
                        const uint32_t c0f = c1.z, c0g = c1.w;
                        ring_next_pair(ls.cc, ls.fetch, ring_lane, stream_lane, c0, c1);
                        const uint32_t fc = look4(pc, c0f, c0.x, c0.z, c1.x), gc = look4(pc, c0g, c0.y, c0.w, c1.y);   // leaves 2k, 2k+1
                        leaf(c1.z, fc);
                        leaf(c1.w, gc);
                        ring_next_pair(ls.cc, ls.fetch, ring_lane, stream_lane, c0, c1);
                        leaf(c0.x, fc >> 8);
                        leaf(c0.y, gc >> 8);
                        leaf(c0.z, fc >> 16);
                        leaf(c0.w, gc >> 16);
                        leaf(c1.x, fc >> 24);
                        leaf(c1.y, gc >> 24);
                        ls.cur = c1;
                        ls.q = 2;
                        srt = false;
                        continue;
                    }
                    ls.q = 4;
#pragma unroll 1
                    for (int c4 = 0; c4 < 4; ++c4) {
                        const int pos = 2 * c4;
                        uint4 c0, c1;
                        if (FAST) { c0 = next_chunk(); c1 = next_chunk(); }
                        else ring_next_pair(ls.cc, ls.fetch, ring_lane, stream_lane, c0, c1);
                        if ((c4 & 1) == 0) {
                            // depth top node: four lookups, f (c4 == 0) or g with u = partial sums 0..3 of the left half
                            const uint32_t S = pb_lane(w3), H = pb_amt(w3);
                            uint32_t R = 0;
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const uint32_t sel = k == 0 ? 0x3214u : k == 1 ? 0x3240u : k == 2 ? 0x3410u : 0x4210u;
                                uint32_t wv = __shfl_sync(kFull, c0.x, (int)(S >> (8 * k)));
                                if (c4 != 0) {
                                    const uint32_t w1v = __shfl_sync(kFull, c0.y, (int)(S >> (8 * k)));
                                    wv = ((xb >> k) & 1u) ? w1v : wv;
                                }
                                R = __byte_perm(R, __funnelshift_r(wv, 0u, H >> (8 * k)), sel);
                            }
                            R &= 0x0f0f0f0fu;                                   // o0 o1 o2 o3, one per byte
                            const uint32_t w2p = (R | (R >> 12)) & 0xffffu;     // pair bytes (o0,o2) (o1,o3) of the left / right child
                            // depth top+1 node, f
                            const uint32_t S2 = pb_lane(w2p), H2 = pb_amt(w2p);
                            const uint32_t r0 = __funnelshift_r(__shfl_sync(kFull, c0.z, (int)S2), 0u, H2);
                            const uint32_t r1 = __funnelshift_r(__shfl_sync(kFull, c0.z, (int)(S2 >> 8)), 0u, H2 >> 8);
                            w21 = w2p | ((r0 & 15u) << 16) | ((r1 & 15u) << 20);
                        } else {
                            // depth top+1 node, g with u = the two partial sums of its left child
                            const uint32_t w2p = w21 & 0xffffu;
                            const uint32_t S2 = pb_lane(w2p), H2 = pb_amt(w2p);
                            const uint32_t a0 = __shfl_sync(kFull, c0.x, (int)S2), a1 = __shfl_sync(kFull, c0.y, (int)S2);
                            const uint32_t b0 = __shfl_sync(kFull, c0.x, (int)(S2 >> 8)), b1 = __shfl_sync(kFull, c0.y, (int)(S2 >> 8));
                            const uint32_t r0 = __funnelshift_r(((xb >> (pos - 2)) & 1u) ? a1 : a0, 0u, H2);
                            const uint32_t r1 = __funnelshift_r(((xb >> (pos - 1)) & 1u) ? b1 : b0, 0u, H2 >> 8);
                            w21 = w2p | ((r0 & 15u) << 16) | ((r1 & 15u) << 20);
                        }
#pragma unroll(FAST ? 1 : 2)
                        for (int side = 0; side < 2; ++side) {
                            // leaf symbol through the depth n-1 node: f table (left leaf) or g tables with u = left leaf's bit
                            const uint32_t cp = w21 >> 16;
                            const int cl = (int)(((cp & 15u) << 1) | (cp >> 7));
                            const uint32_t ca_ = (cp >> 2) & 0x1cu;
                            uint32_t wv;
                            if (side == 0) {
                                wv = __shfl_sync(kFull, c0.w, cl);
                            } else {
                                const uint32_t s0 = __shfl_sync(kFull, c1.y, cl), s1 = __shfl_sync(kFull, c1.z, cl);
                                wv = ((xb >> pos) & 1u) ? s1 : s0;
                            }
                            const uint32_t sym = (wv >> ca_) & 15u;
                            const int lp = pos + side;
                            const bool frozen = (fz >> lp) & 1u;
                            // leaf decision (PD/src/SCLUTDecoder.cpp:59-67 / SCLLUTDecoder.cpp:92-145)
                            const double DM = llr_of(side == 0 ? c1.x : c1.w, sym);
                            if (L == 1) {
                                if (!frozen && DM <= 0) xb |= 1u << lp;
                            } else if (frozen) {
                                if (DM < 0) PM += fabs(DM);
                                srt = false;
                            } else {
                                const uint32_t dec = (DM < 0) ? 1u : 0u;
                                int p;
                                uint32_t fl;
                                fork(PM, PM + fabs(DM), p, fl, srt);
                                xb |= (__shfl_sync(kFull, dec, p) ^ fl) << lp;
                            }
                        }
                        xb ^= ((xb >> (pos + 1)) & 1u) << pos;                 // combine of the depth n-1 node
                        if (c4 & 1) xb ^= ((xb >> pos) & 3u) << (pos - 2);     // combine of the depth n-2 node
                    }
                    xb ^= (xb >> 4) & 15u;                                     // combine of the subtree root
                }
                // publish the partial sums in the lane's own slot: SUB8 its 8, SUB16 the 16 of the depth top-1 node
                const uint32_t nb = FAST ? 8u : 16u;
                const uint32_t xv = FAST ? (xb & 0xffu) : ((((xb >> 8) ^ xb) & 0xffu) | ((xb & 0xffu) << 8));
                uint32_t *xo = X + ((nb * onode) >> 5) * 32 + lane;
                const int sh = (int)((nb * onode) & 31u);
                *xo = (*xo & ~(((1u << nb) - 1u) << sh)) | (xv << sh);
                if (L > 1 && (onode & 1u) == 0) setown(pu, FAST ? top : top - 1);
                __syncwarp();
                break;
            }
            case FOP_SPAIR: if (FAST) {    // one leaf pair of a subtree that contains special nodes: 5 lines
                const int s = (int)(onode >> 2);
                const uint32_t fz = (__ldg(fp.frozen_words + (s >> 2)) >> ((s & 3) * 8)) & 0xffu;
                const int c4 = (int)(onode & 3u), pos = 2 * c4;
                uint4 c0, c1;
                c0.x = c0.y = c0.z = 0;
                c0.w = next_line();
                c1.x = next_line(); c1.y = next_line(); c1.z = next_line(); c1.w = next_line();
#pragma unroll 1
                for (int side = 0; side < 2; ++side) {
                    const uint32_t w1 = w21 >> 16;
                    const uint32_t a = nib(w1, 0), b = nib(w1, 1);
                    uint32_t sym;
                    if (side == 0) {
                        sym = lut16(c0.w, a, b);
                    } else {
                        const uint32_t s0 = lut16(c1.y, a, b), s1 = lut16(c1.z, a, b);
                        sym = ((xb >> pos) & 1u) ? s1 : s0;
                    }
                    const int lp = pos + side;
                    const bool frozen = (fz >> lp) & 1u;
                    const double DM = llr_of(side == 0 ? c1.x : c1.w, sym);
                    uint32_t bit = 0;
                    if (L == 1) {
                        bit = (!frozen && DM <= 0) ? 1u : 0u;
                    } else if (frozen) {
                        if (DM < 0) PM += fabs(DM);
                        srt = false;
                    } else {
                        const uint32_t dec = (DM < 0) ? 1u : 0u;
                        int p;
                        uint32_t fl;
                        fork(PM, PM + fabs(DM), p, fl, srt);
                        bit = __shfl_sync(kFull, dec, p) ^ fl;
                    }
                    xb = (xb & ~(1u << lp)) | (bit << lp);
                }
                xb ^= ((xb >> (pos + 1)) & 1u) << pos;                          // combine of the depth n-1 node
                break;
            }
            default: break;
            }
        }

        // ---------------- epilogue: choose the path, u = x F^{(x)n}, gather the information bits ----------------
        const int NW = N >> 5;
        // scratch for u: SC[w*FPW + grp]; for L == 1 every lane transforms its own X column in place
        uint32_t *SC = (L == 1) ? X : SCR;
        auto transform_from = [&](int src_lane) {
            __syncwarp();
            for (int w = me; w < NW; w += L) {
                uint32_t x = X[w * 32 + src_lane];
                x ^= (x >> 1) & 0x55555555u;
                x ^= (x >> 2) & 0x33333333u;
                x ^= (x >> 4) & 0x0f0f0f0fu;
                x ^= (x >> 8) & 0x00ff00ffu;
                x ^= (x >> 16) & 0x0000ffffu;
                SC[w * FPW + grp] = x;
            }
            __syncwarp();
            for (int m = 1; m < NW; m <<= 1) {
                for (int t = me; t < NW / 2; t += L) {
                    const int w = ((t & ~(m - 1)) << 1) | (t & (m - 1));
                    SC[w * FPW + grp] ^= SC[(w + m) * FPW + grp];
                }
                __syncwarp();
            }
        };
        auto ubit = [&](int pos) -> uint32_t { return (SC[(pos >> 5) * FPW + grp] >> (pos & 31)) & 1u; };

        int winner = lane;
        if (L > 1) {
            __syncwarp();
            KS[lane] = PM;
            __syncwarp();
            const double mine = KS[lane];
            int rank = 0, best = 0;
            double bk = KS[gbase];
#pragma unroll
            for (int j = 0; j < L; ++j) {
                const double kj = KS[gbase + j];
                rank += (kj < mine) || (kj == mine && j < me);
                if (kj < bk) { bk = kj; best = j; }   // std::min_element: first minimum
            }
            winner = gbase | best;
            if (CA) {   // PD/src/CASCLLUTDecoder.cpp:264-289: candidates in argsort(PML) order, first CRC pass wins
                SEL[gbase + rank] = (uint32_t)me;
                __syncwarp();
                winner = gbase | (int)SEL[gbase];
                bool decided = false;
                for (int t = 0; t < L; ++t) {
                    const int cand = gbase | (int)SEL[gbase + t];
                    transform_from(cand);
                    uint32_t acc = 0;
                    for (int k = me; k < d.A + d.crc_check; k += L) {
                        const uint32_t bitv = ubit(d.info_pos[k]);
                        const uint32_t contrib = (k < d.A) ? __ldg(fp.crc_rem + k) : (1u << (d.crc_n - 1 - (k - d.A)));
                        acc ^= bitv ? contrib : 0u;
                    }
#pragma unroll
                    for (int o = 1; o < L; o <<= 1) acc ^= __shfl_xor_sync(kFull, acc, o);
                    const bool pass = (acc & fp.crc_checkmask) == 0;
                    if (pass && !decided) { winner = cand; decided = true; }
                    if (__all_sync(kFull, decided)) break;
                }
            }
        }
        transform_from(winner);
        {
            long long frame = g * FPW + grp;
            if (frame < B) {
                uint8_t *o = out + (size_t)frame * d.Kout;
                if (!FAST && (d.Kout & 3) == 0 && ((uintptr_t)o & 3) == 0 && ((uintptr_t)d.info_pos & 15) == 0) {
                    // 4 consecutive output bytes per lane and step: one 16-byte load of positions, four independent bit
                    // reads, one 4-byte store (the Fast-SSC kernels keep the byte loop: code size)
#pragma unroll 1
                    for (int k0 = 4 * me; k0 < d.Kout; k0 += 4 * L) {
                        const int4 p = __ldg(reinterpret_cast<const int4 *>(d.info_pos + k0));
                        __stcs(reinterpret_cast<uint32_t *>(o + k0), ubit(p.x) | (ubit(p.y) << 8) | (ubit(p.z) << 16) | (ubit(p.w) << 24));
                    }
                } else {
                    for (int k = me; k < d.Kout; k += L) __stcs(o + k, (uint8_t)ubit(d.info_pos[k]));
                }
                if (dbg_pm && L > 1) dbg_pm[(size_t)frame * L + me] = PM;
                if (dbg_pm && L == 1) dbg_pm[frame] = 0.0;
                if (dbg_win && me == 0) dbg_win[frame] = winner - gbase;
            }
        }
        __syncwarp();
#ifdef PB_HOST_EMU
        if (ls.cc - cc_pass > (uint32_t)fp.n_chunks) { fprintf(stderr, "scl_lut_warp: pass consumed %u chunks, stream has %d\n", ls.cc - cc_pass, fp.n_chunks); abort(); }
#endif
        // consume the rest of the pass's stream (its zero padding at the end), so that the next pass starts with chunk 0
        // (n_chunks is a multiple of kRingChunks; the rounded bound makes 8 instructions less code in the Fast-SSC kernels)
        while (ls.cc - cc_pass != (uint32_t)fp.n_chunks / kRingChunks * kRingChunks) (void)next_chunk();
        if (!FAST) {
#ifdef PB_HOST_EMU
            if (ls.fetch != (uint32_t)(fp.n_chunks + kRingChunks - 1) * 512u) { fprintf(stderr, "scl_lut_warp: prefetch at byte %u after a pass of %d chunks\n", ls.fetch, fp.n_chunks); abort(); }
#endif
            ls.fetch = (kRingChunks - 1) * 512u;   // the ring holds the copies of chunks 0..kRingChunks-2: go on with the original's next one
        }
    }
    cp_async_wait<0>();
}

// ------------------------------------------------------------------------------------------------
// host side
inline void free_fast_plan(FastPlan *p) {
    for (void *q : p->allocs) cudaFree(q);
    p->allocs.clear();
    p->ok = false;
}

// Kernel instantiations live in their own translation units (pb_kernels.cu, compiled in parallel); the host side only
// sees the dispatcher.
const void *fast_kernel_fn(int logL, bool ca, bool fast);
#ifdef PB_TU_SCL
template <int LOGL, bool FAST>
inline const void *fast_kernel_fn_l(bool ca) {
    if (LOGL == 0 || !ca) return PB_KFN(scl_lut_warp_kernel<LOGL, false, FAST>);
    return PB_KFN(scl_lut_warp_kernel<LOGL, (LOGL > 0), FAST>);
}
#endif

// Decide whether the specialised kernel applies; if so compile the reference's tree walk into the op list and
// lay the tables out as one stream in consumption order.
//   node_type / max_special: Fast kinds only (max_special = 2 for the list decoders, 3 for FastSCLUT, -1 otherwise)
inline void plan_fast_lut(const Dev &d, bool eligible_kind, const int32_t *node_type, int max_special,
                          const std::vector<NodeTab> &tabs, const std::vector<uint8_t> &pool,
                          const std::vector<double> &llr, const std::vector<uint32_t> &llr_off,
                          const int64_t *llr_off64, const int32_t *frozen, uint32_t crc_taps, FastPlan *pl) {
    pl->ok = false;
    pl->why = "";
    if (!eligible_kind) return;
    const int N = d.N, n = d.n, L = d.list ? d.L : 1;
    if (N < 32) { pl->why = "N < 32"; return; }
    int logL = 0;
    while ((1 << logL) < L) logL++;
    if ((1 << logL) != L || L > 8) { pl->why = "list size not in {1,2,4,8}"; return; }
    if (d.list && L == 1) { pl->why = "list decoder with L = 1"; return; }   // list rules with a single path (bit = llr<0, ...) differ from SC's: generic kernel
    for (int p = 0; p < N - 1; ++p) {
        const NodeTab &t = tabs[p];
        if (t.f_pstride || t.g_pstride) { pl->why = "per-position tables inside a node"; return; }
        if (t.f_qb > 16 || t.g_qb > 16 || t.f_sz / t.f_qb > 16 || t.g_sz / t.g_qb > 16) { pl->why = "a table wider than 16 x 16"; return; }
    }
    auto is_special = [&](int depth, int node) -> int {   // -1 or the special type
        if (max_special < 0 || depth >= n) return -1;
        int t = node_type[(1 << depth) + node - 1];
        return (t >= 0 && t <= max_special) ? t : -1;
    };
    // ---- the stream, in the exact order scl_lut_warp_kernel consumes it ----
    std::vector<uint32_t> stream;
    auto push_table = [&](uint32_t off, int qa, int qb) {
        uint32_t line[32];
        memset(line, 0, sizeof line);
        for (int a = 0; a < qa; ++a)
            for (int b = 0; b < qb; ++b) {
                uint32_t v = pool[off + a * qb + b];
                line[a * 2 + (b >> 3)] |= (v & 15u) << ((b & 7) * 4);
            }
        stream.insert(stream.end(), line, line + 32);
    };
    auto push_f = [&](int p) { push_table(tabs[p].f_off, tabs[p].f_sz / tabs[p].f_qb, tabs[p].f_qb); };
    auto push_g = [&](int p) {
        push_table(tabs[p].g_off, tabs[p].g_sz / tabs[p].g_qb, tabs[p].g_qb);
        push_table(tabs[p].g_off + tabs[p].g_sz, tabs[p].g_sz / tabs[p].g_qb, tabs[p].g_qb);
    };
    // The walk (same recursion as the reference's state machine, SURVEY App. A.2) emits ops and, in the same
    // order, the lines each op consumes:
    //   UF: f | UG: g0 g1 | SP: one LLR line per element (none for the non-list R0) | SF3/SF2: f | SG3/SG2: g0 g1
    //   SPAIR: C.f llr(left) C.g0 C.g1 llr(right)
    //   SUB8 (chunk aligned): per leaf pair c4 two chunks [P0 P1 P2 C.f] [llr C.g0 C.g1 llr] with
    //        (P0,P1,P2) = (A.f,-,B.f) for c4=0, (A.g0,A.g1,B.f) for c4=2, (B.g0,B.g1,-) for c4 odd
    //   SUB16 (plain walks only): f, the left SUB8's chunks, g0 g1, the right SUB8's chunks; f and g0 g1 end a chunk.
    //        arg bit h = the 8 leaves of half h are all frozen: at L = 1 the half has no lines at all (nor its f or g0 g1),
    //        at L > 1 its chunks carry only the f and g0 tables and the LLR rows (push_sub8_rate0), 22 lines, and the
    //        next op's lines go on in its last chunk
    const int top = n - 3;
    auto heap = [&](int depth, int node) { return (1 << depth) + node - 1; };
    auto push_pad = [&]() { stream.insert(stream.end(), 32, 0u); };
    std::vector<uint2> ops;
    std::vector<std::vector<uint32_t>> op_lines;   // the lines each op consumes, in order
    auto emit = [&](uint32_t type, int depth, int arg, uint32_t node) {
        if (!ops.empty()) op_lines.back().swap(stream);   // `stream` collects the lines of the op being emitted
        stream.clear();
        ops.push_back(make_uint2(type | ((uint32_t)depth << 8) | ((uint32_t)arg << 16), node));
        op_lines.emplace_back();
    };
    bool ok = true, has_r1 = false;
    auto push_llr_row = [&](int level, int pos) {
        int64_t r = (int64_t)level * N + pos;
        int len = (int)(llr_off64[r + 1] - llr_off64[r]);
        if (len > 16) { ok = false; pl->why = "an LLR row longer than 16"; len = 16; }
        uint32_t line[32];
        memset(line, 0, sizeof line);
        for (int e = 0; e < len; ++e) {   // lane e: low word of entry e, lane 16+e: high word (llr_of)
            uint64_t bits;
            memcpy(&bits, &llr[llr_off[r] + e], 8);
            line[e] = (uint32_t)bits;
            line[16 + e] = (uint32_t)(bits >> 32);
        }
        stream.insert(stream.end(), line, line + 32);
    };
    // list R1 node: dense ranks of |llr| over all (element, symbol) of the node + the sign bits, 16 bits per entry
    // ((rank << 1) | (llr < 0)), entry (j, s) in half (s & 1) of word (j & 3) * 8 + (s >> 1) of line j >> 2
    auto push_r1_ranks = [&](int depth, int node) {
        const int temp = N >> depth;
        std::vector<double> vals;
        for (int j = 0; j < temp; ++j) {
            const int64_t r = (int64_t)(depth - 1) * N + node * temp + j;
            const int len = (int)(llr_off64[r + 1] - llr_off64[r]);
            if (len > 16) { ok = false; pl->why = "an LLR row longer than 16"; return; }
            for (int sidx = 0; sidx < len; ++sidx) {
                const double v = llr[llr_off[r] + sidx];
                if (v != v) { ok = false; pl->why = "NaN in an LLR row of an R1 node"; return; }   // NaN has no rank: generic kernel
                vals.push_back(std::fabs(v));
            }
        }
        std::sort(vals.begin(), vals.end());
        vals.erase(std::unique(vals.begin(), vals.end()), vals.end());
        for (int j0 = 0; j0 < temp; j0 += 4) {
            uint32_t line[32];
            memset(line, 0, sizeof line);
            for (int j = j0; j < std::min(temp, j0 + 4); ++j) {
                const int64_t r = (int64_t)(depth - 1) * N + node * temp + j;
                const int len = (int)(llr_off64[r + 1] - llr_off64[r]);
                for (int sidx = 0; sidx < len; ++sidx) {
                    const double v = llr[llr_off[r] + sidx];
                    const uint32_t rank = (uint32_t)(std::lower_bound(vals.begin(), vals.end(), std::fabs(v)) - vals.begin());
                    const uint32_t e = (rank << 1) | (v < 0 ? 1u : 0u);
                    line[(j & 3) * 8 + (sidx >> 1)] |= e << (16 * (sidx & 1));
                }
            }
            stream.insert(stream.end(), line, line + 32);
        }
    };
    std::function<bool(int, int)> plain = [&](int depth, int node) -> bool {   // no special node in this subtree
        if (depth >= n) return true;
        if (is_special(depth, node) >= 0) return false;
        return plain(depth + 1, 2 * node) && plain(depth + 1, 2 * node + 1);
    };
    auto push_sub8 = [&](int node) {   // the lines of the 8-leaf subtree at depth top
        for (int c4 = 0; c4 < 4; ++c4) {
            const int Bn = heap(top + 1, 2 * node + (c4 >> 1));
            if (c4 == 0) { push_f(heap(top, node)); push_pad(); push_f(Bn); }
            else if (c4 == 2) { push_g(heap(top, node)); push_f(Bn); }
            else { push_g(Bn); push_pad(); }
            const int Cn = heap(top + 2, 4 * node + c4), leaf0 = 8 * node + 2 * c4;
            push_f(Cn);
            push_llr_row(n - 1, leaf0);
            push_g(Cn);
            push_llr_row(n - 1, leaf0 + 1);
        }
    };
    auto push_g0 = [&](int p) { push_table(tabs[p].g_off, tabs[p].g_sz / tabs[p].g_qb, tabs[p].g_qb); };
    auto push_sub8_rate0 = [&](int node) {   // the lines of an all-frozen one, in the kernel's feed-forward order
        for (int dd = top; dd <= top + 2; ++dd)
            for (int k = 0; k < 1 << (dd - top); ++k) { push_f(heap(dd, (node << (dd - top)) + k)); push_g0(heap(dd, (node << (dd - top)) + k)); }
        for (int j = 0; j < 8; ++j) push_llr_row(n - 1, 8 * node + j);
    };
    auto rate0_8 = [&](int node) { for (int j = 0; j < 8; ++j) if (frozen[8 * node + j] != 1) return false; return true; };
    std::function<void(int, int)> walk = [&](int depth, int node) {
        const int p = heap(depth, node), temp = N >> depth;
        const int st = is_special(depth, node);
        if (st >= 0) {
            if (L > 1 && st == 1) { has_r1 = true; if (temp > 32) { ok = false; pl->why = "a list R1 node wider than 32 leaves"; } }
            emit(FOP_SP, depth, st, (uint32_t)node);
            if (L > 1 && st == 1) push_r1_ranks(depth, node);
            else if (!(L == 1 && st == 0))
                for (int j = 0; j < temp; ++j) push_llr_row(depth - 1, node * temp + j);
            return;
        }
        if (depth == top - 1 && max_special < 0) {   // plain walk (the plain kernels have no SUB8 case)
            const int m = (int)rate0_8(2 * node) | ((int)rate0_8(2 * node + 1) << 1);
            emit(FOP_SUB16, depth, m, (uint32_t)node);
            for (int h = 0; h < 2; ++h) {
                if (L == 1 && ((m >> h) & 1)) continue;
                if (h == 0) push_f(p);
                else push_g(p);
                if ((m >> h) & 1) push_sub8_rate0(2 * node + h);
                else push_sub8(2 * node + h);
            }
        } else if (depth < top) {
            emit(FOP_UF, depth, 0, (uint32_t)node); push_f(p);
            walk(depth + 1, 2 * node);
            emit(FOP_UG, depth, 0, (uint32_t)node); push_g(p);
            walk(depth + 1, 2 * node + 1);
            emit(FOP_UC, depth, 0, (uint32_t)node);
        } else if (depth == top) {
            if (plain(depth, node)) {
                emit(FOP_SUB8, depth, 0, (uint32_t)node);
                push_sub8(node);
            } else {
                emit(FOP_SBEGIN, depth, 0, (uint32_t)node);
                emit(FOP_SF3, depth, 0, (uint32_t)node); push_f(p);
                walk(depth + 1, 2 * node);
                emit(FOP_SG3, depth, 0, (uint32_t)node); push_g(p);
                walk(depth + 1, 2 * node + 1);
                emit(FOP_SC3, depth, 0, (uint32_t)node);
                emit(FOP_SEND, depth, 0, (uint32_t)node);
            }
        } else if (depth == top + 1) {
            const int m = node & 1;
            emit(FOP_SF2, depth, m, (uint32_t)node); push_f(p);
            walk(depth + 1, 2 * node);
            emit(FOP_SG2, depth, m, (uint32_t)node); push_g(p);
            walk(depth + 1, 2 * node + 1);
            emit(FOP_SC2, depth, m, (uint32_t)node);
        } else {   // depth == top + 2 == n - 1: an ordinary leaf pair; node = 4*s + c4
            emit(FOP_SPAIR, depth, 0, (uint32_t)node);
            push_f(p);
            push_llr_row(n - 1, 2 * node);
            push_g(p);
            push_llr_row(n - 1, 2 * node + 1);
        }
    };
    walk(0, 0);
    if (!ok || ops.empty()) { if (!*pl->why) pl->why = "empty walk"; return; }
    op_lines.back().swap(stream);
    FastParams &P = pl->p;
    P = FastParams{};
    // value levels 1..mem_top (nibble-packed, (N>>lev)/8 words each): the big ones (> 8 words per lane) go to the
    // global workspace -- they are touched only a handful of times per frame and stay L2-resident --, the small,
    // hot ones stay in shared memory.  This is what sets the occupancy (warps per SM).
    const int FPW = 32 / L;
    // the workspace starts with the packed level-0 (channel) words, [word][frame in warp]: N/8 * FPW words
    int gl = 0, goff = std::max(1, (N / 8) * FPW / 32), soff = 0;
    // (the Fast-SSC walk is latency bound and gains 7 % from the extra resident warps of a 4-word cut; the plain walk is
    //  issue bound and indifferent: measured on N=1024, L=8)
    const int smem_level_words = getenv("POLAR_B200_SMEM_LEVEL_WORDS") ? atoi(getenv("POLAR_B200_SMEM_LEVEL_WORDS")) : 4;
    P.voff[0] = 0;
    // (a plain walk keeps level top = n-3 in registers: SUB16)
    const int mem_top = max_special < 0 ? n - 4 : n - 3;
    for (int lev = 1; lev <= mem_top; ++lev) {
        int words = (N >> lev) / 8;
        if (words > smem_level_words) { P.voff[lev] = goff; goff += words; gl = lev; }
        else { P.voff[lev] = soff; soff += words; }
    }
    P.gl = gl;
    P.gwords = std::max(goff, 1);
    P.vwords = std::max(soff, 1);
    // plain walks: the constants of every upper f / g / combine step go into its op entry (kOpOffMask and the others,
    // next to FastParams), so that the kernel does not derive them from the depth and the node on every step
    if (max_special < 0) {
        for (uint2 &o : ops) {
            const uint32_t ty = o.x & 0xffu, dd = (o.x >> 8) & 0xffu, node = o.y;
            if (ty != FOP_UF && ty != FOP_UG && ty != FOP_UC) continue;
            const uint32_t leaf0 = 2u * node * (uint32_t)(N >> (dd + 1));   // first leaf of the node's left child
            if (ty == FOP_UC) {
                o.y = (dd >= 1 && (node & 1u) == 0 ? kOpOwnLeft : 0u) | (leaf0 << kOpLeafShift);
                continue;
            }
            const uint32_t so = (uint32_t)P.voff[dd] * 32u, dof = (uint32_t)P.voff[dd + 1] * 32u;
            if (so > kOpOffMask || dof > kOpOffMask) { pl->why = "a value level offset too large for the op entry"; return; }
            o.x = (o.x & 0xffffu) | ((so | ((int)dd <= gl ? kOpInWs : 0u)) << 16);
            o.y = dof | ((int)dd + 1 <= gl ? kOpInWs : 0u) | (ty == FOP_UF && node == 0 ? kOpLeftmost : 0u) | (leaf0 << kOpLeafShift);
        }
    }
    // assemble: every 16 ops one "op line" (op k of the batch = words 2k, 2k+1), then each op's own lines; a SUB8
    // op, and each SUB8 part of a SUB16 op, starts on a chunk boundary.  The ops thus ride the same prefetched stream as
    // the tables they drive.
    stream.clear();
    for (size_t i = 0; i < ops.size(); ++i) {
        if (i % 16 == 0) {
            uint32_t line[32];
            for (int k = 0; k < 16; ++k) {
                const bool have = i + k < ops.size();
                line[2 * k] = have ? ops[i + k].x : 0xffu;
                line[2 * k + 1] = have ? ops[i + k].y : 0u;
            }
            stream.insert(stream.end(), line, line + 32);
        }
        const uint32_t oty = ops[i].x & 0xffu;
        auto pad_chunk = [&]() { while ((stream.size() / 32) % 4) stream.insert(stream.end(), 32, 0u); };
        if (oty == FOP_SUB16) {   // [.. f] SUB8 [- - g0 g1] SUB8: the node's lines end the chunk before each SUB8 part
            const uint32_t m = (ops[i].x >> 16) & 3u;
            auto it = op_lines[i].begin();
            for (int h = 0; h < 2; ++h) {
                if (L == 1 && ((m >> h) & 1u)) continue;
                const int sub_lines = ((m >> h) & 1u) ? 22 : 32;
                while ((stream.size() / 32) % 4 != 3u - h) stream.insert(stream.end(), 32, 0u);
                stream.insert(stream.end(), it, it + 32 * (1 + h)); it += 32 * (1 + h);
                stream.insert(stream.end(), it, it + 32 * sub_lines); it += 32 * sub_lines;
            }
            continue;
        }
        const bool list_r1 = oty == FOP_SP && L > 1 && ((ops[i].x >> 16) & 0xffu) == 1u;
        if (oty == FOP_SUB8 || (oty == FOP_SP && !op_lines[i].empty() && !list_r1))
            pad_chunk();
        stream.insert(stream.end(), op_lines[i].begin(), op_lines[i].end());
    }
    // pad to a multiple of kRingChunks chunks of 4 lines and transpose each chunk to [lane][4]
    while ((stream.size() / 32) % (4 * kRingChunks)) stream.insert(stream.end(), 32, 0u);
    const int n_lines = (int)(stream.size() / 32);
    {
        std::vector<uint32_t> tr(stream.size());
        for (int c = 0; c < n_lines / 4; ++c)
            for (int l = 0; l < 32; ++l)
                for (int q = 0; q < 4; ++q) tr[((size_t)c * 32 + l) * 4 + q] = stream[((size_t)c * 4 + q) * 32 + l];
        stream.swap(tr);
    }
    // copies of the first kRingChunks - 1 chunks after the end: the plain kernels' prefetch runs on into them at the end
    // of a pass instead of testing for the wrap on every chunk (n_chunks below stays the pass length)
    {
        const std::vector<uint32_t> head(stream.begin(), stream.begin() + (size_t)(kRingChunks - 1) * 128);
        stream.insert(stream.end(), head.begin(), head.end());
    }
    P.n_chunks = n_lines / 4;
    if (P.n_chunks < 1) return;
    std::vector<uint32_t> fw((N + 31) / 32, 0);
    for (int i = 0; i < N; ++i) if (frozen[i] == 1) fw[i >> 5] |= 1u << (i & 31);
    if (upload(pl->allocs, stream.data(), stream.size(), &P.stream) || upload(pl->allocs, fw.data(), fw.size(), &P.frozen_words)) {
        free_fast_plan(pl);
        return;
    }
    if (d.ca) {
        // remainder of the unit message e_k under the reference's long division (utils.cpp:77-93): linear, so the
        // CRC of a word is the XOR of the remainders of its set bits
        std::vector<uint32_t> rem(d.A);
        const uint32_t msb = 1u << (d.crc_n - 1), mask = d.crc_n >= 32 ? 0xffffffffu : ((1u << d.crc_n) - 1u);
        for (int k = 0; k < d.A; ++k) {
            uint32_t reg = 0;
            for (int i = k; i < d.A; ++i) {
                uint32_t top = ((reg & msb) ? 1u : 0u) ^ (i == k ? 1u : 0u);
                reg = (reg << 1) & mask;
                if (top) reg ^= crc_taps;
            }
            rem[k] = reg;
        }
        if (upload(pl->allocs, rem.data(), rem.size(), &P.crc_rem)) { free_fast_plan(pl); return; }
        uint32_t cm = 0;
        for (int k = 0; k < d.crc_check; ++k) cm |= 1u << (d.crc_n - 1 - k);
        P.crc_checkmask = cm;
    }
    P.xwords = N / 32;
    P.scrwords = (L == 1) ? 0 : (((N / 32) * FPW + 3) & ~3);
    // the value levels are dead once the last leaf is decided: the epilogue scratch goes on top of them when it fits
    if (P.scrwords <= P.vwords * 32 && !getenv("POLAR_B200_NO_SCR_ALIAS")) { P.scr_off = 0; P.scrwords = 0; }
    else P.scr_off = (P.vwords + P.xwords) * 32;
    P.n_ops = (int)ops.size();
    pl->ops = ops;
    if (getenv("POLAR_B200_DEBUG")) {
        int hist[16] = {0};   // by op type
        for (auto &o : ops) hist[o.x & 15u]++;
        fprintf(stderr, "[polar_b200] fast plan: L=%d n_ops=%d chunks=%d fastk=%d max_special=%d hist:", L, (int)ops.size(), n_lines / 4, (int)(max_special >= 0), max_special);
        for (int i = 0; i <= FOP_SUB16; ++i) fprintf(stderr, " %d", hist[i]);
        fprintf(stderr, "\n");
    }
    P.r1_words = has_r1 ? 7 * 32 * 3 : 0;
    P.warp_words = (int)(((size_t)P.vwords * 32 + (size_t)P.xwords * 32 + (size_t)P.scrwords + 128 + 32 + P.r1_words + 3) & ~(size_t)3);
    pl->logL = logL;
    pl->ca = d.ca != 0;
    pl->fastk = max_special >= 0;
    const void *fn = fast_kernel_fn(logL, pl->ca, pl->fastk);
    // CTA shape: as many warps per CTA as keep the SM's warp slots full; POLAR_B200_WARPS_PER_CTA overrides (tuning knob)
    auto smem_for = [&](int w) { return (size_t)w * (P.warp_words * 4 + (size_t)kRingChunks * 512); };
    int best_w = 0, best_occ = 0, best_score = 0;
    const int warp_cap = (pl->fastk && L > 1 && !getenv("POLAR_B200_CTAS_PER_SM")) ? 12 : 1 << 20;   // resident warps per SM wanted at most
    const int want_w = getenv("POLAR_B200_WARPS_PER_CTA") ? atoi(getenv("POLAR_B200_WARPS_PER_CTA")) : 0;
    if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess) { cudaGetLastError(); free_fast_plan(pl); return; }
    for (int w = kMaxWarps; w >= 1; --w) {
        if (want_w && w != std::min(want_w, kMaxWarps)) continue;
        const size_t smem = smem_for(w);
        if (smem > 200 * 1024) continue;
        int occ = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, w * 32, smem) != cudaSuccess) { cudaGetLastError(); continue; }
        // The Fast-SSC list variants are bound by instruction fetch (65 KB of code, 39 % of the stall samples "no
        // instruction"): every extra resident warp adds misses.  Measured on N=1024, L=8 (profiles/r2/README.md): 8 warps per
        // SM 9.1e6 frames/s, 12: 8.9e6, 16: 8.6e6, 21 (all that fit): 7.7e6.  They get 12 warps, in CTAs of 4 when those fit.
        const int score = std::min(occ * w, warp_cap);
        if (score > best_score) { best_w = w; best_occ = occ; best_score = score; }
    }
    if (best_w >= 1) best_occ = std::min(best_occ, std::max(1, warp_cap / best_w));
    if (best_w < 1 || best_occ < 1) { free_fast_plan(pl); return; }
    P.warps = best_w;
    P.dbg = getenv("POLAR_B200_KDEBUG") ? atoi(getenv("POLAR_B200_KDEBUG")) : 0;
    if (const char *e = getenv("POLAR_B200_CTAS_PER_SM")) best_occ = std::max(1, std::min(best_occ, atoi(e)));   // tuning / debug knob
    pl->smem = smem_for(best_w);
    pl->ws_bytes_per_cta = (size_t)P.gwords * 32 * 4 * best_w;
    pl->ctas_per_sm = best_occ;
    pl->ok = true;
}

inline int fast_grid(const FastPlan &pl, long long B, int sm_count) {
    const int L = 1 << pl.logL, FPW = 32 / L;
    long long groups = (B + FPW - 1) / FPW;
    long long ctas = (groups + pl.p.warps - 1) / pl.p.warps;
    return (int)std::max<long long>(1, std::min<long long>(ctas, (long long)sm_count * pl.ctas_per_sm));
}

inline int launch_fast_lut(const Dev &d, const FastPlan &pl, const void *d_in, int dtype, long long B, uint8_t *d_out,
                           cudaStream_t s, uint32_t *ws, int *d_err, double *dbg_pm, int *dbg_win, int sm_count) {
    const int grid = fast_grid(pl, B, sm_count);
    void *args[] = {(void *)&d, (void *)&pl.p, (void *)&d_in, (void *)&dtype, (void *)&d_out, (void *)&B, (void *)&ws,
                    (void *)&d_err, (void *)&dbg_pm, (void *)&dbg_win};
    cudaError_t e0 = cudaMemsetAsync(ws, 0, kWsHeadWords * 4, s);   // the group counter of the dynamic schedule
    if (e0 != cudaSuccess) return (int)e0;
    cudaError_t e = cudaLaunchKernel(fast_kernel_fn(pl.logL, pl.ca, pl.fastk), dim3(grid), dim3(pl.p.warps * 32), args, pl.smem, s);
    if (e != cudaSuccess) return (int)e;
    return (int)cudaGetLastError();
}

}  // namespace pb
