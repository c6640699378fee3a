// path_cta: CTA-level, schedule-driven decoder for the list classes with L in {64, 128, 256}.
//
// path_warp's design (one thread per list path, lazy pointer copy, in-place bit partial sums, parallel rank fork with an
// exact fallback) carried from one warp to L/32 warps: ONE CTA DECODES ONE FRAME AT A TIME, thread i is path slot i, and
// the CTA grid-strides over the batch.
//
// Values of level d (1..n) live at  base[(voff[d] + j) * L + slot]  -- slot-interleaved, so a warp access is one coalesced
// row whatever the slot permutation -- in a per-CTA global workspace for the large levels and in shared memory for the
// last three (4+2+1 elements).  Partial sums stay in place, N/32 words per path, in shared memory (128 KB at N=4096,
// L=256).  Two pointer rows per path, one 8-bit slot id per level (n <= 12: 96 bits, two 64-bit words each), say which
// physical slot holds level d of this logical path (pv: values, pu: left-child partial sums).
//
// Nothing here is warp-synchronous across warps: every exchange between paths goes through shared memory between two
// __syncthreads.  A list permutation publishes every path's pointer rows (and one payload word) to shared memory, and
// each path reads its parent's.
//
// Fork (mink, PD/src/SCLLUTDecoder.cpp:8-22): the 2L keys go to shared memory in PM2 order (index i < L the keep key of
// slot i, i >= L the flip key of slot i-L), and each thread ranks its two keys against all of them (a stable rank).
// libstdc++'s std::sort orders EQUAL keys in an algorithm-defined way (SURVEY App. B1), so the rank is used only when no
// two live (< 1e300) keys are equal -- any correct sort then gives the same permutation of the live paths, and the order
// of dead paths is unobservable.  Otherwise, and always for the Fast list kinds (their R1 rule reads the ordering held by
// the destination slot, dead or not), thread 0 runs the exact emulation (pb::std_sort_idx) over the 2L keys.  The choice
// is made once per CTA with __syncthreads_or.
//
// The blind-detection kinds never run here: PD_BD_CASCL keeps L <= 32 and PD_BD_DMETRIC is not a list kind.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>

#include "pb_generic.cuh"
#include "pb_internal.h"

namespace pb {

constexpr size_t kCtaSmemCap = 227 * 1024;            // largest dynamic shared memory of one CTA on sm_100
constexpr size_t kCtaWsBudget = (size_t)1 << 30;      // global workspace of one launch: the grid is capped to stay below

struct CtaParams {
    int gl;            // value levels 1..gl live in the global workspace, gl+1..n in shared memory
    int xwords;        // N/32
    int scrwords;      // epilogue scratch words (N/32, rounded up to an even count)
    int r1_tmax;       // largest R1 node (list Fast kinds), 0 if none
    size_t vbytes;     // shared-memory bytes of the value levels (16-byte multiple)
    size_t r1_off;     // byte offset of the R1 scratch inside the per-CTA workspace
    size_t ws_stride;  // workspace bytes per CTA
    int voff[kMaxLog + 2];
};

struct CtaPlan {
    bool ok = false;
    int logL = 0;
    CtaParams p{};
    size_t smem = 0;
    size_t ws_bytes_per_cta = 0;
    int ctas_per_sm = 0;
    int max_grid = 0;     // CTAs whose workspace fits kCtaWsBudget
};

// 8-bit slot id per level 1..12: levels 1..8 in lo, 9..12 in hi
struct SlotPtr {
    unsigned long long lo, hi;
};
__device__ __forceinline__ int slot_get(const SlotPtr &p, int lev) {
    return lev <= 8 ? (int)((p.lo >> (8 * (lev - 1))) & 255ull) : (int)((p.hi >> (8 * (lev - 9))) & 255ull);
}
__device__ __forceinline__ void slot_own(SlotPtr &p, int lev, int me) {
    if (lev <= 8) p.lo = (p.lo & ~(255ull << (8 * (lev - 1)))) | ((unsigned long long)me << (8 * (lev - 1)));
    else p.hi = (p.hi & ~(255ull << (8 * (lev - 9)))) | ((unsigned long long)me << (8 * (lev - 9)));
}

template <int DOM, int LOGL>
__global__ void __launch_bounds__(1 << LOGL)
path_cta_kernel(const __grid_constant__ Dev d, const __grid_constant__ CtaParams pp, const void *__restrict__ in, int in_dtype,
                uint8_t *__restrict__ out, long long B, char *__restrict__ ws, int *err_flag, double *dbg_pm, int *dbg_win) {
    using T = typename Val<DOM>::T;
    constexpr int L = 1 << LOGL;
    PB_DYN_SMEM(unsigned char, smraw);
    const int me = threadIdx.x;
    const int N = d.N, n = d.n;

    T *V = reinterpret_cast<T *>(smraw);                                        // levels gl+1..n, [elem][slot]
    uint32_t *X = reinterpret_cast<uint32_t *>(smraw + pp.vbytes);              // partial sums, in place, [word][slot]
    uint32_t *SCR = X + (size_t)pp.xwords * L;                                  // epilogue: u of one candidate
    double *KS = reinterpret_cast<double *>(SCR + pp.scrwords);                 // [2L] fork keys in PM2 order
    unsigned long long *PT = reinterpret_cast<unsigned long long *>(KS + 2 * L);   // [4][L] published pointer rows
    int *ORD = reinterpret_cast<int *>(PT + 4 * L);                             // [2L] exact sort order
    uint32_t *SEL = reinterpret_cast<uint32_t *>(ORD + 2 * L);                  // [L] rank -> (flip << 8) | parent
    int *EX = reinterpret_cast<int *>(SEL + L);                                 // [L] payload word of the fork
    int *MISC = EX + L;                                                         // [4] broadcasts of the epilogue
    char *wsc = ws + (size_t)blockIdx.x * pp.ws_stride;
    T *G = reinterpret_cast<T *>(wsc);                                          // levels 1..gl, [elem][slot]
    double *R1K = reinterpret_cast<double *>(wsc + pp.r1_off);                  // [L][r1_tmax] |llr| rows
    int *R1I = reinterpret_cast<int *>(wsc + pp.r1_off + (size_t)L * pp.r1_tmax * 8);   // [L][r1_tmax] argsort rows

    for (long long frame = blockIdx.x; frame < B; frame += gridDim.x) {
        const uint8_t *in8 = reinterpret_cast<const uint8_t *>(in) + (size_t)frame * N;
        const int32_t *in32 = reinterpret_cast<const int32_t *>(in) + (size_t)frame * N;
        const double *in64 = reinterpret_cast<const double *>(in) + (size_t)frame * N;
        auto in0 = [&](int j) -> T {
            if (DOM == DOM_LUT) {
                int s = (in_dtype == 0) ? (int)__ldg(in8 + j) : __ldg(in32 + j);
                const int bound = (j < N / 2) ? d.root_qa : d.root_qb;
                if (s < 0 || s >= bound) { *err_flag = 1; s = 0; }
                return (T)s;
            } else {
                return (T)__ldg(in64 + j);
            }
        };

        double PM = (me == 0) ? 0.0 : d.pm_init;
        const unsigned long long own8 = 0x0101010101010101ull * (unsigned long long)me;   // every 8-bit field = me
        SlotPtr pv{own8, own8}, pu{own8, own8};
        auto level_ptr = [&](int lev, int sl) -> T * { return (lev <= pp.gl ? G : V) + (size_t)pp.voff[lev] * L + sl; };
        auto read_val = [&](int dd, const T *src, int j) -> T { return dd == 0 ? in0(j) : src[(size_t)j * L]; };
        // LLR of element j of the node at (dd >= 1, node): float domains the value itself, LUT the table row of level dd-1
        auto elem_llr = [&](int dd, unsigned node, const T *src, int j) -> double {
            const T v = src[(size_t)j * L];
            if (DOM == DOM_LUT) {
                const int pos = (int)(node << (n - dd)) + j;
                return __ldg(d.llr + __ldg(d.llr_off + (size_t)(dd - 1) * N + pos) + (int)v);
            } else {
                return (double)v;
            }
        };
        auto xbit_range_write = [&](int dd, unsigned node, auto word_of) {
            // word_of(w) -> the 32 result bits of word w of the node's range (or the low bits for a sub-word range)
            const int temp = N >> dd;
            const unsigned base = node * (unsigned)temp;
            uint32_t *xo = X + (size_t)(base >> 5) * L + me;
            if (temp >= 32) {
                for (int w = 0; w < (temp >> 5); ++w) xo[(size_t)w * L] = word_of(w);
            } else {
                const int sh = (int)(base & 31u);
                const uint32_t mask = ((1u << temp) - 1u) << sh;
                *xo = (*xo & ~mask) | ((word_of(0) << sh) & mask);
            }
            if (dd >= 1 && (node & 1u) == 0) slot_own(pu, dd, me);
            __syncthreads();
        };

        // mink + list permutation (see the header comment); returns the parent's payload `ex`
        auto fork = [&](double K0, double K1, int ex, int &p, uint32_t &fl) -> int {
            __syncthreads();   // every reader of the previous fork's shared state is done
            KS[me] = K0;
            KS[L + me] = K1;
            PT[me] = pv.lo; PT[L + me] = pv.hi; PT[2 * L + me] = pu.lo; PT[3 * L + me] = pu.hi;
            EX[me] = ex;
            ORD[me] = me;
            ORD[L + me] = L + me;
            __syncthreads();
            int r0 = 0, r1 = 0;
            bool tie = false;
            if (d.r1_tmax == 0) {   // (the Fast list kinds with R1 nodes always take the exact sort)
#pragma unroll 4
                for (int j = 0; j < L; ++j) {
                    const double kx = KS[j], ky = KS[L + j];
                    const bool jb = j < me;
                    r0 += (jb ? !(K0 < kx) : (kx < K0)) + (ky < K0);
                    r1 += !(K1 < kx) + (jb ? !(K1 < ky) : (ky < K1));
                    tie |= (j != me && kx == K0 && K0 < 1e300) || (ky == K0 && K0 < 1e300);
                    tie |= (j != me && ky == K1 && K1 < 1e300);
                }
            }
            // exact libstdc++ order is needed when two live keys are equal, and always for the Fast list kinds: their R1 rule
            // flips the bit named by the ordering the DESTINATION slot held before the permutation (FastSCLDecoder.cpp:197-233)
            const bool need = __syncthreads_or(d.r1_tmax > 0 || tie) != 0;
            if (need) {
                if (me == 0) std_sort_idx(ORD, 2 * L, KS);
                __syncthreads();
                const int idx = ORD[me];
                p = idx >= L ? idx - L : idx;
                fl = idx >= L ? 1u : 0u;
            } else {
                if (r0 < L) SEL[r0] = (uint32_t)me;
                if (r1 < L) SEL[r1] = (uint32_t)me | 256u;
                __syncthreads();
                const uint32_t sv = SEL[me];
                p = (int)(sv & 255u);
                fl = sv >> 8;
            }
            PM = KS[fl ? L + p : p];
            pv.lo = PT[p]; pv.hi = PT[L + p]; pu.lo = PT[2 * L + p]; pu.hi = PT[3 * L + p];
            return EX[p];
        };

        Step st_next = d.steps[0];
        for (int si = 0; si < d.n_steps; ++si) {
            const Step st = st_next;
            if (si + 1 < d.n_steps) st_next = d.steps[si + 1];
            const int dd = st.depth;
            const unsigned node = st.node;
            const int temp = N >> dd;
            switch (st.op) {
            case OP_F:
            case OP_G: {
                const int ct = temp >> 1;
                const int p = (1 << dd) + (int)node - 1;
                const bool isg = st.op == OP_G;
                NodeTab tb;
                if (DOM == DOM_LUT) tb = d.tabs[p];
                double r = 0, M = 0;
                const double *bnd = nullptr, *rec = nullptr;
                if (DOM == DOM_UNIFORM) { r = isg ? d.r_g[p] : d.r_f[p]; M = (isg ? d.mg_mul : d.mf_mul) * r; }
                if (DOM == DOM_LLOYD) {
                    bnd = (isg ? d.bnd_g : d.bnd_f) + (size_t)p * d.nb;
                    rec = (isg ? d.rec_g : d.rec_f) + (size_t)p * d.nr;
                }
                const T *src = dd == 0 ? nullptr : level_ptr(dd, slot_get(pv, dd));
                T *dst = level_ptr(dd + 1, me);
                const uint32_t *xsrc = X + slot_get(pu, dd + 1);
                const unsigned ub0 = (2u * node) * (unsigned)ct;
                auto one = [&](int j, T a, T b) {
                    int u = 0;
                    if (isg) { const unsigned bit = ub0 + (unsigned)j; u = (int)((xsrc[(size_t)(bit >> 5) * L] >> (bit & 31u)) & 1u); }
                    T o;
                    if (DOM == DOM_LUT) {
                        if (!isg) o = (T)__ldg(d.lut + tb.f_off + (size_t)j * tb.f_pstride + (unsigned)a * tb.f_qb + (unsigned)b);
                        else o = (T)__ldg(d.lut + tb.g_off + (size_t)j * tb.g_pstride + (unsigned)u * tb.g_sz + (unsigned)a * tb.g_qb + (unsigned)b);
                    } else {
                        double x = isg ? dev_g((double)a, (double)b, u) : dev_minsum((double)a, (double)b);
                        if (DOM == DOM_UNIFORM) x = dev_Q(x, r, M);
                        if (DOM == DOM_LLOYD) x = dev_bisect(x, bnd, d.nb, rec);
                        o = (T)x;
                    }
                    dst[(size_t)j * L] = o;
                };
                int j = 0;
                for (; j + 4 <= ct; j += 4) {      // operands first (the big levels come from L2), then the math
                    T a[4], b[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) { a[q] = read_val(dd, src, j + q); b[q] = read_val(dd, src, j + q + ct); }
#pragma unroll
                    for (int q = 0; q < 4; ++q) one(j + q, a[q], b[q]);
                }
                for (; j < ct; ++j) one(j, read_val(dd, src, j), read_val(dd, src, j + ct));
                slot_own(pv, dd + 1, me);
                __syncthreads();
                break;
            }
            case OP_C: {
                const int ct = temp >> 1;
                const unsigned lo = node * 2u * (unsigned)ct;
                const uint32_t *xl = X + slot_get(pu, dd + 1);
                uint32_t *xo = X + me;
                if (ct >= 32) {
                    const int nw = ct >> 5, lw = (int)(lo >> 5);
                    for (int w = 0; w < nw; ++w) {   // (another path may read the word this one overwrites)
                        const uint32_t v = xl[(size_t)(lw + w) * L] ^ xo[(size_t)(lw + nw + w) * L];
                        __syncthreads();
                        xo[(size_t)(lw + w) * L] = v;
                    }
                } else {
                    const int W = (int)(lo >> 5), sh = (int)(lo & 31u);
                    const uint32_t lwv = xl[(size_t)W * L];
                    uint32_t ow = xo[(size_t)W * L];
                    const uint32_t mask = ((1u << ct) - 1u) << sh;
                    ow = (ow & ~mask) | ((lwv ^ (ow >> ct)) & mask);
                    __syncthreads();
                    xo[(size_t)W * L] = ow;
                }
                if (dd >= 1 && (node & 1u) == 0) slot_own(pu, dd, me);
                __syncthreads();
                break;
            }
            case OP_LEAF: {
                uint32_t bit = 0;
                const double DM = elem_llr(n, node, level_ptr(n, slot_get(pv, n)), 0);
                if (st.flag) {
                    PM += fabs(DM) * (double)(DM < 0);                         // PD/src/SCLDecoder.cpp:62-66
                } else {
                    int p;
                    uint32_t fl;
                    bit = (uint32_t)fork(PM, PM + fabs(DM), DM < 0 ? 1 : 0, p, fl) ^ fl;
                }
                uint32_t *xo = X + (size_t)(node >> 5) * L + me;
                *xo = (*xo & ~(1u << (node & 31u))) | (bit << (node & 31u));
                if ((node & 1u) == 0) slot_own(pu, n, me);
                __syncthreads();
                break;
            }
            case OP_R0: {      // PD/src/FastSCLDecoder.cpp:124-136
                const T *src = level_ptr(dd, slot_get(pv, dd));
                for (int j = 0; j < temp; ++j) {
                    const double l = elem_llr(dd, node, src, j);
                    PM += (double)(float)(l < 0) * fabs(l);
                }
                xbit_range_write(dd, node, [&](int) -> uint32_t { return 0u; });
                break;
            }
            case OP_REP: {     // PD/src/FastSCLDecoder.cpp:208-251
                const T *src = level_ptr(dd, slot_get(pv, dd));
                double a0 = PM, a1 = PM;
                for (int j = 0; j < temp; ++j) {
                    const double l = elem_llr(dd, node, src, j);
                    a0 += (double)(l < 0) * fabs(l);
                    a1 += (double)(l >= 0) * fabs(l);
                }
                int p;
                uint32_t fl;
                fork(a0, a1, 0, p, fl);
                const uint32_t fill = fl ? 0xffffffffu : 0u;
                xbit_range_write(dd, node, [&](int) -> uint32_t { return fill; });
                break;
            }
            case OP_R1: {      // PD/src/FastSCLDecoder.cpp:139-205 incl. the flip-index quirk (SURVEY App. B4)
                const T *src = level_ptr(dd, slot_get(pv, dd));
                const unsigned base = node * (unsigned)temp;
                const int w0 = (int)(base >> 5), sh0 = (int)(base & 31u);
                const int nwords = temp >= 32 ? (temp >> 5) : 1;
                double *myk = R1K + (size_t)me * pp.r1_tmax;
                int *myi = R1I + (size_t)me * pp.r1_tmax;
                // hard decisions straight into the own X range; |llr| and the identity permutation into the path's scratch row
                {
                    uint32_t bits = 0;
                    for (int j = 0; j < temp; ++j) {
                        const double l = elem_llr(dd, node, src, j);
                        myk[j] = fabs(l);
                        myi[j] = j;
                        bits |= (l < 0 ? 1u : 0u) << (j & 31);
                        if ((j & 31) == 31 || j == temp - 1) {
                            uint32_t *xo = X + (size_t)(w0 + (j >> 5)) * L + me;
                            if (temp >= 32) *xo = bits;
                            else { const uint32_t mask = ((1u << temp) - 1u) << sh0; *xo = (*xo & ~mask) | ((bits << sh0) & mask); }
                            bits = 0;
                        }
                    }
                }
                std_sort_idx(myi, temp, myk);           // argsort(abs_llr), libstdc++ tie order, one path per thread
                const int rounds = (L - 1 < temp) ? L - 1 : temp;
                int row = me;                            // slot whose scratch rows (abs_llr, sorted idx) this path carries
                for (int layer = 0; layer < rounds; ++layer) {
                    const int q = R1I[(size_t)row * pp.r1_tmax + layer];
                    int p;
                    uint32_t fl;
                    const int prow = fork(PM, PM + R1K[(size_t)row * pp.r1_tmax + q], row, p, fl);
                    // decision rows follow the parent; the flip goes to this slot's OWN pre-permutation position q
                    for (int w = 0; w < nwords; ++w) {
                        uint32_t v = X[(size_t)(w0 + w) * L + p];
                        if (temp < 32) {
                            const uint32_t mask = ((1u << temp) - 1u) << sh0;
                            const uint32_t own = X[(size_t)(w0 + w) * L + me];
                            v = (own & ~mask) | (v & mask);
                        }
                        if (fl && (q >> 5) == w) v ^= 1u << ((q & 31) + (temp < 32 ? sh0 : 0));
                        __syncthreads();
                        X[(size_t)(w0 + w) * L + me] = v;
                        __syncthreads();
                    }
                    row = prow;
                }
                if ((node & 1u) == 0) slot_own(pu, dd, me);
                __syncthreads();
                break;
            }
            default: break;   // (OP_SPC: non-list kinds only)
            }
        }

        // ---------------- epilogue: choose the path, u = x F^{(x)n}, gather ----------------
        const int NW = N >> 5;
        auto transform_from = [&](int src_slot) {
            __syncthreads();
            for (int w = me; w < NW; w += L) {
                uint32_t x = X[(size_t)w * L + src_slot];
                x ^= (x >> 1) & 0x55555555u;
                x ^= (x >> 2) & 0x33333333u;
                x ^= (x >> 4) & 0x0f0f0f0fu;
                x ^= (x >> 8) & 0x00ff00ffu;
                x ^= (x >> 16) & 0x0000ffffu;
                SCR[w] = x;
            }
            __syncthreads();
            for (int m = 1; m < NW; m <<= 1) {
                for (int t = me; t < NW / 2; t += L) {
                    const int w = ((t & ~(m - 1)) << 1) | (t & (m - 1));
                    SCR[w] ^= SCR[w + m];
                }
                __syncthreads();
            }
        };
        auto ubit = [&](int pos) -> uint32_t { return (SCR[pos >> 5] >> (pos & 31)) & 1u; };

        __syncthreads();
        KS[me] = PM;
        ORD[me] = me;
        __syncthreads();
        if (me == 0) {
            int best = 0;
            for (int j = 1; j < L; ++j)
                if (KS[j] < KS[best]) best = j;                  // std::min_element: first minimum
            if (d.ca) std_sort_idx(ORD, L, KS);                  // argsort(PML) (std::sort), PD/src/CASCLDecoder.cpp:203-234
            MISC[0] = d.ca ? ORD[0] : best;
        }
        __syncthreads();
        int winner = MISC[0];
        if (d.ca) {   // candidates in argsort(PML) order, first CRC pass wins; none passes: the first candidate
            for (int t = 0; t < L; ++t) {
                const int cand = ORD[t];
                transform_from(cand);
                if (me == 0) {   // CRC long division of the first A info bits, compare crc_check bits (utils.cpp:77-93)
                    uint32_t reg = 0;
                    const uint32_t msb = 1u << (d.crc_n - 1);
                    const uint32_t mask = (d.crc_n >= 32) ? 0xffffffffu : ((1u << d.crc_n) - 1u);
                    for (int k = 0; k < d.A; ++k) {
                        const uint32_t topb = ((reg & msb) ? 1u : 0u) ^ ubit(d.info_pos[k]);
                        reg = (reg << 1) & mask;
                        if (topb) reg ^= d.crc_taps;
                    }
                    int pass = 1;
                    for (int k = 0; k < d.crc_check; ++k) {
                        const uint32_t bit = (reg >> (d.crc_n - 1 - k)) & 1u;
                        if (bit != ubit(d.info_pos[d.A + k])) { pass = 0; break; }
                    }
                    MISC[1] = pass;
                }
                __syncthreads();
                if (MISC[1]) { winner = cand; break; }   // (uniform: every thread reads the same word)
            }
        }
        transform_from(winner);
        if (out) {
            uint8_t *o = out + (size_t)frame * d.Kout;
            for (int k = me; k < d.Kout; k += L) o[k] = (uint8_t)ubit(d.info_pos[k]);
        }
        if (dbg_pm) dbg_pm[(size_t)frame * L + me] = PM;
        if (dbg_win && me == 0) dbg_win[frame] = winner;
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
const void *path_cta_kernel_fn(int dom, int logL);   // instantiations: pb_kernels.cu (PB_TU 10)
#ifdef PB_TU_PATH_CTA
template <int DOM>
inline const void *path_cta_kernel_fn_d(int logL) {
    switch (logL) {
    case 6: return PB_KFN(path_cta_kernel<DOM, 6>);
    case 7: return PB_KFN(path_cta_kernel<DOM, 7>);
    default: return PB_KFN(path_cta_kernel<DOM, 8>);
    }
}
inline const void *path_cta_kernel_fn_all(int dom, int logL) {
    switch (dom) {
    case DOM_LUT: return path_cta_kernel_fn_d<DOM_LUT>(logL);
    case DOM_FLOAT: return path_cta_kernel_fn_d<DOM_FLOAT>(logL);
    case DOM_UNIFORM: return path_cta_kernel_fn_d<DOM_UNIFORM>(logL);
    default: return path_cta_kernel_fn_d<DOM_LLOYD>(logL);
    }
}
#endif

// Carve and launch geometry.  Returns nullptr on success, else why the shape cannot run.
inline const char *plan_path_cta(const Dev &d, CtaPlan *pl) {
    pl->ok = false;
    const int N = d.N, n = d.n, L = d.L;
    int logL = 0;
    while ((1 << logL) < L) logL++;
    if (!d.list || logL < 6 || logL > 8 || (1 << logL) != L) return "list size not in {64, 128, 256}";
    if (N < 32) return "N < 32 (partial sums are stored as 32-bit words per path)";
    CtaParams &P = pl->p;
    P = CtaParams{};
    const size_t sz = d.domain == DOM_LUT ? 1 : 8;
    int gl = 0, goff = 0, soff = 0;
    for (int lev = 1; lev <= n; ++lev) {   // levels of <= 4 elements (4+2+1) in shared memory, as in path_warp
        const int elems = N >> lev;
        if (elems > 4) { P.voff[lev] = goff; goff += elems; gl = lev; }
        else { P.voff[lev] = soff; soff += elems; }
    }
    P.gl = gl;
    P.xwords = N / 32;
    P.scrwords = (P.xwords + 1) & ~1;      // keeps the fp64 keys behind it 8-byte aligned
    P.r1_tmax = d.r1_tmax;
    P.vbytes = (((size_t)std::max(soff, 1) * L * sz) + 15) & ~(size_t)15;
    P.r1_off = (((size_t)std::max(goff, 1) * L * sz) + 255) & ~(size_t)255;
    P.ws_stride = (P.r1_off + (size_t)L * P.r1_tmax * 12 + 255) & ~(size_t)255;
    // V | X | SCR | KS[2L] | PT[4L] | ORD[2L] | SEL[L] | EX[L] | MISC[4]
    pl->smem = P.vbytes + (size_t)P.xwords * L * 4 + (size_t)P.scrwords * 4 + (size_t)2 * L * 8 + (size_t)4 * L * 8 +
               (size_t)2 * L * 4 + (size_t)L * 4 + (size_t)L * 4 + 16;
    // (N = 4096, L = 256, fp64: 158.5 KB; every accepted shape fits, the partial sums never have to leave shared memory)
    if (pl->smem > kCtaSmemCap) return "shared-memory carve exceeds 227 KB";
    pl->ws_bytes_per_cta = P.ws_stride;
    pl->logL = logL;
    pl->max_grid = (int)std::max<size_t>(1, std::min<size_t>(kCtaWsBudget / P.ws_stride, 1 << 20));
    const void *fn = path_cta_kernel_fn(d.domain, logL);
    // (per-function state shared by every decoder of this domain and list size: always the cap, see plan_generic)
    if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCtaSmemCap) != cudaSuccess) {
        cudaGetLastError();
        return "cudaFuncSetAttribute failed";
    }
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, L, pl->smem) != cudaSuccess || occ < 1) {
        cudaGetLastError();
        return "the kernel does not fit on the device";
    }
    pl->ctas_per_sm = occ;
    pl->ok = true;
    return nullptr;
}

inline int path_cta_grid(const CtaPlan &pl, long long B, int sm_count) {
    const long long g = std::min<long long>((long long)sm_count * pl.ctas_per_sm, pl.max_grid);
    return (int)std::max<long long>(1, std::min<long long>(B, g));
}

inline int launch_path_cta(const Dev &d, const CtaPlan &pl, const void *d_in, int dtype, long long B, uint8_t *d_out,
                           cudaStream_t s, char *ws, int *d_err, double *dbg_pm, int *dbg_win, int sm_count) {
    const int grid = path_cta_grid(pl, B, sm_count);
    void *args[] = {(void *)&d, (void *)&pl.p, (void *)&d_in, (void *)&dtype, (void *)&d_out, (void *)&B, (void *)&ws,
                    (void *)&d_err, (void *)&dbg_pm, (void *)&dbg_win};
    cudaError_t e = cudaLaunchKernel(path_cta_kernel_fn(d.domain, pl.logL), dim3(grid), dim3(1 << pl.logL), args, pl.smem, s);
    if (e != cudaSuccess) return (int)e;
    return (int)cudaGetLastError();
}

}  // namespace pb
