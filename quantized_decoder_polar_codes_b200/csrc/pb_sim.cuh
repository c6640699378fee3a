// On-device frame generator ("next" row f1): message -> [CRC] -> polar encode -> BPSK + AWGN -> LLR -> channel
// quantizer, one warp per frame.  Mirrors the loop body of the reference drivers
// (mainQuantizedDecoder_LLRDomain.py:151-176) and the encoder / CRC conventions of SURVEY.md 8(c):
//   u[non-frozen] = msg || crc(msg),  x = u F^{(x)n} in natural order,  y = 1-2x + sigma*n,  llr = 2y/sigma^2,
// then stores, per SimDev::mode (the PD_SIM_* values of include/polar_b200.h), what the driver in question feeds its decoder:
//   PD_SIM_LLR          llr (fp64)
//   PD_SIM_LLR_QUANT    0 if llr <= edges[0], Qc-1 if llr >= edges[M], else lut[bisect_left(edges[:-1], llr) - 1]  (uint8;
//                       LLR-domain driver, mainQuantizedDecoder_LLRDomain.py:167-176)
//   PD_SIM_Y_QUANT      0 if y <= edges[0], Qc-1 if y >= edges[M], else bisect_left(edges, y) - 1  (uint8; M = Qc;
//                       probability-domain driver, mainQuantizedDecoder_ProbabilityDomain.py:153-177)
//   PD_SIM_LLR_UNIFORM  QUniform: copysign(sat, llr) if |llr| > bound, else (floor(llr/r) + 0.5) r  (fp64;
//                       continuous-domain driver, mainQuantizedDecoder_ContinuousDomain.py:29-32)
// The mode only picks the last step: message, code word and noise are the same in every mode.
// Noise is Philox4x32-10 keyed by (seed, frame, lane): frame i sees the same noise however the run is split.
#pragma once
#include <cuda_runtime.h>
#include <curand_kernel.h>

#include <cstdint>

#include "../../include/polar_b200.h"

namespace pb {

struct SimDev {
    int N, K, A, crc_n;
    const int32_t *info_pos;     // [K]
    const uint32_t *crc_rem;     // [A] remainder of unit message bit k (MSB-first long division), crc_n <= 32
    const double *edges;         // [n_edges] (LLR_QUANT, Y_QUANT) or nullptr
    int n_edges;
    const uint8_t *chan_lut;     // [n_edges-1] (LLR_QUANT)
    int q_channel;
    int mode;                    // PD_SIM_*
    double r, bound, sat;        // LLR_UNIFORM: step, saturation threshold and saturated value (computed on the host)
};

__global__ void __launch_bounds__(128)
sim_generate_kernel(const SimDev s, double sigma, long long B, unsigned long long seed, unsigned long long first_frame,
                    uint8_t *__restrict__ msg_out, void *__restrict__ out) {
    extern __shared__ uint32_t sm_u[];                       // [warps][N/32] code bits
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int N = s.N, NW = N >> 5;
    uint32_t *U = sm_u + wib * NW;
    const double inv = 2.0 / (sigma * sigma);
    for (long long f = (long long)blockIdx.x * wpb + wib; f < B; f += (long long)gridDim.x * wpb) {
        curandStatePhilox4_32_10_t st;
        curand_init(seed, (first_frame + (unsigned long long)f) * 32ull + (unsigned long long)lane, 0ull, &st);
        for (int w = lane; w < NW; w += 32) U[w] = 0;
        __syncwarp();
        // message bits: lane draws 32 bits per call and owns message words lane, lane+32, ...
        uint32_t crc = 0;
        for (int w = lane; w * 32 < s.A; w += 32) {
            uint32_t bits = curand(&st);
            const int cnt = min(32, s.A - w * 32);
            if (cnt < 32) bits &= (1u << cnt) - 1u;
            for (int b = 0; b < cnt; ++b) {
                const int k = w * 32 + b;
                const uint32_t bit = (bits >> b) & 1u;
                msg_out[(size_t)f * s.A + k] = (uint8_t)bit;
                if (bit) {
                    if (s.crc_n > 0) crc ^= s.crc_rem[k];
                    const int pos = s.info_pos[k];
                    atomicOr(&U[pos >> 5], 1u << (pos & 31));
                }
            }
        }
        if (s.crc_n > 0) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) crc ^= __shfl_xor_sync(0xffffffffu, crc, o);
            for (int k = lane; k < s.crc_n; k += 32) {
                if ((crc >> (s.crc_n - 1 - k)) & 1u) {
                    const int pos = s.info_pos[s.A + k];
                    atomicOr(&U[pos >> 5], 1u << (pos & 31));
                }
            }
        }
        __syncwarp();
        // x = u F^{(x)n}: butterfly x[i] ^= x[i+m] for i with bit m clear
        for (int w = lane; w < NW; w += 32) {
            uint32_t x = U[w];
            x ^= (x >> 1) & 0x55555555u;
            x ^= (x >> 2) & 0x33333333u;
            x ^= (x >> 4) & 0x0f0f0f0fu;
            x ^= (x >> 8) & 0x00ff00ffu;
            x ^= (x >> 16) & 0x0000ffffu;
            U[w] = x;
        }
        __syncwarp();
        for (int m = 1; m < NW; m <<= 1) {
            for (int t = lane; t < NW / 2; t += 32) {
                const int w = ((t & ~(m - 1)) << 1) | (t & (m - 1));
                U[w] ^= U[w + m];
            }
            __syncwarp();
        }
        // channel: positions p = lane, lane+32, ... (coalesced stores)
        for (int p0 = 0; p0 < N; p0 += 64) {
            const double2 nz = curand_normal2_double(&st);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int p = p0 + 32 * h + lane;
                if (p >= N) break;
                const uint32_t xb = (U[p >> 5] >> (p & 31)) & 1u;
                const double y = (1.0 - 2.0 * (double)xb) + sigma * (h ? nz.y : nz.x);
                const double llr = y * inv;
                const size_t o = (size_t)f * N + p;
                if (s.mode == PD_SIM_LLR) {
                    reinterpret_cast<double *>(out)[o] = llr;
                } else if (s.mode == PD_SIM_LLR_UNIFORM) {
                    reinterpret_cast<double *>(out)[o] = fabs(llr) > s.bound ? copysign(s.sat, llr) : (floor(llr / s.r) + 0.5) * s.r;
                } else {
                    const double v = s.mode == PD_SIM_Y_QUANT ? y : llr;
                    int sym;
                    const int M = s.n_edges - 1;
                    if (v <= s.edges[0]) sym = 0;
                    else if (v >= s.edges[M]) sym = s.q_channel - 1;
                    else {   // bisect_left(edges[0..M-1], v); v < edges[M], so it is also bisect_left over all M+1 edges
                        int lo = 0, hi = M;
                        while (lo < hi) {
                            const int mid = (lo + hi) >> 1;
                            if (s.edges[mid] < v) lo = mid + 1; else hi = mid;
                        }
                        sym = s.mode == PD_SIM_Y_QUANT ? lo - 1 : s.chan_lut[lo - 1];
                    }
                    reinterpret_cast<uint8_t *>(out)[o] = (uint8_t)sym;
                }
            }
        }
        __syncwarp();
    }
}

}  // namespace pb
