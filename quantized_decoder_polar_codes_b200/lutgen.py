"""LLR-domain lookup-table generation on the GPU (SURVEY.md 8f row f3): what the reference's
GenerateLookUpTable_LLRDomain.py does through QuantizeDensityEvolution/QLLRDensityEvolution_MinDistortion.py
(`LLRQuantizerSC.run`) -- quantized density evolution over the polar tree with a minimum-distortion quantizer after
every f and g step -- with all quantizer problems of a tree level solved in ONE batched launch (pd_optls_quantize,
csrc/pb_lutgen.cuh) instead of one slow dynamic programme per node.

    gen = MinDistortionLUTGenerator(N=1024, v=16)
    llr_density, llr_quanta, lut_f, lut_g = gen.run(channel_density, channel_quanta)
    kwargs = gen.decoder_tables(lut_f, lut_g, llr_quanta)       # LUT_f / LUT_g / virtual_channel_llr for the decoders

Results are bit-identical to the reference generator driven with its own numpy quantizer
(MinDistortionQuantizer.find_OptLS_quantizer) -- tests/test_lutgen.py, golden vectors made by that code.  The cheap glue
(product distributions, merging equal values with numpy's own np.unique / np.sum) stays in numpy on the host; the
quantizer, which is > 99 % of the reference's run time, is the CUDA kernel.  There is no CPU fallback for it."""
import numpy as np

from . import capi


def optls_quantize_batch(densities, quantas, K, device=0):
    """Batched LLRQuantizer.find_OptLS_quantizer.  densities / quantas: lists of 1-D arrays, each sorted by strictly
    ascending quanta (np.unique output) with more than K entries.  -> (density [P,K], quanta [P,K], list of int32 luts)."""
    P = len(densities)
    M = np.array([len(d) for d in densities], np.int32)
    stride = int(M.max())
    D = np.zeros((P, stride))
    Q = np.zeros((P, stride))
    for p in range(P):
        D[p, :M[p]] = densities[p]
        Q[p, :M[p]] = quantas[p]
    od, oq = np.empty((P, K)), np.empty((P, K))
    lut = np.empty((P, stride), np.int32)
    capi.check(capi.lib().pd_optls_quantize(D.ctypes.data, Q.ctypes.data, M.ctypes.data, stride, P, int(K),
                                            od.ctypes.data, oq.ctypes.data, lut.ctypes.data, int(device)))
    return od, oq, [lut[p, :M[p]].copy() for p in range(P)]


def _merge_equal(density, quanta):
    """LLRQuantizerSC.get_unique_quanta (QLLRDensityEvolution_MinDistortion.py:44-51): symbols with the same value are
    merged first; the masses are added with np.sum over the selected entries, like the reference."""
    uq, inverse = np.unique(quanta, return_inverse=True)
    ud = np.array([np.sum(density[quanta == u]) for u in uq])
    return ud, uq, inverse.astype(np.int32)


class MinDistortionLUTGenerator:
    def __init__(self, N, v, device=0):
        self.N, self.v, self.device = int(N), int(v), int(device)
        self.n = int(np.log2(N))
        if 1 << self.n != self.N:
            raise ValueError("N must be a power of two")

    def _quantize_level(self, problems):
        """problems: list of (density, quanta) after merging equal values -> list of (density[v], quanta[v], lut_merge)."""
        v = self.v
        res = [None] * len(problems)
        big = [i for i, (d, q) in enumerate(problems) if len(d) > v]
        if big:
            od, oq, luts = optls_quantize_batch([problems[i][0] for i in big], [problems[i][1] for i in big], v, self.device)
            for k, i in enumerate(big):
                res[i] = (od[k], oq[k], luts[k])
        for i, (d, q) in enumerate(problems):
            if res[i] is None:      # at most v distinct values: nothing to merge (identity on the sorted symbols, zero padded)
                dd, qq = np.zeros(v), np.zeros(v)
                dd[:len(d)], qq[:len(q)] = d, q
                res[i] = (dd, qq, np.arange(len(d), dtype=np.int32))
        return res

    def run(self, channel_llr_density, channel_llr_quanta):
        """-> llr_density [n+1,N,v], llr_quanta [n+1,N,v] (= virtual_channel_llr), lut_f [N-1,v,v], lut_g [N-1,2,v,v]
        (heap order, one table per node: the reference replicates it for every position of the node)."""
        N, n, v = self.N, self.n, self.v
        dens = np.zeros((n + 1, N, v))
        quan = np.zeros((n + 1, N, v))
        dens[0, :, :] = channel_llr_density
        quan[0, :, :] = channel_llr_quanta
        lut_f = np.zeros((N - 1, v, v), np.int32)
        lut_g = np.zeros((N - 1, 2, v, v), np.int32)
        for level in range(n):
            nb = 1 << (n - level)
            half = nb // 2
            nodes = 1 << level
            problems, erasure = [], []
            for node in range(nodes):
                off = node * nb
                d1, d2 = dens[level, off], dens[level, off + half]
                q1, q2 = quan[level, off], quan[level, off + half]
                # f: min-sum of the two symbols, joint probability (QLLRDensityEvolution_MinDistortion.py:15-31)
                a, b = q1[:, None], q2[None, :]
                qf = (np.sign(a) * np.sign(b) * np.minimum(np.abs(a), np.abs(b))).reshape(-1)
                df = (d1[:, None] * d2[None, :]).reshape(-1)
                # g: (1-2u)a + b for u = 0, 1, each with half of the joint probability (:18-42)
                u = np.arange(2)[:, None, None]
                qg = ((1 - 2 * u) * a[None] + b[None]).reshape(-1)
                dg = np.broadcast_to((0.5 * d1[:, None] * d2[None, :])[None], (2, v, v)).reshape(-1)
                for d_, q_ in ((df, qf), (dg, qg)):
                    ud, uq, inv = _merge_equal(d_, q_)
                    problems.append((ud, uq))
                    erasure.append(inv)
            solved = self._quantize_level(problems)
            for node in range(nodes):
                off = node * nb
                p = (1 << level) + node - 1
                (cdf, cqf, mf), (cdg, cqg, mg) = solved[2 * node], solved[2 * node + 1]
                lut_f[p] = mf[erasure[2 * node]].reshape(v, v)
                lut_g[p] = mg[erasure[2 * node + 1]].reshape(2, v, v)
                dens[level + 1, off:off + half] = cdf
                quan[level + 1, off:off + half] = cqf
                dens[level + 1, off + half:off + nb] = cdg
                quan[level + 1, off + half:off + nb] = cqg
        return dens, quan, lut_f, lut_g

    @staticmethod
    def decoder_tables(lut_f, lut_g, llr_quanta):
        """Constructor arguments of the LUT decoders in the compact one-table-per-node form they accept."""
        return dict(LUT_f=[t[None] for t in lut_f], LUT_g=[t[None] for t in lut_g], virtual_channel_llr=llr_quanta)


# ----------------------------------------------------------------------------------------------------------------------
# Probability-domain tables (maximum mutual information): GenerateLookUpTable_ProbabilityDomain.py ->
# QuantizeDensityEvolution/QDensityEvolution_MMI.py (QDensityEvolutionMMI.run) with MMIQuantizer.find_opt_quantizer on the
# f and g output distribution of every node.  The quantizer's cost table and dynamic programme run on the GPU
# (pd_mmi_slice_sums / pd_mmi_design, csrc/pb_lutgen.cuh); the logarithms in between are numpy's, the cheap glue
# (normalisation, Kronecker products, LLRs) is the reference's numpy arithmetic on the host.  Bit-identical to the reference
# generator driven with its numpy quantizer (QuantizeDensityEvolution/MMIQuantizer.py) under the two conventions written
# down in tests/golden/make_mmi_golden.py: equal likelihood ratios keep their index order (stable sort) and the joint
# distribution is float64 (the C++ binding's py::array_t<double>).

def mmi_quantize_batch(joints, K, device=0, px1=0.5, px_minus1=0.5, sort=True):
    """Batched MMIQuantizer.find_opt_quantizer (MMIQuantizer.cpp:73-165 / MMIQuantizer.py:158-225).
    joints: [P, 2, M] float64, K < M.  -> Q [P, K, M] int32 (Q[p,i,j] = 1: input j goes to output i), pzx [P, 2, K] = P(z|x),
    Az [P, K+1] cluster boundaries in sorted order, perm [P, M] the sort.  sort=False is find_opt_quantizer_AWGN (:264-325)."""
    joints = np.ascontiguousarray(joints, dtype=np.float64)
    P, _, M = joints.shape
    K = int(K)
    if sort:
        with np.errstate(divide="ignore", invalid="ignore"):
            llr = np.log2(joints[:, 0] / joints[:, 1])
        perm = np.argsort(llr, axis=1, kind="stable")
    else:
        perm = np.broadcast_to(np.arange(M), (P, M)).copy()
    p1 = np.ascontiguousarray(np.take_along_axis(joints[:, 0], perm, axis=1))
    p2 = np.ascontiguousarray(np.take_along_axis(joints[:, 1], perm, axis=1))
    W = M - K + 1
    lib = capi.lib()
    Az = np.zeros((P, K + 1), np.int32)
    step = max(1, (1 << 24) // (M * W))          # <= 128 MiB per table per call
    for p0 in range(0, P, step):
        sl = slice(p0, min(P, p0 + step))
        n = sl.stop - sl.start
        a1, a2 = np.ascontiguousarray(p1[sl]), np.ascontiguousarray(p2[sl])
        S1, S2 = np.empty((n, M, W)), np.empty((n, M, W))
        capi.check(lib.pd_mmi_slice_sums(a1.ctypes.data, a2.ctypes.data, n, M, K, S1.ctypes.data, S2.ctypes.data, int(device)))
        # compute_partial_entropy (MMIQuantizer.py:46-63): cluster likelihoods and their logarithms, numpy's own
        with np.errstate(divide="ignore", invalid="ignore"):
            pn = px1 * S1 + px_minus1 * S2
            ok = pn != 0
            c1 = np.where(ok, S1 / np.where(ok, pn, 1.0), 0.0)
            c2 = np.where(ok, S2 / np.where(ok, pn, 1.0), 0.0)
            L1 = np.where(c1 == 0, 0.0, np.log2(np.where(c1 == 0, 1.0, c1)))
            L2 = np.where(c2 == 0, 0.0, np.log2(np.where(c2 == 0, 1.0, c2)))
        az = np.zeros((n, K + 1), np.int32)
        capi.check(lib.pd_mmi_design(a1.ctypes.data, a2.ctypes.data, np.ascontiguousarray(L1).ctypes.data,
                                     np.ascontiguousarray(L2).ctypes.data, float(px1), float(px_minus1), n, M, K,
                                     az.ctypes.data, int(device)))
        Az[sl] = az
    Q = np.zeros((P, K, M), np.int32)
    pzx = np.zeros((P, 2, K))
    for p in range(P):
        for i in range(K):
            idx = perm[p, Az[p, i]:Az[p, i + 1]]
            Q[p, i, idx] = 1
            for j in idx:                        # MMIQuantizer.cpp:151-160: accumulated one by one in sorted order
                pzx[p, 0, i] += joints[p, 0, j]
                pzx[p, 1, i] += joints[p, 1, j]
    return Q, pzx, Az, perm


def _log2_stable(value):
    """PyIBQuantizer/inf_theory_tools.py:3-12"""
    if np.any(value <= 0):
        result = np.empty_like(value)
        result[value > 0] = np.log2(value[value > 0])
        result[value <= 0] = -1e6
        return result
    return np.log2(value)


class MMILUTGenerator:
    """QDensityEvolutionMMI(N, quantization_level_decoder).run(channel_symbol_probs) (QDensityEvolution_MMI.py:34-122)."""

    def __init__(self, N, v, device=0):
        self.N, self.v, self.device = int(N), int(v), int(device)
        self.n = int(np.log2(N))
        if 1 << self.n != self.N:
            raise ValueError("N must be a power of two")

    def run(self, channel_symbol_probs):
        """channel_symbol_probs: P(z|x) of the channel quantizer, [2, Qc].  -> lut_f, lut_g (lists over heap ids of
        [Qa,Qb] / [2,Qa,Qb] int32 tables: Qc x Qc at the root, v x v below), virtual_channel_llrs [n, N, v],
        virtual_channel_transition_probs [n, N, 2, v]."""
        N, n, v = self.N, self.n, self.v
        probs_lvl = np.zeros((n, N, 2, v))
        llrs = np.zeros((n, N, v))
        chan = np.expand_dims(np.asarray(channel_symbol_probs, dtype=np.float64), axis=0).repeat(N, axis=0)
        qc = chan.shape[2]
        lut_f, lut_g = [None] * (N - 1), [None] * (N - 1)
        for level in range(n):
            nb = 1 << (n - level)
            half = nb // 2
            nodes = 1 << level
            probs = chan if level == 0 else probs_lvl[level - 1]
            ny = qc if level == 0 else v
            jf, jg = [], []
            for node in range(nodes):
                off = node * nb
                A, Bm = probs[off], probs[off + half]
                # (the reference normalises the rows in place, :70-73)
                A[0] /= np.sum(A[0]); A[1] /= np.sum(A[1]); Bm[0] /= np.sum(Bm[0]); Bm[1] /= np.sum(Bm[1])
                # u0 -> (y0,y1) (:76-79)
                f0 = 0.5 * (np.kron(A[0], Bm[0]) + np.kron(A[1], Bm[1]))
                f1 = 0.5 * (np.kron(A[1], Bm[0]) + np.kron(A[0], Bm[1]))
                jf.append(np.array([[f0], [f1]]).squeeze().astype(np.float32))
                # u1 -> (y0,y1,u0) (:96-105): symbols ordered (y0, y1, u0)
                g00, g10 = 0.5 * np.kron(A[0], Bm[0]), 0.5 * np.kron(A[1], Bm[0])
                t0 = np.dstack((g00, g10)).squeeze()
                g01, g11 = 0.5 * np.kron(A[1], Bm[1]), 0.5 * np.kron(A[0], Bm[1])
                t1 = np.dstack((g01, g11)).squeeze()
                jg.append(np.array([[np.reshape(t0, [2 * t0.shape[0]])], [np.reshape(t1, [2 * t1.shape[0]])]]).squeeze().astype(np.float32))
            Qf, Pf, _, _ = mmi_quantize_batch(np.stack(jf), v, self.device)
            Qg, Pg, _, _ = mmi_quantize_batch(np.stack(jg), v, self.device)
            for node in range(nodes):
                off = node * nb
                p = (1 << level) + node - 1
                probs_lvl[level, off:off + half] = Pf[node]
                llrs[level, off:off + half] = _log2_stable(Pf[node][0] / (Pf[node][1] + 1e-31))
                lut_f[p] = np.argmax(Qf[node], axis=0).astype(np.int32).reshape(ny, ny)          # get_lut_from_Q 'f' (:13-20)
                probs_lvl[level, off + half:off + nb] = Pg[node]
                llrs[level, off + half:off + nb] = _log2_stable(Pg[node][0] / (Pg[node][1] + 1e-31))
                lut_g[p] = np.argmax(Qg[node], axis=0).astype(np.int32).reshape(ny, ny, 2).transpose(2, 0, 1).copy()   # 'g' (:21-29)
        return lut_f, lut_g, llrs, probs_lvl

    @staticmethod
    def decoder_tables(lut_f, lut_g, llrs):
        """Constructor arguments of the LUT decoders (levels = n: row l holds the outputs of level l, which is how the
        decoders index it, PD/src/SCLLUTDecoder.cpp:97)."""
        return dict(LUT_f=[t[None] for t in lut_f], LUT_g=[t[None] for t in lut_g], virtual_channel_llr=llrs)


def channel_transition_probability_table(M, low, high, mu, sigma):
    """utils.py:16-28 of the reference: P(y in cell i | x = mu) for M uniform cells on [low, high], integrated on a 1e-4
    grid (both cell edges inclusive, np.sum of the selected samples) -- kept in this exact form because the table
    generator and the drivers build their channel quantizers from it."""
    delta = 0.0001
    x = np.arange(low, high + delta, delta)
    pdf = 1 / np.sqrt(2 * np.pi * sigma ** 2) * np.exp(-(x - mu) ** 2 / (2 * sigma ** 2))
    edges = np.linspace(low, high, M + 1)
    pyx = np.zeros(M)
    for i in range(M):
        pyx[i] = np.sum(pdf[np.bitwise_and(x >= edges[i], x <= edges[i + 1])]) * delta
    return pyx, edges


def mmi_channel_quantizer(sigma, q_uniform=128, q_channel=16, device=0):
    """The channel quantizer the probability-domain generator and driver build for a noise level
    (GenerateLookUpTable_ProbabilityDomain.py:45-62, mainQuantizedDecoder_ProbabilityDomain.py:137-152):
    uniform cells on [-1-3 sigma, 1+3 sigma] merged to q_channel symbols by MMIQuantizer.find_opt_quantizer_AWGN.
    -> pzx [2, q_channel] = P(z|x=+1), P(z|x=-1); cell edges interval_x [q_uniform+1]; channel_lut [q_channel+1]."""
    hi, lo = 1 + 3 * sigma, -1 - 3 * sigma
    pyx1, interval_x = channel_transition_probability_table(q_uniform, lo, hi, 1, sigma)
    pyxm, _ = channel_transition_probability_table(q_uniform, lo, hi, -1, sigma)
    joint = np.zeros((2, q_uniform)).astype(np.float32)
    joint[0], joint[1] = pyx1, pyxm
    _, _, Az, _ = mmi_quantize_batch(joint[None].astype(np.float64), q_channel, device, sort=False)
    channel_lut = Az[0].astype(np.int64)
    pzx = np.zeros((2, q_channel))
    for i in range(q_channel):
        pzx[0, i] = np.sum(pyx1[channel_lut[i]:channel_lut[i + 1]])
        pzx[1, i] = np.sum(pyxm[channel_lut[i]:channel_lut[i + 1]])
    return pzx, interval_x, channel_lut


def channel_llr_density_table(M, low, high, mu1, mu2, sigma):
    """utils.py:30-44 of the reference: density and centroid of M uniform LLR cells on [low, high] under the equiprobable
    mixture N(mu1, sigma^2) / N(mu2, sigma^2), integrated on a 1e-4 grid like channel_transition_probability_table."""
    delta = 0.0001
    x = np.arange(low, high + delta, delta)
    pdf = 0.5 * (1 / np.sqrt(2 * np.pi * sigma ** 2) * np.exp(-(x - mu1) ** 2 / (2 * sigma ** 2)) +
                 1 / np.sqrt(2 * np.pi * sigma ** 2) * np.exp(-(x - mu2) ** 2 / (2 * sigma ** 2)))
    edges = np.linspace(low, high, M + 1)
    quanta, pyx = np.zeros(M), np.zeros(M)
    for i in range(M):
        sel = np.bitwise_and(x >= edges[i], x <= edges[i + 1])
        d = pdf[sel]
        pyx[i] = np.sum(d) * delta
        quanta[i] = np.sum(x[sel] * d) / np.sum(d)
    return pyx, edges, quanta


def llr_channel_quantizer(sigma, q_uniform=128, q_channel=16, device=0):
    """The channel quantizer the LLR-domain driver builds for a noise level (mainQuantizedDecoder_LLRDomain.py:143-145):
    q_uniform uniform LLR cells on [-E-3D, E+3D] (E = 2/sigma^2, D = sqrt(2E)) merged to q_channel symbols by the
    minimum-distortion quantizer (LLRQuantizer.find_OptLS_quantizer, here optls_quantize_batch).  The counterpart of
    mmi_channel_quantizer.  -> cell edges interval_x [q_uniform+1] float64, channel_lut [q_uniform] uint8: the arguments of
    simulate.LLRQuantizer."""
    E = 2 / sigma ** 2
    D = np.sqrt(2 * E)
    pyx, interval_x, quanta = channel_llr_density_table(q_uniform, -E - 3 * D, E + 3 * D, E, -E, D)
    _, _, luts = optls_quantize_batch([pyx], [quanta], q_channel, device)
    return interval_x, luts[0].astype(np.uint8)
