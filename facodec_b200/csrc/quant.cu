// Quantizer-side kernels: fused factorised / residual VQ (+ timbre AdaLN), WaveNet and
// StyleEncoder glue, 2-head self-attention, pooling, transposes.
//
// The VQ follows dac/nn/quantize.py:58-94 (VectorQuantize.forward / decode_latents) and
// :127-198 (ResidualVectorQuantize.forward, eval), which is arithmetic-identical to
// quantize/fvq.py:35-116 + quantize/rvq.py:27-75; FAquantizer.forward_v2
// (modules/quantize.py:375-454) chains three RVQs and a LayerNorm*gamma+beta per frame.
// Every step is per-frame, so ONE warp owns ONE frame: the 1024-dim residual lives in
// registers (32 per lane), the 1024->8 projection is a warp-shuffle reduction, the 1024-way
// argmin is lane-strided with a (score, index) shuffle reduction (ties -> lowest index, like
// torch.max on CPU), and the 8->1024 out-projection updates the residual in place.
#include "common.cuh"
#include "kernels.h"

namespace fac {

constexpr int VQ_D = 1024;
constexpr int VQ_CD = 8;
constexpr int VQ_N = 1024;

__device__ __forceinline__ void load_frame(const float* __restrict__ p, float (&v)[32], int lane) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        float4 t = *reinterpret_cast<const float4*>(p + i * 128 + lane * 4);
        v[i * 4 + 0] = t.x; v[i * 4 + 1] = t.y; v[i * 4 + 2] = t.z; v[i * 4 + 3] = t.w;
    }
}
__device__ __forceinline__ void store_frame(float* __restrict__ p, const float (&v)[32], int lane) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
        *reinterpret_cast<float4*>(p + i * 128 + lane * 4) = make_float4(v[i * 4], v[i * 4 + 1], v[i * 4 + 2], v[i * 4 + 3]);
}

// out_proj (8 -> 1024) of F frames at once, channel chunk i (c = i*128 + lane*4 + 0..3):
// o[f] = b_out + sum_k w_out[k] * zq[f][k], fmaf in k order; each w_out slice is loaded once for all F frames.
template <int F>
__device__ __forceinline__ void out_proj_chunk(const VqWeights& W, const float (&zq)[F][VQ_CD], int i, int lane,
                                               float4 (&o)[F]) {
    const float4 bo = __ldg(reinterpret_cast<const float4*>(W.b_out + i * 128 + lane * 4));
#pragma unroll
    for (int f = 0; f < F; ++f) o[f] = bo;
#pragma unroll
    for (int k = 0; k < VQ_CD; ++k) {
        const float4 w = __ldg(reinterpret_cast<const float4*>(W.w_out + k * VQ_D + i * 128 + lane * 4));
#pragma unroll
        for (int f = 0; f < F; ++f) {
            o[f].x = fmaf(w.x, zq[f][k], o[f].x);
            o[f].y = fmaf(w.y, zq[f][k], o[f].y);
            o[f].z = fmaf(w.z, zq[f][k], o[f].z);
            o[f].w = fmaf(w.w, zq[f][k], o[f].w);
        }
    }
}

// FAquantizer.forward_v2 tail on one frame (modules/quantize.py:445-449), in place: timbre_norm = LayerNorm(1024, no
// affine, eps 1e-5), then * gamma + beta with gb = [gamma[1024] | beta[1024]] of the frame's utterance.
__device__ __forceinline__ void ada_ln(float (&v)[32], const float* __restrict__ gb, int lane) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) s += v[i];
    float mean = warp_sum(s) * (1.0f / VQ_D);
    float var = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        float d = v[i] - mean;
        var = fmaf(d, d, var);
    }
    float rstd = rsqrtf(warp_sum(var) * (1.0f / VQ_D) + 1e-5f);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        float4 g = __ldg(reinterpret_cast<const float4*>(gb + i * 128 + lane * 4));
        float4 be = __ldg(reinterpret_cast<const float4*>(gb + VQ_D + i * 128 + lane * 4));
        v[i * 4 + 0] = (v[i * 4 + 0] - mean) * rstd * g.x + be.x;
        v[i * 4 + 1] = (v[i * 4 + 1] - mean) * rstd * g.y + be.y;
        v[i * 4 + 2] = (v[i * 4 + 2] - mean) * rstd * g.z + be.z;
        v[i * 4 + 3] = (v[i * 4 + 3] - mean) * rstd * g.w + be.w;
    }
}

// One VectorQuantize.forward on the frame held in r (channel c = i*128 + lane*4 + j <-> r[i*4+j]).
// Writes out[] = out_proj(z_q), returns the code index; sqerr = sum_k (z_e - z_q)^2.
__device__ __forceinline__ int vq_stage(const VqWeights& W, const float (&r)[32], float (&out)[32], float& sqerr,
                                        int lane) {
    float ze[VQ_CD];
#pragma unroll
    for (int k = 0; k < VQ_CD; ++k) {
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float4 w = __ldg(reinterpret_cast<const float4*>(W.w_in + k * VQ_D + i * 128 + lane * 4));
            acc = fmaf(w.x, r[i * 4], acc);
            acc = fmaf(w.y, r[i * 4 + 1], acc);
            acc = fmaf(w.z, r[i * 4 + 2], acc);
            acc = fmaf(w.w, r[i * 4 + 3], acc);
        }
        ze[k] = warp_sum(acc) + __ldg(W.b_in + k);
    }
    // F.normalize(encodings): x / max(||x||_2, 1e-12)
    float n2 = 0.f;
#pragma unroll
    for (int k = 0; k < VQ_CD; ++k) n2 = fmaf(ze[k], ze[k], n2);
    float nrm = fmaxf(sqrtf(n2), 1e-12f);
    float en[VQ_CD];
    float e2 = 0.f;
#pragma unroll
    for (int k = 0; k < VQ_CD; ++k) {
        en[k] = ze[k] / nrm;
        e2 = fmaf(en[k], en[k], e2);
    }
    // dist = e2 - (2 enc) @ cb^T + c2 ; indices = argmax(-dist), first maximum wins
    float best = -3.0e38f;
    int bidx = 0;
#pragma unroll 4
    for (int m = 0; m < VQ_N / 32; ++m) {
        int j = lane + 32 * m;
        float4 c0 = __ldg(reinterpret_cast<const float4*>(W.cbn + j * VQ_CD));
        float4 c1 = __ldg(reinterpret_cast<const float4*>(W.cbn + j * VQ_CD + 4));
        float dot = en[0] * c0.x;
        dot = fmaf(en[1], c0.y, dot);
        dot = fmaf(en[2], c0.z, dot);
        dot = fmaf(en[3], c0.w, dot);
        dot = fmaf(en[4], c1.x, dot);
        dot = fmaf(en[5], c1.y, dot);
        dot = fmaf(en[6], c1.z, dot);
        dot = fmaf(en[7], c1.w, dot);
        float d = (e2 - 2.0f * dot) + __ldg(W.cbn2 + j);
        float s = -d;
        if (s > best) { best = s; bidx = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float os = __shfl_xor_sync(0xffffffffu, best, o);
        int oj = __shfl_xor_sync(0xffffffffu, bidx, o);
        if (os > best || (os == best && oj < bidx)) { best = os; bidx = oj; }
    }
    float4 q0 = __ldg(reinterpret_cast<const float4*>(W.cb + bidx * VQ_CD));
    float4 q1 = __ldg(reinterpret_cast<const float4*>(W.cb + bidx * VQ_CD + 4));
    float zq[1][VQ_CD] = {{q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w}};
    float se = 0.f;
#pragma unroll
    for (int k = 0; k < VQ_CD; ++k) {
        float df = ze[k] - zq[0][k];
        se = fmaf(df, df, se);
        zq[0][k] = ze[k] + (zq[0][k] - ze[k]);   // straight-through estimator, forward value
    }
    sqerr = se;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        float4 o[1];
        out_proj_chunk<1>(W, zq, i, lane, o);
        out[i * 4] = o[0].x; out[i * 4 + 1] = o[0].y; out[i * 4 + 2] = o[0].z; out[i * 4 + 3] = o[0].w;
    }
    return bidx;
}

// FAquantizer.forward_v2 per frame (eval): prosody RVQ(1) on f0, content RVQ(n_c) on z,
// residual RVQ(3) on z - z_p - z_c, outs = LN(z_p + z_c + z_r) * gamma + beta.
__global__ void __launch_bounds__(128) fa_quantize_kernel(FaqParams p) {
    const int lane = threadIdx.x & 31;
    const int frame = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int nframes = p.B * p.Tq;
    if (frame >= nframes) return;
    const int b = frame / p.Tq, t = frame - b * p.Tq;
    const size_t fo = (size_t)frame * VQ_D;

    float r[32], out[32], zp[32], zc[32];
    float se;
    // prosody
    load_frame(p.f0 + ((size_t)b * p.Tf0 + t) * VQ_D, r, lane);
    int idx = vq_stage(p.vq[0], r, zp, se, lane);
    if (lane == 0) {
        p.codes_p[(size_t)b * p.Tq + t] = idx;
        p.sqerr[(size_t)0 * nframes + frame] = se;
    }
    if (p.zp) store_frame(p.zp + fo, zp, lane);
    // content
    float x[32];
    load_frame(p.z + ((size_t)b * p.Tz + t) * VQ_D, x, lane);
#pragma unroll
    for (int i = 0; i < 32; ++i) r[i] = x[i];
    idx = vq_stage(p.vq[1], r, zc, se, lane);
    if (lane == 0) {
        p.codes_c[((size_t)b * p.n_c + 0) * p.Tq + t] = idx;
        p.sqerr[(size_t)1 * nframes + frame] = se;
    }
    if (p.n_c > 1) {
#pragma unroll
        for (int i = 0; i < 32; ++i) r[i] -= zc[i];
        idx = vq_stage(p.vq[2], r, out, se, lane);
#pragma unroll
        for (int i = 0; i < 32; ++i) zc[i] += out[i];
        if (lane == 0) {
            p.codes_c[((size_t)b * p.n_c + 1) * p.Tq + t] = idx;
            p.sqerr[(size_t)2 * nframes + frame] = se;
        }
    } else if (lane == 0) {
        p.sqerr[(size_t)2 * nframes + frame] = 0.f;
    }
    if (p.zc) store_frame(p.zc + fo, zc, lane);
    // residual feature = x - z_p - z_c
#pragma unroll
    for (int i = 0; i < 32; ++i) r[i] = (x[i] - zp[i]) - zc[i];
    float zr[32];
    idx = vq_stage(p.vq[3], r, zr, se, lane);
    if (lane == 0) {
        p.codes_r[((size_t)b * 3 + 0) * p.Tq + t] = idx;
        p.sqerr[(size_t)3 * nframes + frame] = se;
    }
#pragma unroll
    for (int q = 1; q < 3; ++q) {
#pragma unroll
        for (int i = 0; i < 32; ++i) r[i] -= (q == 1 ? zr[i] : out[i]);
        idx = vq_stage(p.vq[3 + q], r, out, se, lane);
#pragma unroll
        for (int i = 0; i < 32; ++i) zr[i] += out[i];
        if (lane == 0) {
            p.codes_r[((size_t)b * 3 + q) * p.Tq + t] = idx;
            p.sqerr[(size_t)(3 + q) * nframes + frame] = se;
        }
    }
    if (p.zr) store_frame(p.zr + fo, zr, lane);
    // outs = z_p + z_c + z_r ; timbre_norm = LayerNorm(1024, no affine), eps 1e-5 ; * gamma + beta
#pragma unroll
    for (int i = 0; i < 32; ++i) out[i] = (zp[i] + zc[i]) + zr[i];
    ada_ln(out, p.gamma_beta + (size_t)b * 2 * VQ_D, lane);
    store_frame(p.outs + fo, out, lane);
}

cudaError_t launch_fa_quantize(const FaqParams& p, cudaStream_t st) {
    int nframes = p.B * p.Tq;
    if (nframes <= 0) return cudaSuccess;
    fa_quantize_kernel<<<(nframes + 3) / 4, 128, 0, st>>>(p);
    return cudaGetLastError();
}

// Decoding from codes: ResidualVectorQuantize.from_codes (dac/nn/quantize.py:200-220) of the prosody, content and
// residual quantizers, then the forward_v2 tail (modules/quantize.py:435-449).  Per group z_g = 0 + sum_q (W_out_q
// cb_q[idx_q] + b_out_q) in codebook order, on the RAW codebook row (there is no z_e to straight-through against);
// outs = (z_p + z_c) + z_r with z_r = 0 when n_r = 0; then ada_ln as fa_quantize_kernel.  One warp owns DQ_F consecutive
// frames (lane/channel map of fa_quantize_kernel), so each w_out slice is read once per DQ_F frames (the rvq_kernel
// lesson).  The work is chunked by channel slice i: the three group sums of one slice only need four registers per frame,
// and the codebook rows (32 bytes, the same address for the whole warp) are re-read per slice from L1.  DQ_F = 2: the
// 32-channel outs of four frames in registers need more than 255 registers and spill (ptxas -v); two use 226, no spills.
// An index outside [0, 1024) is never used as an address: it reads as NaN, and every channel of that frame's outs is NaN.
constexpr int DQ_F = 2;
__global__ void __launch_bounds__(128) dequantize_kernel(DequantParams p) {
    const int lane = threadIdx.x & 31;
    const size_t nframes = (size_t)p.B * p.T;
    const size_t f0 = ((size_t)blockIdx.x * 4 + (threadIdx.x >> 5)) * DQ_F;
    if (f0 >= nframes) return;
    size_t fr[DQ_F];
    int bu[DQ_F];
    int idx[DQ_F][6];      // codebook row per VQ (prosody, content0, content1, residual0..2); -1 = out of range
    bool bad[DQ_F];
#pragma unroll
    for (int f = 0; f < DQ_F; ++f) {
        fr[f] = f0 + f < nframes ? f0 + f : nframes - 1;   // tail: duplicate the last frame, store only valid ones
        const int b = (int)(fr[f] / p.T), t = (int)(fr[f] - (size_t)b * p.T);
        bu[f] = b;
        long long raw[6];
        raw[0] = p.codes_p[(size_t)b * p.T + t];
#pragma unroll
        for (int q = 0; q < 2; ++q) raw[1 + q] = q < p.n_c ? p.codes_c[((size_t)b * p.n_c_rows + q) * p.T + t] : 0;
#pragma unroll
        for (int q = 0; q < 3; ++q) raw[3 + q] = q < p.n_r ? p.codes_r[((size_t)b * p.n_r_rows + q) * p.T + t] : 0;
        bad[f] = false;
#pragma unroll
        for (int q = 0; q < 6; ++q) {
            const bool ok = raw[q] >= 0 && raw[q] < VQ_N;
            idx[f][q] = ok ? (int)raw[q] : -1;
            bad[f] |= !ok;
        }
    }
    // one group's slice i: g[f] = 0 + sum over the group's first nq VQs (compile-time indices q0 .. q0 + 2)
    auto group = [&](int q0, int nq, int i, float4 (&g)[DQ_F]) {
#pragma unroll
        for (int f = 0; f < DQ_F; ++f) g[f] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int q = q0; q < q0 + 3 && q < 6; ++q) {
            if (q - q0 >= nq) break;
            const VqWeights& W = p.vq[q];
            float zq[DQ_F][VQ_CD];
#pragma unroll
            for (int f = 0; f < DQ_F; ++f) {
                const int j = idx[f][q];
                float4 c0 = make_float4(__int_as_float(0x7fffffff), __int_as_float(0x7fffffff), __int_as_float(0x7fffffff),
                                        __int_as_float(0x7fffffff));
                float4 c1 = c0;
                if (j >= 0) {
                    c0 = __ldg(reinterpret_cast<const float4*>(W.cb + j * VQ_CD));
                    c1 = __ldg(reinterpret_cast<const float4*>(W.cb + j * VQ_CD + 4));
                }
                zq[f][0] = c0.x; zq[f][1] = c0.y; zq[f][2] = c0.z; zq[f][3] = c0.w;
                zq[f][4] = c1.x; zq[f][5] = c1.y; zq[f][6] = c1.z; zq[f][7] = c1.w;
            }
            float4 o[DQ_F];
            out_proj_chunk<DQ_F>(W, zq, i, lane, o);
#pragma unroll
            for (int f = 0; f < DQ_F; ++f) {
                g[f].x += o[f].x; g[f].y += o[f].y; g[f].z += o[f].z; g[f].w += o[f].w;
            }
        }
    };
    auto store4 = [&](float* base, int f, int i, const float4& v) {
        if (base && f0 + f < nframes) *reinterpret_cast<float4*>(base + fr[f] * VQ_D + i * 128 + lane * 4) = v;
    };
    float outs[DQ_F][32];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        float4 g[DQ_F];
        group(0, 1, i, g);                              // z_p
#pragma unroll
        for (int f = 0; f < DQ_F; ++f) {
            outs[f][i * 4] = g[f].x; outs[f][i * 4 + 1] = g[f].y; outs[f][i * 4 + 2] = g[f].z; outs[f][i * 4 + 3] = g[f].w;
            store4(p.zp, f, i, g[f]);
        }
        group(1, p.n_c, i, g);                          // z_c
#pragma unroll
        for (int f = 0; f < DQ_F; ++f) {
            outs[f][i * 4] += g[f].x; outs[f][i * 4 + 1] += g[f].y; outs[f][i * 4 + 2] += g[f].z; outs[f][i * 4 + 3] += g[f].w;
            store4(p.zc, f, i, g[f]);
        }
        group(3, p.n_r, i, g);                          // z_r (zeros when n_r = 0)
#pragma unroll
        for (int f = 0; f < DQ_F; ++f) {
            outs[f][i * 4] += g[f].x; outs[f][i * 4 + 1] += g[f].y; outs[f][i * 4 + 2] += g[f].z; outs[f][i * 4 + 3] += g[f].w;
            store4(p.zr, f, i, g[f]);
        }
    }
#pragma unroll
    for (int f = 0; f < DQ_F; ++f) {
        ada_ln(outs[f], p.gamma_beta + (size_t)bu[f] * 2 * VQ_D, lane);
        if (bad[f]) {
#pragma unroll
            for (int i = 0; i < 32; ++i) outs[f][i] = __int_as_float(0x7fffffff);
        }
        if (f0 + f < nframes) store_frame(p.outs + fr[f] * VQ_D, outs[f], lane);
    }
}

cudaError_t launch_dequantize(const DequantParams& p, cudaStream_t st) {
    const size_t nframes = (size_t)p.B * p.T;
    if (nframes == 0) return cudaSuccess;
    if (p.n_c < 1 || p.n_c > 2 || p.n_r < 0 || p.n_r > 3) return cudaErrorInvalidValue;
    const size_t per_cta = 4 * DQ_F;
    const size_t nblk = (nframes + per_cta - 1) / per_cta;
    if (nblk > 0x7fffffffULL) return cudaErrorInvalidValue;
    dequantize_kernel<<<(unsigned)nblk, 128, 0, st>>>(p);
    return cudaGetLastError();
}

// commitment = codebook (forward values) = sum_q mean_b( sum_t sqerr / (8 Tq) ), fixed order, fp64
__global__ void vq_loss_reduce_kernel(const float* __restrict__ sqerr, int nq, int B, int Tq, float* losses2) {
    __shared__ double part[256];
    double total = 0.0;
    for (int q = 0; q < nq; ++q) {
        double acc = 0.0;
        for (int i = threadIdx.x; i < B * Tq; i += blockDim.x) acc += (double)sqerr[(size_t)q * B * Tq + i];
        part[threadIdx.x] = acc;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (threadIdx.x < o) part[threadIdx.x] += part[threadIdx.x + o];
            __syncthreads();
        }
        total += part[0] / ((double)VQ_CD * Tq * B);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        losses2[0] = (float)total;
        losses2[1] = (float)total;
    }
}
cudaError_t launch_vq_loss_reduce(const float* sqerr, int nq, int B, int Tq, float* losses2, cudaStream_t st) {
    vq_loss_reduce_kernel<<<1, 256, 0, st>>>(sqerr, nq, B, Tq, losses2);
    return cudaGetLastError();
}

// Generic residual VQ (quantize/rvq.py:27-75 over quantize/fvq.py:35-83, eval), BASELINE configs[3].
// One warp owns F = 4 consecutive frames at once: the first version (one frame per warp, vq_stage above) re-read the 96 KB
// of projection / codebook weights of every stage through L1 for every single frame and ran at the LSU's bandwidth
// (41 Mframes/s = 0.05 of the HBM roofline, bench.py --workload vq); with four frames in registers each weight vector is
// loaded once per four frames.  Same arithmetic per frame as vq_stage (same reduction orders): indices are bit-identical.
constexpr int RVQ_F = 4;
__global__ void __launch_bounds__(128) rvq_kernel(RvqParams p) {
    const int lane = threadIdx.x & 31;
    const size_t nframes = (size_t)p.B * p.T;
    const size_t f0 = ((size_t)blockIdx.x * 4 + (threadIdx.x >> 5)) * RVQ_F;
    if (f0 >= nframes) return;
    float r[RVQ_F][32];
    size_t fr[RVQ_F];
#pragma unroll
    for (int f = 0; f < RVQ_F; ++f) {
        fr[f] = f0 + f < nframes ? f0 + f : nframes - 1;        // tail: duplicate the last frame, store only valid ones
        load_frame(p.x + fr[f] * VQ_D, r[f], lane);
    }
    for (int q = 0; q < p.nq; ++q) {
        const VqWeights& W = p.vq[q];
        // ---- in_proj 1024 -> 8 ----
        float ze[RVQ_F][VQ_CD];
#pragma unroll
        for (int k = 0; k < VQ_CD; ++k) {
            float acc[RVQ_F];
#pragma unroll
            for (int f = 0; f < RVQ_F; ++f) acc[f] = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 w = __ldg(reinterpret_cast<const float4*>(W.w_in + k * VQ_D + i * 128 + lane * 4));
#pragma unroll
                for (int f = 0; f < RVQ_F; ++f) {
                    acc[f] = fmaf(w.x, r[f][i * 4], acc[f]);
                    acc[f] = fmaf(w.y, r[f][i * 4 + 1], acc[f]);
                    acc[f] = fmaf(w.z, r[f][i * 4 + 2], acc[f]);
                    acc[f] = fmaf(w.w, r[f][i * 4 + 3], acc[f]);
                }
            }
            const float bk = __ldg(W.b_in + k);
#pragma unroll
            for (int f = 0; f < RVQ_F; ++f) ze[f][k] = warp_sum(acc[f]) + bk;
        }
        // ---- F.normalize, distances, argmax(-dist) (first maximum wins) ----
        float en[RVQ_F][VQ_CD], e2[RVQ_F], best[RVQ_F];
        int bidx[RVQ_F];
#pragma unroll
        for (int f = 0; f < RVQ_F; ++f) {
            float n2 = 0.f;
#pragma unroll
            for (int k = 0; k < VQ_CD; ++k) n2 = fmaf(ze[f][k], ze[f][k], n2);
            const float nrm = fmaxf(sqrtf(n2), 1e-12f);
            e2[f] = 0.f;
#pragma unroll
            for (int k = 0; k < VQ_CD; ++k) { en[f][k] = ze[f][k] / nrm; e2[f] = fmaf(en[f][k], en[f][k], e2[f]); }
            best[f] = -3.0e38f; bidx[f] = 0;
        }
#pragma unroll 2
        for (int m = 0; m < VQ_N / 32; ++m) {
            const int j = lane + 32 * m;
            const float4 c0 = __ldg(reinterpret_cast<const float4*>(W.cbn + j * VQ_CD));
            const float4 c1 = __ldg(reinterpret_cast<const float4*>(W.cbn + j * VQ_CD + 4));
            const float c2 = __ldg(W.cbn2 + j);
#pragma unroll
            for (int f = 0; f < RVQ_F; ++f) {
                float dot = en[f][0] * c0.x;
                dot = fmaf(en[f][1], c0.y, dot);
                dot = fmaf(en[f][2], c0.z, dot);
                dot = fmaf(en[f][3], c0.w, dot);
                dot = fmaf(en[f][4], c1.x, dot);
                dot = fmaf(en[f][5], c1.y, dot);
                dot = fmaf(en[f][6], c1.z, dot);
                dot = fmaf(en[f][7], c1.w, dot);
                const float sc = -((e2[f] - 2.0f * dot) + c2);
                if (sc > best[f]) { best[f] = sc; bidx[f] = j; }
            }
        }
#pragma unroll
        for (int f = 0; f < RVQ_F; ++f) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float os = __shfl_xor_sync(0xffffffffu, best[f], o);
                const int oj = __shfl_xor_sync(0xffffffffu, bidx[f], o);
                if (os > best[f] || (os == best[f] && oj < bidx[f])) { best[f] = os; bidx[f] = oj; }
            }
            if (lane == 0 && f0 + f < nframes) p.idx[(size_t)q * nframes + f0 + f] = bidx[f];
        }
        // ---- z_q = codebook[idx] (straight-through forward value), out_proj 8 -> 1024, residual update ----
        float zq[RVQ_F][VQ_CD];
#pragma unroll
        for (int f = 0; f < RVQ_F; ++f) {
            const float4 q0 = __ldg(reinterpret_cast<const float4*>(W.cb + bidx[f] * VQ_CD));
            const float4 q1 = __ldg(reinterpret_cast<const float4*>(W.cb + bidx[f] * VQ_CD + 4));
            const float t[VQ_CD] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
            for (int k = 0; k < VQ_CD; ++k) zq[f][k] = ze[f][k] + (t[k] - ze[f][k]);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 bo = __ldg(reinterpret_cast<const float4*>(W.b_out + i * 128 + lane * 4));
            float4 o[RVQ_F];
#pragma unroll
            for (int f = 0; f < RVQ_F; ++f) o[f] = bo;
#pragma unroll
            for (int k = 0; k < VQ_CD; ++k) {
                const float4 w = __ldg(reinterpret_cast<const float4*>(W.w_out + k * VQ_D + i * 128 + lane * 4));
#pragma unroll
                for (int f = 0; f < RVQ_F; ++f) {
                    o[f].x = fmaf(w.x, zq[f][k], o[f].x);
                    o[f].y = fmaf(w.y, zq[f][k], o[f].y);
                    o[f].z = fmaf(w.z, zq[f][k], o[f].z);
                    o[f].w = fmaf(w.w, zq[f][k], o[f].w);
                }
            }
#pragma unroll
            for (int f = 0; f < RVQ_F; ++f) {
                r[f][i * 4] -= o[f].x; r[f][i * 4 + 1] -= o[f].y; r[f][i * 4 + 2] -= o[f].z; r[f][i * 4 + 3] -= o[f].w;
                if (p.allq && f0 + f < nframes)
                    *reinterpret_cast<float4*>(p.allq + ((size_t)q * nframes + f0 + f) * VQ_D + i * 128 + lane * 4) = o[f];
            }
        }
    }
    // quantized_out = sum of the stages' outputs = x - final residual, re-summed in the reference's order is not needed: the
    // stage outputs were subtracted one by one (r = ((x - o1) - o2) - ...), so x - r differs from o1 + o2 + ... by fp32
    // round-off (<= 1e-6 here); both are inside the 1e-5 bar of the parity tests.
#pragma unroll
    for (int f = 0; f < RVQ_F; ++f) {
        if (f0 + f >= nframes) break;
        const float* xp = p.x + (f0 + f) * VQ_D;
        float* qp = p.qout + (f0 + f) * VQ_D;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 xv = *reinterpret_cast<const float4*>(xp + i * 128 + lane * 4);
            *reinterpret_cast<float4*>(qp + i * 128 + lane * 4) =
                make_float4(xv.x - r[f][i * 4], xv.y - r[f][i * 4 + 1], xv.z - r[f][i * 4 + 2], xv.w - r[f][i * 4 + 3]);
        }
    }
}
cudaError_t launch_rvq(const RvqParams& p, cudaStream_t st) {
    size_t nframes = (size_t)p.B * p.T;
    if (nframes == 0) return cudaSuccess;
    const size_t per_cta = 4 * RVQ_F;
    const size_t nblk = (nframes + per_cta - 1) / per_cta;
    if (nblk > 0x7fffffffULL) return cudaErrorInvalidValue;
    rvq_kernel<<<(unsigned)nblk, 128, 0, st>>>(p);
    return cudaGetLastError();
}

// ---- small ops -------------------------------------------------------------------------------
__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int R, int C) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const float* ib = in + (size_t)b * R * C;
    float* ob = out + (size_t)b * R * C;
    int c = blockIdx.x * 32 + threadIdx.x;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int r = blockIdx.y * 32 + i;
        if (r < R && c < C) tile[i][threadIdx.x] = ib[(size_t)r * C + c];
    }
    __syncthreads();
    int r2 = blockIdx.y * 32 + threadIdx.x;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int c2 = blockIdx.x * 32 + i;
        if (r2 < R && c2 < C) ob[(size_t)c2 * R + r2] = tile[threadIdx.x][i];
    }
}
cudaError_t launch_transpose(const float* in, float* out, int B, int R, int C, cudaStream_t st) {
    if (B <= 0 || R <= 0 || C <= 0) return cudaSuccess;
    if ((R + 31) / 32 > 65535) return cudaErrorInvalidValue;
    dim3 block(32, 8);
    for (int b0 = 0; b0 < B; b0 += 65535) {     // grid.z is limited to 65535
        const int nb = B - b0 < 65535 ? B - b0 : 65535;
        dim3 grid((C + 31) / 32, (R + 31) / 32, nb);
        transpose_kernel<<<grid, block, 0, st>>>(in + (size_t)b0 * R * C, out + (size_t)b0 * R * C, R, C);
    }
    return cudaGetLastError();
}

// fused_add_tanh_sigmoid_multiply (modules/commons.py:113-120): acts = tanh(x_in[:H] + g_l[:H]) * sigmoid(x_in[H:] + g_l[H:]).
// g (or null = zeros, the codec's own WN call) is the layer's slice of cond_layer(g) (modules/wavenet.py:143-151): one
// [2H] row per utterance, utterance = row / rows_per_utt, consecutive utterances g_stride floats apart.
__global__ void wn_gate_kernel(const float* __restrict__ xin, float* __restrict__ acts, size_t n_rows, int hidden,
                               const float* __restrict__ g, size_t rows_per_utt, size_t g_stride) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows * hidden) return;
    size_t row = i / hidden;
    int c = (int)(i - row * hidden);
    float ga = 0.0f, gs = 0.0f;
    if (g) {
        const float* gr = g + (row / rows_per_utt) * g_stride;
        ga = gr[c]; gs = gr[hidden + c];
    }
    float a = xin[row * 2 * hidden + c] + ga;
    float s = xin[row * 2 * hidden + hidden + c] + gs;
    acts[i] = tanhf(a) * sigmoid_f(s);
}
cudaError_t launch_wn_gate(const float* xin, float* acts, size_t n_rows, int hidden, cudaStream_t st, const float* g,
                           size_t rows_per_utt, size_t g_stride) {
    size_t n = n_rows * hidden;
    if (n == 0) return cudaSuccess;
    wn_gate_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(xin, acts, n_rows, hidden, g, rows_per_utt ? rows_per_utt : 1, g_stride);
    return cudaGetLastError();
}
// WN.forward residual/skip split, modules/wavenet.py:159-165
__global__ void wn_update_kernel(const float* __restrict__ rs, float* __restrict__ x, float* __restrict__ out,
                                 size_t n_rows, int hidden, int last) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows * hidden) return;
    size_t row = i / hidden;
    int c = (int)(i - row * hidden);
    if (!last) {
        x[i] = x[i] + rs[row * 2 * hidden + c];
        out[i] = out[i] + rs[row * 2 * hidden + hidden + c];
    } else {
        out[i] = out[i] + rs[row * hidden + c];
    }
}
cudaError_t launch_wn_update(const float* rs, float* x, float* out, size_t n_rows, int hidden, int last,
                             cudaStream_t st) {
    size_t n = n_rows * hidden;
    if (n == 0) return cudaSuccess;
    wn_update_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(rs, x, out, n_rows, hidden, last);
    return cudaGetLastError();
}

// Conv1dGLU tail (modules/style_encoder.py:26-31): x = x + y[:C] * sigmoid(y[C:]), optional mask
__global__ void glu_res_kernel(const float* __restrict__ y, float* __restrict__ x, int T, int C,
                               const int* __restrict__ valid_len) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    int b = blockIdx.y;
    if (i >= (size_t)T * C) return;
    int t = (int)(i / C), c = (int)(i - (size_t)t * C);
    size_t row = (size_t)b * T + t;
    float v = x[row * C + c] + y[row * 2 * C + c] * sigmoid_f(y[row * 2 * C + C + c]);
    if (valid_len && t >= valid_len[b]) v = 0.f;
    x[row * C + c] = v;
}
cudaError_t launch_glu_res(const float* y, float* x, int B, int T, int C, const int* valid_len, cudaStream_t st) {
    size_t n = (size_t)T * C;
    if (n == 0 || B <= 0) return cudaSuccess;
    dim3 grid((unsigned)((n + 255) / 256), B);
    glu_res_kernel<<<grid, 256, 0, st>>>(y, x, T, C, valid_len);
    return cudaGetLastError();
}

// MultiHeadAttention.attention (modules/attentions.py:168-199, window_size=None): per (b, head),
// 16 queries per CTA; K then V tiles of 32 rows staged in shared memory.
constexpr int ATT_Q = 16;
constexpr int ATT_DK = 256;
__global__ void __launch_bounds__(256) attention_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                        const float* __restrict__ v, float* __restrict__ o, int T,
                                                        int heads, const int* __restrict__ valid_len) {
    extern __shared__ __align__(16) float sm[];
    float* qs = sm;                              // [16][256]
    float* tile = qs + ATT_Q * ATT_DK;           // [32][257]
    float* sc = tile + 32 * (ATT_DK + 1);        // [16][T]
    const int C = heads * ATT_DK;
    const int bh = blockIdx.y, b = bh / heads, h = bh % heads;
    const int q0 = blockIdx.x * ATT_Q;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int vlen = valid_len ? valid_len[b] : T;
    const float* qb = q + (size_t)b * T * C + h * ATT_DK;
    const float* kb = k + (size_t)b * T * C + h * ATT_DK;
    const float* vb = v + (size_t)b * T * C + h * ATT_DK;
    for (int i = tid; i < ATT_Q * ATT_DK; i += 256) {
        int qi = i / ATT_DK, d = i % ATT_DK;
        int t = q0 + qi;
        qs[i] = (t < T) ? qb[(size_t)t * C + d] * (1.0f / 16.0f) : 0.f;   // query / sqrt(k_channels)
    }
    // ---- scores ----
    for (int s0 = 0; s0 < T; s0 += 32) {
        __syncthreads();
        for (int i = tid; i < 32 * ATT_DK; i += 256) {
            int r = i / ATT_DK, d = i % ATT_DK;
            tile[r * (ATT_DK + 1) + d] = (s0 + r < T) ? kb[(size_t)(s0 + r) * C + d] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int qq = 0; qq < 2; ++qq) {
            int qi = warp * 2 + qq;
            float acc = 0.f;
            const float* qr = qs + qi * ATT_DK;
            const float* kr = tile + lane * (ATT_DK + 1);
#pragma unroll 8
            for (int d = 0; d < ATT_DK; ++d) acc = fmaf(qr[d], kr[d], acc);
            int s = s0 + lane;
            if (s < T) {
                bool ok = (q0 + qi < vlen) && (s < vlen);
                sc[qi * T + s] = ok ? acc : -1e4f;
            }
        }
    }
    __syncthreads();
    // ---- softmax over keys (one warp per query row) ----
#pragma unroll
    for (int qq = 0; qq < 2; ++qq) {
        int qi = warp * 2 + qq;
        float* row = sc + qi * T;
        float mx = -3.0e38f;
        for (int s = lane; s < T; s += 32) mx = fmaxf(mx, row[s]);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
        float sum = 0.f;
        for (int s = lane; s < T; s += 32) {
            float e = expf(row[s] - mx);
            row[s] = e;
            sum += e;
        }
        sum = warp_sum(sum);
        float inv = 1.0f / sum;
        for (int s = lane; s < T; s += 32) row[s] *= inv;
    }
    // ---- out = P V ----
    float acc[2][8];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[a][j] = 0.f;
    for (int s0 = 0; s0 < T; s0 += 32) {
        __syncthreads();
        for (int i = tid; i < 32 * ATT_DK; i += 256) {
            int r = i / ATT_DK, d = i % ATT_DK;
            tile[r * (ATT_DK + 1) + d] = (s0 + r < T) ? vb[(size_t)(s0 + r) * C + d] : 0.f;
        }
        __syncthreads();
        int smax = min(32, T - s0);
        for (int s = 0; s < smax; ++s) {
            const float* vr = tile + s * (ATT_DK + 1);
#pragma unroll
            for (int qq = 0; qq < 2; ++qq) {
                float pw = sc[(warp * 2 + qq) * T + s0 + s];
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[qq][j] = fmaf(pw, vr[lane + 32 * j], acc[qq][j]);
            }
        }
    }
#pragma unroll
    for (int qq = 0; qq < 2; ++qq) {
        int t = q0 + warp * 2 + qq;
        if (t < T) {
            float* ob = o + ((size_t)b * T + t) * C + h * ATT_DK;
#pragma unroll
            for (int j = 0; j < 8; ++j) ob[lane + 32 * j] = acc[qq][j];
        }
    }
}
// Long sequences (the [16][T] score block above no longer fits shared memory, T > ~2700 frames = 34 s): same
// attention with the scores RECOMPUTED instead of stored.  Pass 1 walks the key tiles keeping a running row maximum and
// the sum of exp(s - max) (rescaled when the maximum moves); pass 2 recomputes each tile's scores, normalises them and
// accumulates P V.  Shared memory no longer depends on T; the probabilities differ from the stored-score kernel only by
// the rescaling round-off (~1e-7 relative).
__global__ void __launch_bounds__(256) attention_stream_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                               const float* __restrict__ v, float* __restrict__ o, int T,
                                                               int heads, const int* __restrict__ valid_len) {
    extern __shared__ __align__(16) float sm[];
    float* qs = sm;                              // [16][256]
    float* tile = qs + ATT_Q * ATT_DK;           // [32][257]
    float* pt = tile + 32 * (ATT_DK + 1);        // [16][32] probabilities of the current key tile
    const int C = heads * ATT_DK;
    const int bh = blockIdx.y, b = bh / heads, h = bh % heads;
    const int q0 = blockIdx.x * ATT_Q;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int vlen = valid_len ? valid_len[b] : T;
    const float* qb = q + (size_t)b * T * C + h * ATT_DK;
    const float* kb = k + (size_t)b * T * C + h * ATT_DK;
    const float* vb = v + (size_t)b * T * C + h * ATT_DK;
    for (int i = tid; i < ATT_Q * ATT_DK; i += 256) {
        int qi = i / ATT_DK, d = i % ATT_DK;
        int t = q0 + qi;
        qs[i] = (t < T) ? qb[(size_t)t * C + d] * (1.0f / 16.0f) : 0.f;
    }
    auto load_tile = [&](const float* base, int s0) {
        for (int i = tid; i < 32 * ATT_DK; i += 256) {
            int r = i / ATT_DK, d = i % ATT_DK;
            tile[r * (ATT_DK + 1) + d] = (s0 + r < T) ? base[(size_t)(s0 + r) * C + d] : 0.f;
        }
    };
    auto score = [&](int qi, int s0) {           // masked score of (query qi, key s0 + lane); -inf beyond T
        float acc = 0.f;
        const float* qr = qs + qi * ATT_DK;
        const float* kr = tile + lane * (ATT_DK + 1);
#pragma unroll 8
        for (int d = 0; d < ATT_DK; ++d) acc = fmaf(qr[d], kr[d], acc);
        const int s = s0 + lane;
        if (s >= T) return -3.0e38f;
        return ((q0 + qi < vlen) && (s < vlen)) ? acc : -1e4f;
    };
    float mrow[2] = {-3.0e38f, -3.0e38f}, lrow[2] = {0.f, 0.f};
    for (int s0 = 0; s0 < T; s0 += 32) {
        __syncthreads();
        load_tile(kb, s0);
        __syncthreads();
#pragma unroll
        for (int qq = 0; qq < 2; ++qq) {
            const float sc = score(warp * 2 + qq, s0);
            float mx = sc;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            const float mnew = fmaxf(mrow[qq], mx);
            const float e = (s0 + lane < T) ? expf(sc - mnew) : 0.f;
            lrow[qq] = lrow[qq] * expf(mrow[qq] - mnew) + warp_sum(e);
            mrow[qq] = mnew;
        }
    }
    float acc[2][8];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[a][j] = 0.f;
    const float inv0 = 1.0f / lrow[0], inv1 = 1.0f / lrow[1];
    for (int s0 = 0; s0 < T; s0 += 32) {
        __syncthreads();
        load_tile(kb, s0);
        __syncthreads();
#pragma unroll
        for (int qq = 0; qq < 2; ++qq) {
            const float sc = score(warp * 2 + qq, s0);
            pt[(warp * 2 + qq) * 32 + lane] = (s0 + lane < T) ? expf(sc - mrow[qq]) * (qq ? inv1 : inv0) : 0.f;
        }
        __syncthreads();
        load_tile(vb, s0);
        __syncthreads();
        const int smax = min(32, T - s0);
        for (int s = 0; s < smax; ++s) {
            const float* vr = tile + s * (ATT_DK + 1);
#pragma unroll
            for (int qq = 0; qq < 2; ++qq) {
                const float pw = pt[(warp * 2 + qq) * 32 + s];
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[qq][j] = fmaf(pw, vr[lane + 32 * j], acc[qq][j]);
            }
        }
    }
#pragma unroll
    for (int qq = 0; qq < 2; ++qq) {
        int t = q0 + warp * 2 + qq;
        if (t < T) {
            float* ob = o + ((size_t)b * T + t) * C + h * ATT_DK;
#pragma unroll
            for (int j = 0; j < 8; ++j) ob[lane + 32 * j] = acc[qq][j];
        }
    }
}
cudaError_t launch_attention(const float* q, const float* k, const float* v, float* o, int B, int T, int heads, int dk,
                             const int* valid_len, cudaStream_t st, int force_stream) {
    if (dk != ATT_DK) return cudaErrorInvalidValue;
    if (B <= 0 || T <= 0) return cudaSuccess;
    if ((long long)B * heads > 65535) return cudaErrorInvalidValue;
    size_t smem = sizeof(float) * ((size_t)ATT_Q * ATT_DK + 32 * (ATT_DK + 1) + (size_t)ATT_Q * T);
    dim3 grid((T + ATT_Q - 1) / ATT_Q, B * heads);
    if (smem > 200 * 1024 || force_stream) {
        smem = sizeof(float) * ((size_t)ATT_Q * ATT_DK + 32 * (ATT_DK + 1) + (size_t)ATT_Q * 32);
        cudaError_t e = cudaFuncSetAttribute(attention_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        attention_stream_kernel<<<grid, 256, smem, st>>>(q, k, v, o, T, heads, valid_len);
        return cudaGetLastError();
    }
    cudaError_t e = cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    attention_kernel<<<grid, 256, smem, st>>>(q, k, v, o, T, heads, valid_len);
    return cudaGetLastError();
}

// StyleEncoder.temporal_avg_pool (modules/style_encoder.py:83-91): sum over ALL frames / len
__global__ void mean_pool_kernel(const float* __restrict__ x, float* __restrict__ out, int T, int C,
                                 const int* __restrict__ valid_len) {
    int b = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float* xb = x + (size_t)b * T * C + c;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int t = 0;
    for (; t + 3 < T; t += 4) {
        a0 += xb[(size_t)t * C];
        a1 += xb[(size_t)(t + 1) * C];
        a2 += xb[(size_t)(t + 2) * C];
        a3 += xb[(size_t)(t + 3) * C];
    }
    for (; t < T; ++t) a0 += xb[(size_t)t * C];
    float len = (float)(valid_len ? valid_len[b] : T);
    out[(size_t)b * C + c] = ((a0 + a1) + (a2 + a3)) / len;
}
cudaError_t launch_mean_pool(const float* x, float* out, int B, int T, int C, const int* valid_len, cudaStream_t st) {
    if (B <= 0) return cudaSuccess;
    dim3 grid((C + 127) / 128, B);
    mean_pool_kernel<<<grid, 128, 0, st>>>(x, out, T, C, valid_len);
    return cudaGetLastError();
}

__global__ void fill_u32_kernel(unsigned int* p, unsigned int v, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
cudaError_t launch_fill_u32(unsigned int* p, unsigned int v, size_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    fill_u32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p, v, n);
    return cudaGetLastError();
}

}  // namespace fac
