// idelucs_b200 — the small latency-bound pieces of the training step that sit between the hot-path kernels and the
// PyTorch/cuBLAS MLP (idelucs/models.py:113-143), each one launch instead of a dozen framework kernels:
//
//   * idl_nce_*         InfoNCE / NT-Xent of idelucs/LossFunctions.py:65-98 on the stacked latent [2B, D], around two strict-fp32
//                       cuBLAS GEMMs issued by the caller (similarity fn fn^T and gradient W fn — dense contractions stay
//                       library calls): F.normalize; self-masked log-sum-exp + cross-entropy against the other view; the
//                       weights W = (P + P^T - 2 Y) / (2B T) written over the similarity in place; the normalisation's
//                       backward.  Four launches of ours + two GEMMs instead of ~25 framework kernels and three mask gathers;
//                       fixed-order reductions (run-to-run identical)
//   * idl_iid_loss      the IIC loss (LossFunctions.py:20-62) and its gradient: C <= 16 clusters in ONE ordinary CTA (the
//                       headline configuration has C = 5, i.e. a 5 x 5 joint); above that two contraction kernels around the
//                       launches of idl_iid_joint_algebra, the C x C algebra the Python layer calls between cuBLAS GEMMs
//   * idl_rmsprop_step  torch.optim.RMSprop's update (alpha, eps, weight_decay; no momentum, not centred — what
//                       idelucs/models.py:86 constructs) on a flat parameter shard in one elementwise pass, so that a
//                       data-parallel step can reduce-scatter the gradient, update 1/N of the parameters per rank and
//                       all-gather them
//   * idl_sgd_step / idl_adam_step  the other two optimisers of idelucs/models.py:86-99 (SGD with momentum, Adam), the step
//                       number read from device memory; the *_allreduce_step variants of all three share one NVLink kernel body
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>

#include "common.h"
#include "core.cuh"

namespace idl {

// ---------------------------------------------------------------------------------------------------------------
// InfoNCE
// ---------------------------------------------------------------------------------------------------------------
constexpr int NCE_NT = 256;          // 8 warps: warp <-> row
constexpr int NCE_RB = NCE_NT / 32;  // rows per CTA

// F.normalize(x, dim=1): x / max(||x||_2, 1e-12)
__global__ void __launch_bounds__(NCE_NT) nce_normalize_kernel(const float* __restrict__ h, int n2, int D, float* __restrict__ fn,
                                                                float* __restrict__ inv_norm) {
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * NCE_RB + (threadIdx.x >> 5);
    if (row >= n2) return;
    float ss = 0.f;
    for (int d = lane; d < D; d += 32) { const float v = h[(size_t)row * D + d]; ss = fmaf(v, v, ss); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);
    for (int d = lane; d < D; d += 32) fn[(size_t)row * D + d] = h[(size_t)row * D + d] * inv;
    if (lane == 0) inv_norm[row] = inv;
}

// Row pass over the similarity matrix S = fn fn^T (one strict-fp32 cuBLAS GEMM, 2B x 2B x D): lse_i = log sum_{j != i} exp(S_ij / T)
// and the row's loss term lse_i - S_i,pos(i) / T.  Warp <-> row, coalesced reads.  |S_ij / T| <= 1 / T, so exp needs no running
// maximum (T = 0.85: e^-1.18 .. e^1.18).
__global__ void __launch_bounds__(NCE_NT) nce_lse_kernel(const float* __restrict__ S, int n2, float inv_t, float* __restrict__ lse,
                                                          float* __restrict__ rowloss) {
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * NCE_RB + (threadIdx.x >> 5);
    if (i >= n2) return;
    const int half = n2 >> 1;
    const int pos = i < half ? i + half : i - half;
    const float* row = S + (size_t)i * n2;
    float sum = 0.f;
    for (int j = lane; j < n2; j += 32)
        if (j != i) sum += __expf(row[j] * inv_t);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);   // fixed tree: the same sum every run
    if (lane == 0) {
        const float l = logf(sum);
        lse[i] = l;
        rowloss[i] = l - row[pos] * inv_t;
    }
}

// In place: S_ij -> W_ij = (g / (n2 T)) (P_ij + P_ji - 2 [j == pos(i)]),  P_ij = exp(S_ij / T - lse_i), W_ii = 0, so that
// g d loss / d fn = W fn (a second GEMM; g = the caller's weight of this loss).  W is symmetric because S is.  CTA <-> NCE_WR rows,
// thread <-> four columns (n2 % 4 == 0; a scalar kernel takes other sizes).  Block 0 also reduces the loss (mean of the row terms).
constexpr int NCE_WR = 4;
__global__ void __launch_bounds__(256) nce_weights_kernel(float* __restrict__ S, const float* __restrict__ lse, const float* __restrict__ rowloss,
                                                           int n2, float inv_t, float gscale, float* __restrict__ loss) {
    const float c = gscale * inv_t / (float)n2;
    const int half = n2 >> 1;
    const int n4 = n2 >> 2;
    const int r0 = blockIdx.x * NCE_WR;
    for (int q = threadIdx.x; q < n4; q += 256) {
        const int j0 = q * 4;
        const float4 lj = *reinterpret_cast<const float4*>(lse + j0);
#pragma unroll
        for (int r = 0; r < NCE_WR; ++r) {
            const int i = r0 + r;
            if (i >= n2) break;
            float4* cell = reinterpret_cast<float4*>(S + (size_t)i * n2) + q;
            const float4 sv = *cell;
            const float li = lse[i];
            const int pos = i < half ? i + half : i - half;
            const float s[4] = {sv.x * inv_t, sv.y * inv_t, sv.z * inv_t, sv.w * inv_t};
            const float l4[4] = {lj.x, lj.y, lj.z, lj.w};
            float w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int j = j0 + e;
                w[e] = 0.f;
                if (j != i) {
                    w[e] = __expf(s[e] - li) + __expf(s[e] - l4[e]);
                    if (j == pos) w[e] -= 2.f;
                }
                w[e] *= c;
            }
            *cell = make_float4(w[0], w[1], w[2], w[3]);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < 32 && loss) {
        float l = 0.f;
        for (int r = threadIdx.x; r < n2; r += 32) l += rowloss[r];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
        if (threadIdx.x == 0) *loss = l / (float)n2;
    }
}

// (n2 not a multiple of 4: element-wise)
__global__ void __launch_bounds__(256) nce_weights_scalar_kernel(float* __restrict__ S, const float* __restrict__ lse, const float* __restrict__ rowloss,
                                                                  int n2, float inv_t, float gscale, float* __restrict__ loss) {
    const float c = gscale * inv_t / (float)n2;
    const int half = n2 >> 1;
    const int i = blockIdx.x;
    const int pos = i < half ? i + half : i - half;
    const float li = lse[i];
    for (int j = threadIdx.x; j < n2; j += 256) {
        const float s = S[(size_t)i * n2 + j] * inv_t;
        float w = 0.f;
        if (j != i) {
            w = __expf(s - li) + __expf(s - lse[j]);
            if (j == pos) w -= 2.f;
        }
        S[(size_t)i * n2 + j] = w * c;
    }
    if (blockIdx.x == 0 && threadIdx.x < 32 && loss) {
        float l = 0.f;
        for (int r = threadIdx.x; r < n2; r += 32) l += rowloss[r];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
        if (threadIdx.x == 0) *loss = l / (float)n2;
    }
}

// through F.normalize: dh_i = inv_i (dfn_i - fn_i (fn_i . dfn_i))
// dfn arrives as n_parts partial products (a split-K GEMM issued by the caller as one batched GEMM: W has 2B x 2B entries but the
// product only 2B x D, so a single GEMM leaves most SMs idle); the parts are added in index order here.
__global__ void __launch_bounds__(NCE_NT) nce_normalize_backward_kernel(const float* __restrict__ dfn, int n_parts, const float* __restrict__ fn,
                                                                         const float* __restrict__ inv_norm, int n2, int D, float* __restrict__ dh) {
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * NCE_RB + (threadIdx.x >> 5);
    if (row >= n2) return;
    const size_t part = (size_t)n2 * D;
    const float inv = inv_norm[row];
    if (D <= 128) {   // the parts' sum stays in registers
        float g[4];
        float dot = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int d = lane + 32 * q;
            g[q] = 0.f;
            if (d < D) {
                for (int p = 0; p < n_parts; ++p) g[q] += dfn[p * part + (size_t)row * D + d];
                dot = fmaf(fn[(size_t)row * D + d], g[q], dot);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int d = lane + 32 * q;
            if (d < D) dh[(size_t)row * D + d] = inv * (g[q] - fn[(size_t)row * D + d] * dot);
        }
        return;
    }
    auto gsum = [&](int d) { float g = 0.f; for (int p = 0; p < n_parts; ++p) g += dfn[p * part + (size_t)row * D + d]; return g; };
    float dot = 0.f;
    for (int d = lane; d < D; d += 32) dot = fmaf(fn[(size_t)row * D + d], gsum(d), dot);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
    for (int d = lane; d < D; d += 32) dh[(size_t)row * D + d] = inv * (gsum(d) - fn[(size_t)row * D + d] * dot);
}

// ---------------------------------------------------------------------------------------------------------------
// IIC loss, C <= 16: one CTA
// ---------------------------------------------------------------------------------------------------------------
constexpr int IS_NT = 512;
constexpr int IS_MAXC = 16;

__global__ void __launch_bounds__(IS_NT) iid_loss_small_kernel(const float* __restrict__ gz1, const float* __restrict__ gz2, int B, int C, float lamb,
                                                                float eps, float* __restrict__ loss, float* __restrict__ joint,
                                                                float* __restrict__ dz1, float* __restrict__ dz2, int staged, float gscale,
                                                                float loss_w, const float* __restrict__ add, float add_w) {
    extern __shared__ __align__(16) float zs[];             // staged: z1 | z2 (2 B C floats) — every later access hits shared memory
    __shared__ float part[IS_NT / 32][IS_MAXC * IS_MAXC];   // per-warp partial S
    __shared__ float S[IS_MAXC][IS_MAXC + 1];               // S, then Ssym
    __shared__ float dS[IS_MAXC][IS_MAXC + 1];
    __shared__ float marg[IS_MAXC], corr[IS_MAXC], gvec[IS_MAXC];
    __shared__ float red[4];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int np = C * C;
    const float* z1 = gz1;
    const float* z2 = gz2;
    if (staged) {   // coalesced, fully pipelined loads instead of a latency chain of dependent row reads
        const int n = B * C;
        for (int i = tid; i < n; i += IS_NT) { zs[i] = __ldg(gz1 + i); zs[n + i] = __ldg(gz2 + i); }
        __syncthreads();
        z1 = zs; z2 = zs + n;
    }
    // ---- S_ij = sum_b z1[b,i] z2[b,j] (LossFunctions.py:54-58): warp <-> rows b = w, w+16, ...; lane <-> pairs ----
    {
        float a[IS_MAXC * IS_MAXC / 32];
#pragma unroll
        for (int q = 0; q < IS_MAXC * IS_MAXC / 32; ++q) a[q] = 0.f;
#pragma unroll 4
        for (int b = w; b < B; b += IS_NT / 32) {
#pragma unroll
            for (int q = 0; q < IS_MAXC * IS_MAXC / 32; ++q) {
                const int pr = lane + 32 * q;
                if (pr < np) { const int i = pr / C, j = pr - i * C; a[q] = fmaf(z1[(size_t)b * C + i], z2[(size_t)b * C + j], a[q]); }
            }
        }
#pragma unroll
        for (int q = 0; q < IS_MAXC * IS_MAXC / 32; ++q) { const int pr = lane + 32 * q; if (pr < np) part[w][pr] = a[q]; }
    }
    __syncthreads();
    if (tid < np) {
        float s = 0.f;
#pragma unroll
        for (int g = 0; g < IS_NT / 32; ++g) s += part[g][tid];   // fixed order
        S[tid / C][tid % C] = s;
    }
    __syncthreads();
    // ---- symmetrise, normalise, marginals (:59-60, :28-34) — one warp, everything fits in a few registers ----
    if (w == 0) {
        float tot = 0.f;
        for (int pr = lane; pr < np; pr += 32) { const int i = pr / C, j = pr - i * C; tot += (S[i][j] + S[j][i]) * 0.5f; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
        if (lane == 0) red[0] = tot;
    }
    __syncthreads();
    const float T = red[0];
    float ssym = 0.f, P = 0.f;
    int pi = 0, pj = 0;
    if (tid < np) {
        pi = tid / C; pj = tid - pi * C;
        ssym = (S[pi][pj] + S[pj][pi]) * 0.5f;
        P = ssym / T;
    }
    __syncthreads();
    if (tid < np) S[pi][pj] = P;          // S now holds the normalised joint
    __syncthreads();
    if (tid < C) {
        float m = 0.f, c = 0.f;
        for (int j = 0; j < C; ++j) { const float v = S[tid][j]; m += v; if (v < eps) c += eps - v; }
        marg[tid] = m; corr[tid] = c;
    }
    __syncthreads();
    // ---- clamp, entropy terms (:36-44) and the pieces of the gradient ----
    float term = 0.f, Aij = 0.f;
    if (tid < np) {
        const bool cl = P < eps;
        const float Pc = cl ? eps : P;
        const float pic = marg[pi] < eps ? eps : marg[pi], pjc = marg[pj] < eps ? eps : marg[pj];
        const float inner = logf(Pc) - lamb * logf(pjc) - lamb * logf(pic);
        term = -Pc * inner;
        Aij = cl ? 0.f : (-inner - 1.f);
        if (joint) joint[pi * C + pj] = P;
    }
    if (tid < C) {
        const float m = marg[tid];
        gvec[tid] = m < eps ? 0.f : lamb * (m + corr[tid]) / m;
    }
    // block sums of term and A.P (np <= 256 values: warps 0..7), fixed order
    {
        float t = term, ap = Aij * P;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { t += __shfl_xor_sync(0xffffffffu, t, o); ap += __shfl_xor_sync(0xffffffffu, ap, o); }
        if (lane == 0) { part[w][0] = t; part[w][1] = ap; }
    }
    __syncthreads();
    if (tid == 0) {
        float l = 0.f, ap = 0.f;
        for (int g = 0; g < IS_NT / 32; ++g) { l += part[g][0]; ap += part[g][1]; }
        float gp = ap;
        for (int i = 0; i < C; ++i) gp += 2.f * gvec[i] * marg[i];
        if (loss) *loss = add ? loss_w * l + add_w * (*add) : loss_w * l;
        red[1] = gp;
    }
    __syncthreads();
    if (!dz1 && !dz2) return;
    if (tid < np) dS[pi][pj] = gscale * (Aij + gvec[pi] + gvec[pj] - red[1]) / T;   // dL/dSsym (symmetric), times the caller's weight
    __syncthreads();
    // ---- dz1[b,i] = sum_j z2[b,j] dS[i,j];  dz2[b,j] = sum_i z1[b,i] dS[i,j] ----
    for (int q = tid; q < B * C; q += IS_NT) {
        const int b = q / C, c = q - b * C;
        float a1 = 0.f, a2 = 0.f;
        for (int j = 0; j < C; ++j) {
            const float d = dS[c][j];
            a1 = fmaf(z2[(size_t)b * C + j], d, a1);
            a2 = fmaf(z1[(size_t)b * C + j], d, a2);
        }
        if (dz1) dz1[q] = a1;
        if (dz2) dz2[q] = a2;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// ReLU + Dropout of the encoder (idelucs/PytorchUtils.py:36-44: Linear - ReLU - Dropout(0.5)) in one pass each way, behind a
// GEMM whose output arrives as n_parts partial products (the inner-dimension split of train._FirstLinear) plus a bias:
//   forward   v = sum_p parts[p] + bias;  out = (v > 0 and kept) ? v / (1 - p) : 0
//   backward  dx = out > 0 ? dy / (1 - p) : 0      (out > 0 exactly where the unit was active AND kept: no mask is stored)
// The keep decision of element e in training step t is one Philox4x32-10 word: counter (e / 4, t lo, t hi, layer tag), key = seed,
// word e % 4 — stateless, so a CUDA graph replays it with the step counter read from device memory.  Replaces the framework's
// reduce + add + clamp + fused_dropout launches (13 us behind the first layer) and masked_scale + threshold_backward.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) relu_dropout_fwd_kernel(const float* __restrict__ parts, int n_parts, const float* __restrict__ bias, long long n4,
                                                               int N4, uint32_t thresh, float inv_keep, unsigned long long seed,
                                                               const long long* __restrict__ step, uint32_t tag, float* __restrict__ out) {
    const long long t = step ? *step : 0;
    const size_t part4 = (size_t)n4;
    for (long long q = (long long)blockIdx.x * 256 + threadIdx.x; q < n4; q += (long long)gridDim.x * 256) {
        float4 v = reinterpret_cast<const float4*>(parts)[q];
        for (int p = 1; p < n_parts; ++p) {
            const float4 w = reinterpret_cast<const float4*>(parts)[p * part4 + q];
            v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
        }
        if (bias) {
            const float4 b = __ldg(reinterpret_cast<const float4*>(bias) + (int)(q % N4));
            v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
        }
        const U4 r = philox4x32_10((uint32_t)q, (uint32_t)t, (uint32_t)((unsigned long long)t >> 32), tag ^ (uint32_t)((unsigned long long)q >> 32),
                                   (uint32_t)seed, (uint32_t)(seed >> 32));
        float4 o;
        o.x = (v.x > 0.f && r.x >= thresh) ? v.x * inv_keep : 0.f;   // dropped with probability thresh / 2^32 = p
        o.y = (v.y > 0.f && r.y >= thresh) ? v.y * inv_keep : 0.f;
        o.z = (v.z > 0.f && r.z >= thresh) ? v.z * inv_keep : 0.f;
        o.w = (v.w > 0.f && r.w >= thresh) ? v.w * inv_keep : 0.f;
        reinterpret_cast<float4*>(out)[q] = o;
    }
}

// out = sum_p parts[p] + bias: the tail of a Linear whose GEMM was split over its inner dimension (no activation)
__global__ void __launch_bounds__(256) sum_parts_bias_kernel(const float* __restrict__ parts, int n_parts, const float* __restrict__ bias, long long n4, int N4,
                                                             float* __restrict__ out) {
    const size_t part4 = (size_t)n4;
    for (long long q = (long long)blockIdx.x * 256 + threadIdx.x; q < n4; q += (long long)gridDim.x * 256) {
        float4 v = reinterpret_cast<const float4*>(parts)[q];
        for (int p = 1; p < n_parts; ++p) {
            const float4 w = reinterpret_cast<const float4*>(parts)[p * part4 + q];
            v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
        }
        if (bias) {
            const float4 b = __ldg(reinterpret_cast<const float4*>(bias) + (int)(q % N4));
            v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
        }
        reinterpret_cast<float4*>(out)[q] = v;
    }
}

__global__ void __launch_bounds__(256) relu_dropout_bwd_kernel(const float* __restrict__ out, const float* __restrict__ dy, long long n4, float inv_keep,
                                                               float* __restrict__ dx) {
    for (long long q = (long long)blockIdx.x * 256 + threadIdx.x; q < n4; q += (long long)gridDim.x * 256) {
        const float4 o = reinterpret_cast<const float4*>(out)[q];
        const float4 g = reinterpret_cast<const float4*>(dy)[q];
        reinterpret_cast<float4*>(dx)[q] = make_float4(o.x > 0.f ? g.x * inv_keep : 0.f, o.y > 0.f ? g.y * inv_keep : 0.f,
                                                       o.z > 0.f ? g.z * inv_keep : 0.f, o.w > 0.f ? g.w * inv_keep : 0.f);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Pair ids -> what the mimic kernel's selection mode wants (idelucs/utils.py:370-389: row r of x_train is sequence r mod N with
// mimic r div N + 1 on the 'modified' side and slot 0 on the 'true' side): item = sequence index, sel = (0, mimic).  One launch
// instead of ten framework kernels of index arithmetic at the head of every training step.
// ---------------------------------------------------------------------------------------------------------------
__global__ void pair_selection_kernel(const long long* __restrict__ pair_ids, int n, long long n_seqs, int* __restrict__ sidx, int* __restrict__ sel) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long id = pair_ids[i];
    const long long m = id / n_seqs;
    sidx[i] = (int)(id - m * n_seqs);
    sel[2 * i] = 0;
    sel[2 * i + 1] = (int)m + 1;
}

// ---------------------------------------------------------------------------------------------------------------
// RMSprop (torch.optim.RMSprop, momentum = 0, centered = False): g = grad * gscale + wd * p; v = alpha v + (1 - alpha) g^2;
// p -= lr * g / (sqrt(v) + eps)
// ---------------------------------------------------------------------------------------------------------------
__global__ void rmsprop_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ v, long long n, float lr, float alpha,
                               float eps, float wd, float gscale) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float pp = p[i];
        const float gg = fmaf(wd, pp, g[i] * gscale);
        const float vv = fmaf(1.0f - alpha, gg * gg, alpha * v[i]);
        v[i] = vv;
        p[i] = pp - lr * (gg / (sqrtf(vv) + eps));
    }
}

// ---------------------------------------------------------------------------------------------------------------
// The other two optimisers of idelucs/models.py:86-99 as per-element updates, shared by the single-rank kernel below and the
// all-reduce kernel: update(g, p, s) takes the (scaled) gradient, the parameter and the optimiser state s[kStates] of one element
// and returns the new parameter.  load() runs once per thread before the first element: the step number t (1-based) is read
// from device memory, so a replayed CUDA graph keeps counting without a host argument.
//   SGD  (torch.optim.SGD(lr, momentum, weight_decay), dampening 0, no Nesterov): d = g + wd p; buf = d at t = 1, else
//        momentum buf + d; p -= lr buf
//   Adam (torch.optim.Adam(lr, betas, eps, weight_decay), no amsgrad): g += wd p; m = m + (1 - b1)(g - m);
//        v = b2 v + (1 - b2) g^2; p -= (lr / (1 - b1^t)) m / (sqrt(v) / sqrt(1 - b2^t) + eps)
// ---------------------------------------------------------------------------------------------------------------
struct RmspropUpdate {
    static constexpr int kStates = 1;
    float lr, alpha, eps, wd;
    __device__ __forceinline__ void load() {}
    __device__ __forceinline__ float update(float g, float p, float (&s)[1]) const {
        const float gg = fmaf(wd, p, g);
        const float vv = fmaf(1.0f - alpha, gg * gg, alpha * s[0]);
        s[0] = vv;
        return p - lr * (gg / (sqrtf(vv) + eps));
    }
};

struct SgdUpdate {
    static constexpr int kStates = 1;
    float lr, momentum, wd;
    const long long* step;
    bool first;
    __device__ __forceinline__ void load() { first = *step <= 1; }
    __device__ __forceinline__ float update(float g, float p, float (&s)[1]) const {
        const float d = fmaf(wd, p, g);
        const float b = first ? d : __fadd_rn(__fmul_rn(momentum, s[0]), d);   // (torch's mul_ then add_: two roundings)
        s[0] = b;
        return p - lr * b;
    }
};

struct AdamUpdate {   // (the betas in double, as torch holds them: 1 - 0.999f is 1.3e-5 away from 1 - 0.999)
    static constexpr int kStates = 2;
    float lr, eps, wd;
    double beta1, beta2;
    const long long* step;
    float c1, b2, c2, step_size, bc2_sqrt;
    __device__ __forceinline__ void load() {   // the bias corrections in double, as torch computes them on the host
        const double t = (double)*step;
        c1 = (float)(1.0 - beta1);
        b2 = (float)beta2;
        c2 = (float)(1.0 - beta2);
        step_size = (float)((double)lr / (1.0 - pow(beta1, t)));
        bc2_sqrt = (float)sqrt(1.0 - pow(beta2, t));
    }
    __device__ __forceinline__ float update(float g, float p, float (&s)[2]) const {
        const float gg = fmaf(wd, p, g);
        const float m = s[0] + c1 * (gg - s[0]);
        const float v = fmaf(c2 * gg, gg, __fmul_rn(s[1], b2));   // (torch's mul_(beta2) then addcmul_)
        s[0] = m; s[1] = v;
        return p - step_size * (m / (sqrtf(v) / bc2_sqrt + eps));
    }
};

constexpr int MAX_STATES = 2;
struct StatePtrs { float* s[MAX_STATES]; };

// single rank: one elementwise pass over a flat buffer (any alignment)
template <class Op>
__global__ void opt_step_kernel(float* __restrict__ p, const float* __restrict__ g, StatePtrs st, long long n, float gscale, Op op) {
    op.load();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float s[Op::kStates];
#pragma unroll
        for (int k = 0; k < Op::kStates; ++k) s[k] = st.s[k][i];
        p[i] = op.update(g[i] * gscale, p[i], s);
#pragma unroll
        for (int k = 0; k < Op::kStates; ++k) st.s[k][i] = s[k];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Data-parallel optimiser step as ONE kernel over NVLink peer memory: gradient all-reduce (mean) + the update of Op + parameter
// broadcast.  Gradients and parameters live in symmetric buffers (the same allocation mapped by every rank).  Rank r owns the
// slice [r * shard, (r + 1) * shard): it reads the SUM of every rank's gradient slice — one multimem.ld_reduce per 16 bytes when
// the buffers have an NVLS multicast mapping (the NVSwitch adds the eight operands), else one load per peer in rank order —
// applies the update to its slice of the parameters and stores the new values into EVERY rank's parameter buffer
// (multimem.st, or one store per peer).  Per GPU that is 1/N of the gradient bytes in and 1/N of the parameter bytes out,
// no staging buffers, no separate optimiser pass, and every replica receives bit-identical parameters (one writer per slice).
// The caller brackets the launch with cross-rank barriers (gradients complete before, parameters visible after).
// ---------------------------------------------------------------------------------------------------------------
constexpr int MAX_PEERS = 16;
struct PeerPtrs { float* p[MAX_PEERS]; };

__device__ __forceinline__ float4 multimem_ld_reduce_add(const float* mc_addr) {
    float4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(mc_addr) : "memory");
    return v;
}
__device__ __forceinline__ void multimem_st(float* mc_addr, float4 v) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// Every thread requests AR_U 16-byte units of the reduced gradient (and of its local state) before it touches the first result:
// the kernel is bound by the NVLink round trip (a few microseconds per dependent access), not by bandwidth — 8.5 MB of gradients
// are 1 MB per rank at 8 GPUs — so the loads of a thread must overlap each other.
constexpr int AR_U = 4;

template <class Op>
__global__ void __launch_bounds__(256) allreduce_step_kernel(const PeerPtrs grads, const PeerPtrs params, const float* grad_mc, float* param_mc,
                                                               const StatePtrs st, long long shard, int rank, int world, Op op) {
    op.load();
    const long long base = (long long)rank * shard;
    const float inv_world = 1.0f / (float)world;
    const long long units = shard / 4, stride = (long long)gridDim.x * blockDim.x;
    for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < units; i0 += stride * AR_U) {
        float4 g[AR_U], p[AR_U], v[Op::kStates][AR_U];
#pragma unroll
        for (int u = 0; u < AR_U; ++u) {
            const long long i4 = i0 + u * stride;
            if (i4 < units) {
                const long long idx = base + i4 * 4;
                if (grad_mc) {
                    g[u] = multimem_ld_reduce_add(grad_mc + idx);
                } else {
                    g[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    for (int r = 0; r < world; ++r) {   // rank order: the same sum on every run
                        const float4 t = *reinterpret_cast<const float4*>(grads.p[r] + idx);
                        g[u].x += t.x; g[u].y += t.y; g[u].z += t.z; g[u].w += t.w;
                    }
                }
                p[u] = *reinterpret_cast<const float4*>(params.p[rank] + idx);
#pragma unroll
                for (int k = 0; k < Op::kStates; ++k) v[k][u] = reinterpret_cast<const float4*>(st.s[k])[i4];
            }
        }
#pragma unroll
        for (int u = 0; u < AR_U; ++u) {
            const long long i4 = i0 + u * stride;
            if (i4 < units) {
                const long long idx = base + i4 * 4;
                float* gp = &g[u].x; float* pp = &p[u].x;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    float s[Op::kStates];
#pragma unroll
                    for (int k = 0; k < Op::kStates; ++k) s[k] = (&v[k][u].x)[e];
                    pp[e] = op.update(gp[e] * inv_world, pp[e], s);
#pragma unroll
                    for (int k = 0; k < Op::kStates; ++k) (&v[k][u].x)[e] = s[k];
                }
#pragma unroll
                for (int k = 0; k < Op::kStates; ++k) reinterpret_cast<float4*>(st.s[k])[i4] = v[k][u];
                if (param_mc) {
                    multimem_st(param_mc + idx, p[u]);
                } else {
                    for (int r = 0; r < world; ++r) *reinterpret_cast<float4*>(params.p[r] + idx) = p[u];
                }
            }
        }
    }
    __threadfence_system();
}

// ---------------------------------------------------------------------------------------------------------------
// IIC loss, C <= 8 (the headline configurations: n_clusters = 3 .. 8): ONE CTA, thread <-> batch row, two CTA barriers.
// A row's 2 C probabilities stay in registers from the joint to the gradient (B <= 512: one row per thread; more rows are
// re-read through L1); the C x C outer products are summed over the warp with a transpose-reduce (31 shuffles per 32 pairs, every
// lane ends with one pair's total) and over the warps by warp 0, which then does the whole C x C algebra (LossFunctions.py:28-44
// and its derivative) with warp shuffles alone.  Fixed-order sums (run-to-run identical).  gscale multiplies the gradients,
// and the loss written is loss_w * loss + add_w * (*add) — the caller's weighting of idelucs/models.py:128 without extra launches.
// ---------------------------------------------------------------------------------------------------------------
constexpr int IR_NT = 512;

template <int NV>
__device__ __forceinline__ float transpose_reduce(float (&v)[NV], int lane) {   // NV = 32: lane l returns sum over the warp of v[l]
    static_assert(NV == 32, "one pair slot per lane");
#pragma unroll
    for (int off = 16, n = 32; off >= 1; off >>= 1, n >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int k = 0; k < n / 2; ++k) {
            const float send = up ? v[k] : v[k + n / 2];
            const float keep = up ? v[k + n / 2] : v[k];
            v[k] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    return v[0];
}

__device__ __forceinline__ float warp_total(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int C>
__global__ void __launch_bounds__(IR_NT) iid_loss_reg_kernel(const float* __restrict__ gz1, const float* __restrict__ gz2, int B, float lamb, float eps,
                                                              float* __restrict__ loss, float* __restrict__ joint, float* __restrict__ dz1,
                                                              float* __restrict__ dz2, float gscale, float loss_w, const float* __restrict__ add,
                                                              float add_w) {
    constexpr int NP = C * C, NG = (NP + 31) / 32;        // pairs, groups of 32 pair slots
    __shared__ float part[IR_NT / 32][NG * 32];
    __shared__ float Sm[C][C + 1], dS[C][C + 1], marg[C], gvec[C];
    __shared__ float sT;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    float z1[C], z2[C];
    // ---- S_ij = sum_b z1[b,i] z2[b,j] (LossFunctions.py:54-58) ----
    {
        float acc[NG][32];
#pragma unroll
        for (int g = 0; g < NG; ++g)
#pragma unroll
            for (int q = 0; q < 32; ++q) acc[g][q] = 0.f;
        for (int b = tid; b < B; b += IR_NT) {
#pragma unroll
            for (int c = 0; c < C; ++c) { z1[c] = __ldg(gz1 + (size_t)b * C + c); z2[c] = __ldg(gz2 + (size_t)b * C + c); }
#pragma unroll
            for (int i = 0; i < C; ++i)
#pragma unroll
                for (int j = 0; j < C; ++j) acc[(i * C + j) / 32][(i * C + j) % 32] = fmaf(z1[i], z2[j], acc[(i * C + j) / 32][(i * C + j) % 32]);
        }
#pragma unroll
        for (int g = 0; g < NG; ++g) part[w][g * 32 + lane] = transpose_reduce<32>(acc[g], lane);
    }
    __syncthreads();
    if (w == 0) {
        int pi[NG], pj[NG];
        bool ok[NG];
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            const int pr = g * 32 + lane;
            ok[g] = pr < NP;
            pi[g] = ok[g] ? pr / C : 0; pj[g] = ok[g] ? pr % C : 0;
            float sacc = 0.f;
#pragma unroll
            for (int q = 0; q < IR_NT / 32; ++q) sacc += part[q][pr];   // fixed order
            if (ok[g]) Sm[pi[g]][pj[g]] = sacc;
        }
        __syncwarp();
        // symmetrise, normalise (:59-60)
        float ssym[NG], P[NG], tsum = 0.f;
#pragma unroll
        for (int g = 0; g < NG; ++g) { ssym[g] = ok[g] ? (Sm[pi[g]][pj[g]] + Sm[pj[g]][pi[g]]) * 0.5f : 0.f; tsum += ssym[g]; }
        const float T = warp_total(tsum);
        __syncwarp();
#pragma unroll
        for (int g = 0; g < NG; ++g) { P[g] = ssym[g] / T; if (ok[g]) { Sm[pi[g]][pj[g]] = P[g]; if (joint) joint[pi[g] * C + pj[g]] = P[g]; } }
        __syncwarp();
        // marginals before clamping, the clamp's correction (:28-38)
        if (lane < C) {
            float m = 0.f, c = 0.f;
#pragma unroll
            for (int j = 0; j < C; ++j) { const float v = Sm[lane][j]; m += v; if (v < eps) c += eps - v; }
            marg[lane] = m;
            gvec[lane] = m < eps ? 0.f : lamb * (m + c) / m;
        }
        __syncwarp();
        float term = 0.f, ap = 0.f, A[NG];
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            A[g] = 0.f;
            if (ok[g]) {
                const bool cl = P[g] < eps;
                const float Pc = cl ? eps : P[g];
                const float mi = marg[pi[g]], mj = marg[pj[g]];
                const float pic = mi < eps ? eps : mi, pjc = mj < eps ? eps : mj;
                const float inner = logf(Pc) - lamb * logf(pjc) - lamb * logf(pic);
                term += -Pc * inner;
                A[g] = cl ? 0.f : (-inner - 1.f);
                ap += A[g] * P[g];
            }
        }
        const float l = warp_total(term);
        float gp = warp_total(ap);
#pragma unroll
        for (int i = 0; i < C; ++i) gp += 2.f * gvec[i] * marg[i];
        if (lane == 0) {
            if (loss) *loss = add ? loss_w * l + add_w * (*add) : loss_w * l;
            sT = T;
        }
#pragma unroll
        for (int g = 0; g < NG; ++g)
            if (ok[g]) dS[pi[g]][pj[g]] = gscale * (A[g] + gvec[pi[g]] + gvec[pj[g]] - gp) / T;   // dL/dSsym (symmetric)
    }
    if (!dz1 && !dz2) return;
    __syncthreads();
    // ---- dz1[b,i] = sum_j z2[b,j] dS[i,j];  dz2[b,i] = sum_j z1[b,j] dS[i,j] ----
    float d[C][C];
#pragma unroll
    for (int i = 0; i < C; ++i)
#pragma unroll
        for (int j = 0; j < C; ++j) d[i][j] = dS[i][j];
    for (int b = tid; b < B; b += IR_NT) {
        if (B > IR_NT) {   // (with at most one row per thread it is still in registers)
#pragma unroll
            for (int c = 0; c < C; ++c) { z1[c] = __ldg(gz1 + (size_t)b * C + c); z2[c] = __ldg(gz2 + (size_t)b * C + c); }
        }
#pragma unroll
        for (int i = 0; i < C; ++i) {
            float a1 = 0.f, a2 = 0.f;
#pragma unroll
            for (int j = 0; j < C; ++j) { a1 = fmaf(z2[j], d[i][j], a1); a2 = fmaf(z1[j], d[i][j], a2); }
            if (dz1) dz1[(size_t)b * C + i] = a1;
            if (dz2) dz2[(size_t)b * C + i] = a2;
        }
    }
}

template <int C>
static void iid_reg_launch(const float* z1, const float* z2, int B, float lamb, float eps, float* loss, float* joint, float* dz1, float* dz2,
                           float gscale, float loss_w, const float* add, float add_w, cudaStream_t st) {
    iid_loss_reg_kernel<C><<<1, IR_NT, 0, st>>>(z1, z2, B, lamb, eps, loss, joint, dz1, dz2, gscale, loss_w, add, add_w);
}

// ---------------------------------------------------------------------------------------------------------------
// IIC loss from a given S2 = S + S^T, S = z1^T z2 (any C): the C x C algebra of LossFunctions.py:28-44, :59-60 and its derivative.
// For large C (C = 200 of the embedding path) the contractions around it (S = z1^T z2, dz1 = z2 dS, dz2 = z1 dS) are small dense
// GEMMs and stay library calls issued by the caller, like InfoNCE's (idl_iid_loss issues them as the two kernels below).  Four
// dependent launches, warp <-> row of the (symmetrised: coalesced row reads only) joint, the few global scalars (T, loss, <A, P>)
// re-derived by every warp from per-row partials in a fixed order — a single CTA doing the same work takes 65 us (instruction-bound
// on one SM).
// scratch: 6 C floats = rowsum | marg | gvec | lgm | rowterm | rowap
// ---------------------------------------------------------------------------------------------------------------
constexpr int IA_NT = 256, IA_RPB = IA_NT / 32;

__device__ __forceinline__ float ordered_total(const float* __restrict__ x, int n, int lane) {   // the same value in every warp that calls it
    float t = 0.f;
    for (int i = lane; i < n; i += 32) t += x[i];
    return warp_total(t);
}

__global__ void __launch_bounds__(IA_NT) iid_alg_rowsum_kernel(const float* __restrict__ S2, int C, float* __restrict__ scratch) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * IA_RPB + (threadIdx.x >> 5);
    if (i >= C) return;
    float t = 0.f;
    for (int j = lane; j < C; j += 32) t += 0.5f * S2[(size_t)i * C + j];   // (S + S^T) / 2 (:59)
    t = warp_total(t);
    if (lane == 0) scratch[i] = t;
}

__global__ void __launch_bounds__(IA_NT) iid_alg_marginal_kernel(const float* __restrict__ S2, int C, float lamb, float eps, float* __restrict__ scratch,
                                                                 float* __restrict__ joint) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * IA_RPB + (threadIdx.x >> 5);
    if (i >= C) return;
    const float T = ordered_total(scratch, C, lane);
    float m = 0.f, c = 0.f;
    for (int j = lane; j < C; j += 32) {   // normalise (:60); marginal before clamping and the clamp's correction (:28-38)
        const float P = 0.5f * S2[(size_t)i * C + j] / T;
        m += P;
        if (P < eps) c += eps - P;
        if (joint) joint[(size_t)i * C + j] = P;
    }
    m = warp_total(m); c = warp_total(c);
    if (lane == 0) {
        scratch[C + i] = m;
        scratch[2 * C + i] = m < eps ? 0.f : lamb * (m + c) / m;
        scratch[3 * C + i] = lamb * logf(m < eps ? eps : m);
    }
}

__global__ void __launch_bounds__(IA_NT) iid_alg_terms_kernel(const float* __restrict__ S2, int C, float eps, float* __restrict__ scratch) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * IA_RPB + (threadIdx.x >> 5);
    if (i >= C) return;
    const float T = ordered_total(scratch, C, lane);
    const float* lgm = scratch + 3 * C;
    const float li = lgm[i];
    float term = 0.f, ap = 0.f;
    for (int j = lane; j < C; j += 32) {   // entropy terms (:40-44) and <A, P>, A = d term / d P (0 where clamped)
        const float P = 0.5f * S2[(size_t)i * C + j] / T;
        const bool cl = P < eps;
        const float Pc = cl ? eps : P;
        const float inner = logf(Pc) - lgm[j] - li;
        term += -Pc * inner;
        if (!cl) ap += (-inner - 1.f) * P;
    }
    term = warp_total(term); ap = warp_total(ap);
    if (lane == 0) { scratch[4 * C + i] = term; scratch[5 * C + i] = ap; }
}

__global__ void __launch_bounds__(IA_NT) iid_alg_grad_kernel(const float* __restrict__ S2, int C, float eps, float gscale, float loss_w,
                                                             const float* __restrict__ add, float add_w, const float* __restrict__ scratch,
                                                             float* __restrict__ loss, float* __restrict__ dS) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, i = blockIdx.x * IA_RPB + w;
    if (blockIdx.x == 0 && w == 0 && loss) {
        const float l = ordered_total(scratch + 4 * C, C, lane);
        if (lane == 0) *loss = add ? loss_w * l + add_w * (*add) : loss_w * l;
    }
    if (i >= C || !dS) return;
    const float T = ordered_total(scratch, C, lane);
    const float* marg = scratch + C;
    const float* gvec = scratch + 2 * C;
    const float* lgm = scratch + 3 * C;
    float gm = 0.f;
    for (int q = lane; q < C; q += 32) gm += 2.f * gvec[q] * marg[q];
    const float gp = ordered_total(scratch + 5 * C, C, lane) + warp_total(gm);
    const float li = lgm[i], gi = gvec[i], sc = gscale / T;
    for (int j = lane; j < C; j += 32) {
        const float P = 0.5f * S2[(size_t)i * C + j] / T;
        const bool cl = P < eps;
        const float inner = logf(cl ? eps : P) - lgm[j] - li;
        const float A = cl ? 0.f : (-inner - 1.f);
        dS[(size_t)i * C + j] = sc * (A + gi + gvec[j] - gp);   // dL/dS_sym (symmetric), times the caller's weight
    }
}

// ---------------------------------------------------------------------------------------------------------------
// IIC loss, 16 < C <= 256, through the C ABI: the contractions around the algebra kernels above as two tiled kernels of our own,
// S2 = S + S^T with S = z1^T z2 before them and dz1 = z2 dS, dz2 = z1 dS after them.  Every thread sums its entries in a fixed
// order (no float atomics), so the results are run-to-run identical.
// ---------------------------------------------------------------------------------------------------------------
constexpr int IC_T = 16;             // tile edge
constexpr int IC_NT = IC_T * IC_T;   // threads per CTA
constexpr int IC_BR = 64;            // batch rows staged per step
constexpr int IID_MAXC = 256;        // idl_iid_loss_max_clusters()

// CTA <-> tile pair (I, J), I <= J, enumerated row by row; thread (ti, tj) sums S_ij and S_ji for i = 16 I + ti, j = 16 J + tj and
// stores S_ij + S_ji to both (i, j) and (j, i), so S2 is exactly symmetric (a diagonal tile stores from its upper triangle only)
__global__ void __launch_bounds__(IC_NT) iid_s2_kernel(const float* __restrict__ z1, const float* __restrict__ z2, int B, int C, int nt,
                                                       float* __restrict__ S2) {
    __shared__ float sA[4][IC_BR][IC_T];   // z1[:, I] z2[:, J] z1[:, J] z2[:, I]
    const int tid = threadIdx.x, ti = tid / IC_T, tj = tid % IC_T;
    int I = 0, rem = blockIdx.x;
    while (rem >= nt - I) { rem -= nt - I; ++I; }
    const int J = I + rem;
    const int I0 = I * IC_T, J0 = J * IC_T;
    float a0 = 0.f, a1 = 0.f, b0 = 0.f, b1 = 0.f;
    for (int r0 = 0; r0 < B; r0 += IC_BR) {
        __syncthreads();
#pragma unroll
        for (int q = 0; q < IC_BR * IC_T / IC_NT; ++q) {
            const int idx = tid + q * IC_NT, row = idx / IC_T, col = idx % IC_T;
            const int b = r0 + row;
            const bool ci = b < B && I0 + col < C, cj = b < B && J0 + col < C;
            sA[0][row][col] = ci ? z1[(size_t)b * C + I0 + col] : 0.f;
            sA[3][row][col] = ci ? z2[(size_t)b * C + I0 + col] : 0.f;
            sA[1][row][col] = cj ? z2[(size_t)b * C + J0 + col] : 0.f;
            sA[2][row][col] = cj ? z1[(size_t)b * C + J0 + col] : 0.f;
        }
        __syncthreads();
#pragma unroll 8
        for (int r = 0; r < IC_BR; r += 2) {
            a0 = fmaf(sA[0][r][ti], sA[1][r][tj], a0);
            b0 = fmaf(sA[2][r][tj], sA[3][r][ti], b0);
            a1 = fmaf(sA[0][r + 1][ti], sA[1][r + 1][tj], a1);
            b1 = fmaf(sA[2][r + 1][tj], sA[3][r + 1][ti], b1);
        }
    }
    const int i = I0 + ti, j = J0 + tj;
    if (i < C && j < C && (I != J || ti <= tj)) {
        const float s = (a0 + a1) + (b0 + b1);
        S2[(size_t)i * C + j] = s;
        S2[(size_t)j * C + i] = s;
    }
}

// CTA <-> 64 rows x 16 columns of dz1 = z2 dS (blockIdx.z = 0) or dz2 = z1 dS (blockIdx.z = 1; a NULL output is skipped); thread
// (ti, tj) sums rows ti, ti + 16, ... of column tj over j in increasing order
__global__ void __launch_bounds__(IC_NT) iid_dz_kernel(const float* __restrict__ z1, const float* __restrict__ z2, const float* __restrict__ dS, int B,
                                                       int C, float* __restrict__ dz1, float* __restrict__ dz2) {
    float* out = blockIdx.z == 0 ? dz1 : dz2;
    if (!out) return;
    const float* zo = blockIdx.z == 0 ? z2 : z1;
    __shared__ float sZ[IC_BR][IC_T];   // zo[r0 .., j0 ..]
    __shared__ float sD[IC_T][IC_T];    // dS[j0 .., c0 ..]
    const int tid = threadIdx.x, ti = tid / IC_T, tj = tid % IC_T;
    const int r0 = blockIdx.x * IC_BR, c0 = blockIdx.y * IC_T;
    float acc[IC_BR / IC_T] = {};
    for (int j0 = 0; j0 < C; j0 += IC_T) {
        __syncthreads();
#pragma unroll
        for (int q = 0; q < IC_BR * IC_T / IC_NT; ++q) {
            const int idx = tid + q * IC_NT, row = idx / IC_T, col = idx % IC_T;
            sZ[row][col] = (r0 + row < B && j0 + col < C) ? zo[(size_t)(r0 + row) * C + j0 + col] : 0.f;
        }
        sD[ti][tj] = (j0 + ti < C && c0 + tj < C) ? dS[(size_t)(j0 + ti) * C + c0 + tj] : 0.f;
        __syncthreads();
#pragma unroll
        for (int jj = 0; jj < IC_T; ++jj) {
            const float d = sD[jj][tj];
#pragma unroll
            for (int q = 0; q < IC_BR / IC_T; ++q) acc[q] = fmaf(sZ[ti + q * IC_T][jj], d, acc[q]);
        }
    }
#pragma unroll
    for (int q = 0; q < IC_BR / IC_T; ++q) {
        const int b = r0 + ti + q * IC_T;
        if (b < B && c0 + tj < C) out[(size_t)b * C + c0 + tj] = acc[q];
    }
}

// C <= 16 (idl_iid_loss_scaled)
static int iid_loss_small_launch(const float* d_z1, const float* d_z2, int B, int C, float lamb, float eps, float* d_loss, float* d_joint, float* d_dz1,
                          float* d_dz2, void* stream, float gscale, float loss_w, const float* d_add, float add_w) {
    cudaStream_t st = (cudaStream_t)stream;
    if (C <= 8) {
        switch (C) {
            case 1: iid_reg_launch<1>(d_z1, d_z2, B, lamb, eps, d_loss, d_joint, d_dz1, d_dz2, gscale, loss_w, d_add, add_w, st); break;
            case 2: iid_reg_launch<2>(d_z1, d_z2, B, lamb, eps, d_loss, d_joint, d_dz1, d_dz2, gscale, loss_w, d_add, add_w, st); break;
            case 3: iid_reg_launch<3>(d_z1, d_z2, B, lamb, eps, d_loss, d_joint, d_dz1, d_dz2, gscale, loss_w, d_add, add_w, st); break;
            case 4: iid_reg_launch<4>(d_z1, d_z2, B, lamb, eps, d_loss, d_joint, d_dz1, d_dz2, gscale, loss_w, d_add, add_w, st); break;
            case 5: iid_reg_launch<5>(d_z1, d_z2, B, lamb, eps, d_loss, d_joint, d_dz1, d_dz2, gscale, loss_w, d_add, add_w, st); break;
            case 6: iid_reg_launch<6>(d_z1, d_z2, B, lamb, eps, d_loss, d_joint, d_dz1, d_dz2, gscale, loss_w, d_add, add_w, st); break;
            case 7: iid_reg_launch<7>(d_z1, d_z2, B, lamb, eps, d_loss, d_joint, d_dz1, d_dz2, gscale, loss_w, d_add, add_w, st); break;
            default: iid_reg_launch<8>(d_z1, d_z2, B, lamb, eps, d_loss, d_joint, d_dz1, d_dz2, gscale, loss_w, d_add, add_w, st); break;
        }
        note_launch();
        IDL_CUDA_CHECK(cudaGetLastError());
        return IDL_OK;
    }
    // both inputs staged in shared memory when they fit (up to 160 KB)
    size_t smem = sizeof(float) * 2 * (size_t)B * C;
    int staged = 1;
    if (smem > 160 * 1024) { smem = 0; staged = 0; }
    if (smem > 24 * 1024) {   // (18.5 KB of static shared memory ride along: opt in before the sum passes 48 KB)
        static bool configured[64] = {false};
        int dev = 0;
        IDL_CUDA_CHECK(cudaGetDevice(&dev));
        if (dev < 0 || dev >= 64 || !configured[dev]) {
            IDL_CUDA_CHECK(cudaFuncSetAttribute(iid_loss_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
            if (dev >= 0 && dev < 64) configured[dev] = true;
        }
    }
    iid_loss_small_kernel<<<1, IS_NT, smem, st>>>(d_z1, d_z2, B, C, lamb, eps, d_loss, d_joint, d_dz1, d_dz2, staged, gscale, loss_w, d_add, add_w); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Global-batch losses of the data-parallel step: W ranks of b pairs each train on the loss of the B = W b pairs together.  The
// global stacked batch is [true rows of rank 0 .. W-1 ; modified rows of rank 0 .. W-1]: rank r's local row q is global row
// r b + q (q < b) or B + r b + (q - b).  What one rank needs of the others is read through peer addresses (symmetric memory, or
// the slots of an all-gathered tensor), always summed in rank order, so every rank computes the same bits without float atomics.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int global_row(int q, int b, int rank, int B) { return q < b ? rank * b + q : B + rank * b + (q - b); }

// s + element i of every rank's buffer, added in rank order.  The table is indexed with compile-time ranks only, so the kernel
// parameter is not copied to local memory.
__device__ __forceinline__ float rank_order_sum(const PeerPtrs& t, int world, size_t i, float s) {
#pragma unroll
    for (int r = 0; r < MAX_PEERS; ++r)
        if (r < world) s += t.p[r][i];
    return s;
}

// IIC, C <= 16: S2 = sum over the ranks' partials S2_r (rank order), the C x C algebra of iid_loss_small_kernel on it, and this
// rank's gradients dz1 = z2 dS, dz2 = z1 dS — ONE CTA, thread <-> joint entry
constexpr int IG_NT = 512;
__global__ void __launch_bounds__(IG_NT) iid_global_small_kernel(const PeerPtrs s2, int world, const float* __restrict__ z1, const float* __restrict__ z2,
                                                                 int B, int C, float lamb, float eps, float gscale, float loss_w,
                                                                 const float* __restrict__ add, float add_w, float* __restrict__ loss,
                                                                 float* __restrict__ dz1, float* __restrict__ dz2) {
    __shared__ float Pm[IS_MAXC][IS_MAXC + 1], dS[IS_MAXC][IS_MAXC + 1];
    __shared__ float marg[IS_MAXC], gvec[IS_MAXC];
    __shared__ float red[IG_NT / 32][2];
    __shared__ float sT, sgp;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int np = C * C;
    const int pi = tid < np ? tid / C : 0, pj = tid < np ? tid - pi * C : 0;
    float ssym = 0.f;
    if (tid < np) {
        ssym = 0.5f * rank_order_sum(s2, world, tid, 0.f);   // (S + S^T) / 2 (LossFunctions.py:59)
    }
    const float t = warp_total(ssym);
    if (lane == 0) red[w][0] = t;
    __syncthreads();
    if (tid == 0) { float T = 0.f; for (int g = 0; g < IG_NT / 32; ++g) T += red[g][0]; sT = T; }
    __syncthreads();
    const float T = sT;
    const float P = ssym / T;   // normalise (:60)
    if (tid < np) Pm[pi][pj] = P;
    __syncthreads();
    if (tid < C) {   // marginals before clamping, the clamp's correction (:28-38)
        float m = 0.f, c = 0.f;
        for (int j = 0; j < C; ++j) { const float v = Pm[tid][j]; m += v; if (v < eps) c += eps - v; }
        marg[tid] = m;
        gvec[tid] = m < eps ? 0.f : lamb * (m + c) / m;
    }
    __syncthreads();
    float term = 0.f, A = 0.f;
    if (tid < np) {   // clamp, entropy terms (:36-44) and the pieces of the gradient
        const bool cl = P < eps;
        const float Pc = cl ? eps : P;
        const float mi = marg[pi], mj = marg[pj];
        const float inner = logf(Pc) - lamb * logf(mj < eps ? eps : mj) - lamb * logf(mi < eps ? eps : mi);
        term = -Pc * inner;
        A = cl ? 0.f : (-inner - 1.f);
    }
    const float tt = warp_total(term), ap = warp_total(A * P);
    if (lane == 0) { red[w][0] = tt; red[w][1] = ap; }
    __syncthreads();
    if (tid == 0) {
        float l = 0.f, gp = 0.f;
        for (int g = 0; g < IG_NT / 32; ++g) { l += red[g][0]; gp += red[g][1]; }
        for (int i = 0; i < C; ++i) gp += 2.f * gvec[i] * marg[i];
        if (loss) *loss = add ? loss_w * l + add_w * (*add) : loss_w * l;
        sgp = gp;
    }
    __syncthreads();
    if (tid < np) dS[pi][pj] = gscale * (A + gvec[pi] + gvec[pj] - sgp) / T;   // dL/dSsym (symmetric), times the caller's weight
    __syncthreads();
    for (int q = tid; q < B * C; q += IG_NT) {
        const int b = q / C, c = q - b * C;
        float a1 = 0.f, a2 = 0.f;
        for (int j = 0; j < C; ++j) {
            const float d = dS[c][j];
            a1 = fmaf(z2[(size_t)b * C + j], d, a1);
            a2 = fmaf(z1[(size_t)b * C + j], d, a2);
        }
        if (dz1) dz1[q] = a1;
        if (dz2) dz2[q] = a2;
    }
}

// IIC, C > 16: S2 = sum over the ranks' partials (rank order) into the workspace, for idl_iid_joint_algebra
__global__ void __launch_bounds__(256) iid_s2_sum_kernel(const PeerPtrs s2, int world, int n, float* __restrict__ out) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    out[i] = rank_order_sum(s2, world, i, 0.f);
}

// fn of every rank ([2b, D] each, local row order) -> fn_all [2B, D] in global row order
__global__ void __launch_bounds__(256) nce_gather_rows_kernel(const PeerPtrs fn, int b, int B, int D, float* __restrict__ out) {
    const long long n = 2LL * B * D;
    for (long long idx = (long long)blockIdx.x * 256 + threadIdx.x; idx < n; idx += (long long)gridDim.x * 256) {
        const int g = (int)(idx / D), d = (int)(idx - (long long)g * D);
        const int side = g >= B ? 1 : 0, rem = g - side * B;
        const int r = rem / b, q = rem - r * b + side * b;
        const float* src = fn.p[0];
#pragma unroll
        for (int k = 1; k < MAX_PEERS; ++k)
            if (k == r) src = fn.p[k];
        out[idx] = src[(size_t)q * D + d];
    }
}

// Row block [2b, 2B] of the global similarity (rows: this rank's, columns: fn_all) -> in place grad_scale G_r with
// G = (P - Y) / (2B T): P_ij = exp(S_ij / T - lse_i) for j != i (0 on the global diagonal), Y the positive pairs.  The whole
// gradient of the global InfoNCE is (G + G^T) fn, i.e. the W of nce_weights_kernel, split by rows.  rowloss[q] = lse - S_pos / T.
// Warp <-> row; |S / T| <= 1 / T, so exp needs no running maximum (as nce_lse_kernel).
__global__ void __launch_bounds__(NCE_NT) nce_rows_kernel(float* __restrict__ S, int b, int rank, int B, float inv_t, float c,
                                                          float* __restrict__ rowloss) {
    const int lane = threadIdx.x & 31;
    const int q = blockIdx.x * NCE_RB + (threadIdx.x >> 5);
    if (q >= 2 * b) return;
    const int n = 2 * B;
    const int gi = global_row(q, b, rank, B);
    const int pos = gi < B ? gi + B : gi - B;
    float* row = S + (size_t)q * n;
    float sum = 0.f;
    for (int j = lane; j < n; j += 32)
        if (j != gi) sum += __expf(row[j] * inv_t);
    sum = warp_total(sum);   // (xor tree: every lane holds the same bits)
    const float lse = logf(sum);
    if (lane == 0) rowloss[q] = lse - row[pos] * inv_t;
    __syncwarp();
    for (int j = lane; j < n; j += 32) {
        float v = 0.f;
        if (j != gi) {
            v = __expf(row[j] * inv_t - lse);
            if (j == pos) v -= 1.f;
        }
        row[j] = c * v;
    }
}

// dh of this rank's rows through F.normalize: dfn = (sum of the local parts G_r fn_all, index order) + (sum over the ranks, rank
// order, of row gi of G_r'^T fn_r'); dh = inv_norm (dfn - fn (fn . dfn)).  Block 0 also writes the global InfoNCE loss: the ranks'
// row losses (stored behind each product) summed rank by rank, over 2B.
__global__ void __launch_bounds__(NCE_NT) nce_normalize_backward_global_kernel(const float* __restrict__ parts, int n_parts, const PeerPtrs prod,
                                                                                int world, const float* __restrict__ fn,
                                                                                const float* __restrict__ inv_norm, int b, int D, int rank,
                                                                                float* __restrict__ dh, float* __restrict__ loss) {
    const int lane = threadIdx.x & 31;
    const int q = blockIdx.x * NCE_RB + (threadIdx.x >> 5);
    const int B = world * b;
    if (blockIdx.x == 0 && threadIdx.x < 32 && loss) {
        const size_t off = (size_t)2 * B * D;
        float tot = 0.f;
#pragma unroll
        for (int r = 0; r < MAX_PEERS; ++r) {
            if (r >= world) break;
            float t = 0.f;
            for (int i = lane; i < 2 * b; i += 32) t += prod.p[r][off + i];
            tot += warp_total(t);
        }
        if (lane == 0) *loss = tot / (float)(2 * B);
    }
    if (q >= 2 * b) return;
    const int gi = global_row(q, b, rank, B);
    const size_t part = (size_t)2 * b * D;
    const float inv = inv_norm[q];
    float g[4];
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int d = lane + 32 * k;
        g[k] = 0.f;
        if (d < D) {
            for (int p = 0; p < n_parts; ++p) g[k] += parts[p * part + (size_t)q * D + d];
            g[k] = rank_order_sum(prod, world, (size_t)gi * D + d, g[k]);
            dot = fmaf(fn[(size_t)q * D + d], g[k], dot);
        }
    }
    dot = warp_total(dot);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int d = lane + 32 * k;
        if (d < D) dh[(size_t)q * D + d] = inv * (g[k] - fn[(size_t)q * D + d] * dot);
    }
}

}  // namespace idl

using namespace idl;

// the float4 kernels below need 16-byte aligned buffers (a torch view at an odd storage offset is not): rejected, not faulted on
static bool misaligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) != 0; }

// single-rank SGD / Adam: one thread per element, up to 8 CTAs per SM
template <class Op>
static int opt_step_launch(float* d_param, const float* d_grad, StatePtrs st, int64_t n, float grad_scale, Op op, void* stream) {
    if (n == 0) return IDL_OK;
    long long grid = (n + 255) / 256;
    if (grid > 148 * 8) grid = 148 * 8;
    opt_step_kernel<Op><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(d_param, d_grad, st, n, grad_scale, op); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

// the argument checks and the launch of the three *_allreduce_step entry points; `who` names the entry point in the error text,
// `state` its state buffers
template <class Op>
static int allreduce_step_launch(const char* who, const char* state, const uint64_t* h_grad_peers, const uint64_t* h_param_peers,
                                 uint64_t grad_multicast, uint64_t param_multicast, StatePtrs st, int64_t n_total, int rank, int world, Op op,
                                 void* stream) {
    bool null_state = false, odd_state = false;
    for (int k = 0; k < Op::kStates; ++k) { null_state |= !st.s[k]; odd_state |= misaligned16(st.s[k]); }
    if (!h_grad_peers || !h_param_peers || null_state || world < 1 || world > MAX_PEERS || rank < 0 || rank >= world || n_total <= 0 ||
        n_total % (4LL * world) != 0)
        return set_error(IDL_EINVAL, "%s: bad argument (n_total must be a multiple of 4 x world, world <= 16)", who);
    if (odd_state || (grad_multicast & 15) || (param_multicast & 15)) {
        char msg[128];
        snprintf(msg, sizeof msg, "%s: misaligned %s / multicast address", who, state);
        return set_error(IDL_EINVAL, "%s", msg);
    }
    PeerPtrs g, p;
    for (int r = 0; r < MAX_PEERS; ++r) { g.p[r] = nullptr; p.p[r] = nullptr; }
    for (int r = 0; r < world; ++r) {
        g.p[r] = reinterpret_cast<float*>((uintptr_t)h_grad_peers[r]);
        p.p[r] = reinterpret_cast<float*>((uintptr_t)h_param_peers[r]);
        if (!g.p[r] || !p.p[r] || (h_grad_peers[r] & 15) || (h_param_peers[r] & 15)) return set_error(IDL_EINVAL, "%s: null / misaligned peer pointer", who);
    }
    const long long shard = n_total / world;
    long long grid = (shard / 4 + 256 * AR_U - 1) / (256 * AR_U);
    if (grid > 148) grid = 148;   // measured on 2 and 8 B200s (tools/symm_probe.py): more CTAs do not move the NVLS-bound kernel
    if (grid < 1) grid = 1;
    allreduce_step_kernel<Op><<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(g, p, reinterpret_cast<const float*>((uintptr_t)grad_multicast),
                                                                                 reinterpret_cast<float*>((uintptr_t)param_multicast), st, shard, rank,
                                                                                 world, op); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

// the step counter the SGD / Adam kernels read: an int64 in device memory, so 8-byte aligned
static bool bad_step(const int64_t* d_step) { return !d_step || (reinterpret_cast<uintptr_t>(d_step) & 7) != 0; }

extern "C" {

int idl_nce_normalize(const float* d_h, int n2, int D, float* d_fn, float* d_inv_norm, void* stream) {
    if (!d_h || !d_fn || !d_inv_norm || n2 < 1 || D < 1) return set_error(IDL_EINVAL, "idl_nce_normalize: bad argument%s", "");
    nce_normalize_kernel<<<(n2 + NCE_RB - 1) / NCE_RB, NCE_NT, 0, (cudaStream_t)stream>>>(d_h, n2, D, d_fn, d_inv_norm); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_nce_softmax_xent_scaled(float* d_sim, int n2, float temperature, float grad_scale, float* d_lse, float* d_rowloss, float* d_loss, void* stream) {
    if (!d_sim || !d_lse || !d_rowloss || n2 < 2 || (n2 & 1) || !(temperature > 0.f)) return set_error(IDL_EINVAL, "idl_nce_softmax_xent: bad argument%s", "");
    cudaStream_t st = (cudaStream_t)stream;
    const float inv_t = 1.0f / temperature;
    nce_lse_kernel<<<(n2 + NCE_RB - 1) / NCE_RB, NCE_NT, 0, st>>>(d_sim, n2, inv_t, d_lse, d_rowloss); note_launch();
    if ((n2 & 3) == 0 && (reinterpret_cast<uintptr_t>(d_sim) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_lse) & 15) == 0)
        nce_weights_kernel<<<(n2 + NCE_WR - 1) / NCE_WR, 256, 0, st>>>(d_sim, d_lse, d_rowloss, n2, inv_t, grad_scale, d_loss);
    else
        nce_weights_scalar_kernel<<<n2, 256, 0, st>>>(d_sim, d_lse, d_rowloss, n2, inv_t, grad_scale, d_loss);
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_nce_softmax_xent(float* d_sim, int n2, float temperature, float* d_lse, float* d_rowloss, float* d_loss, void* stream) {
    return idl_nce_softmax_xent_scaled(d_sim, n2, temperature, 1.0f, d_lse, d_rowloss, d_loss, stream);
}

int idl_nce_normalize_backward_parts(const float* d_dfn_parts, int n_parts, const float* d_fn, const float* d_inv_norm, int n2, int D, float* d_dh,
                                     void* stream) {
    if (!d_dfn_parts || !d_fn || !d_inv_norm || !d_dh || n2 < 1 || D < 1 || n_parts < 1)
        return set_error(IDL_EINVAL, "idl_nce_normalize_backward: bad argument%s", "");
    nce_normalize_backward_kernel<<<(n2 + NCE_RB - 1) / NCE_RB, NCE_NT, 0, (cudaStream_t)stream>>>(d_dfn_parts, n_parts, d_fn, d_inv_norm, n2, D, d_dh);
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_nce_normalize_backward(const float* d_dfn, const float* d_fn, const float* d_inv_norm, int n2, int D, float* d_dh, void* stream) {
    return idl_nce_normalize_backward_parts(d_dfn, 1, d_fn, d_inv_norm, n2, D, d_dh, stream);
}

int idl_iid_joint_algebra(const float* d_S2, int C, float lamb, float eps, float grad_scale, float loss_weight, const float* d_add, float add_weight,
                          float* d_loss, float* d_joint, float* d_dS, float* d_scratch, void* stream) {
    if (!d_S2 || !d_scratch || C < 1) return set_error(IDL_EINVAL, "idl_iid_joint_algebra: bad argument%s", "");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = (C + IA_RPB - 1) / IA_RPB;
    iid_alg_rowsum_kernel<<<grid, IA_NT, 0, st>>>(d_S2, C, d_scratch); note_launch();
    iid_alg_marginal_kernel<<<grid, IA_NT, 0, st>>>(d_S2, C, lamb, eps, d_scratch, d_joint); note_launch();
    if (d_loss || d_dS) {
        iid_alg_terms_kernel<<<grid, IA_NT, 0, st>>>(d_S2, C, eps, d_scratch); note_launch();
        iid_alg_grad_kernel<<<grid, IA_NT, 0, st>>>(d_S2, C, eps, grad_scale, loss_weight, d_add, add_weight, d_scratch, d_loss, d_dS); note_launch();
    }
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_iid_loss_max_clusters(void) { return IID_MAXC; }

size_t idl_iid_loss_workspace_bytes(int C) {
    if (C < 1 || C > IID_MAXC) return 0;
    if (C <= IS_MAXC) return sizeof(float) * (3 + 2 * IID_MAXC + C * C) + 64;   // unused by the single-CTA kernels: the size this has always returned
    return sizeof(float) * (2 * (size_t)C * C + 6 * (size_t)C);                  // S2 | dS | the algebra's scratch
}

int idl_iid_loss_scaled(const float* d_z1, const float* d_z2, int B, int C, float lamb, float eps, float grad_scale, float loss_weight,
                        const float* d_add, float add_weight, float* d_loss, float* d_joint, float* d_dz1, float* d_dz2, void* d_workspace,
                        size_t workspace_bytes, void* stream) {
    if (!d_z1 || !d_z2 || !d_workspace || B < 1 || C < 1) return set_error(IDL_EINVAL, "idl_iid_loss: bad argument%s", "");
    if (C > IID_MAXC) return set_error(IDL_EUNSUPPORTED, "idl_iid_loss: n_clusters > 256 not supported%s (got %lld)", "", C);
    if (workspace_bytes < idl_iid_loss_workspace_bytes(C)) return set_error(IDL_EINVAL, "idl_iid_loss: workspace too small%s", "");
    if (C <= IS_MAXC)
        return iid_loss_small_launch(d_z1, d_z2, B, C, lamb, eps, d_loss, d_joint, d_dz1, d_dz2, stream, grad_scale, loss_weight, d_add, add_weight);
    cudaStream_t st = (cudaStream_t)stream;
    float* S2 = reinterpret_cast<float*>(d_workspace);
    float* dS = S2 + (size_t)C * C;
    float* scratch = dS + (size_t)C * C;
    const int nt = (C + IC_T - 1) / IC_T;
    const bool grad = d_dz1 || d_dz2;
    iid_s2_kernel<<<nt * (nt + 1) / 2, IC_NT, 0, st>>>(d_z1, d_z2, B, C, nt, S2); note_launch();
    const int rc = idl_iid_joint_algebra(S2, C, lamb, eps, grad_scale, loss_weight, d_add, add_weight, d_loss, d_joint, grad ? dS : nullptr, scratch,
                                         stream);
    if (rc != IDL_OK || !grad) return rc;
    iid_dz_kernel<<<dim3((B + IC_BR - 1) / IC_BR, nt, 2), IC_NT, 0, st>>>(d_z1, d_z2, dS, B, C, d_dz1, d_dz2); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_iid_loss(const float* d_z1, const float* d_z2, int B, int C, float lamb, float eps, float* d_loss, float* d_joint, float* d_dz1, float* d_dz2,
                 void* d_workspace, size_t workspace_bytes, void* stream) {
    return idl_iid_loss_scaled(d_z1, d_z2, B, C, lamb, eps, 1.0f, 1.0f, nullptr, 0.0f, d_loss, d_joint, d_dz1, d_dz2, d_workspace, workspace_bytes,
                               stream);
}

int idl_relu_dropout_forward(const float* d_parts, int n_parts, const float* d_bias, int64_t M, int N, float p, uint64_t seed, const int64_t* d_step,
                             uint32_t tag, float* d_out, void* stream) {
    if (!d_parts || !d_out || n_parts < 1 || M < 1 || N < 4 || (N & 3) || !(p >= 0.f) || !(p < 1.f))
        return set_error(IDL_EINVAL, "idl_relu_dropout_forward: bad argument%s (N must be a multiple of 4, 0 <= p < 1)", "");
    if (misaligned16(d_parts) || misaligned16(d_bias) || misaligned16(d_out))
        return set_error(IDL_EINVAL, "idl_relu_dropout_forward: misaligned buffer%s (parts, bias and out are read and written as float4)", "");
    const long long n4 = (long long)M * N / 4;
    const double th = (double)p * 4294967296.0;
    const uint32_t thresh = th >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)th;
    long long grid = (n4 + 255) / 256;
    if (grid > 148 * 8) grid = 148 * 8;
    relu_dropout_fwd_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(d_parts, n_parts, d_bias, n4, N / 4, thresh, 1.0f / (1.0f - p), seed,
                                                                              reinterpret_cast<const long long*>(d_step), tag, d_out);
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_sum_parts_bias(const float* d_parts, int n_parts, const float* d_bias, int64_t M, int N, float* d_out, void* stream) {
    if (!d_parts || !d_out || n_parts < 1 || M < 1 || N < 4 || (N & 3)) return set_error(IDL_EINVAL, "idl_sum_parts_bias: bad argument%s (N must be a multiple of 4)", "");
    if (misaligned16(d_parts) || misaligned16(d_bias) || misaligned16(d_out))
        return set_error(IDL_EINVAL, "idl_sum_parts_bias: misaligned buffer%s (parts, bias and out are read and written as float4)", "");
    const long long n4 = (long long)M * N / 4;
    long long grid = (n4 + 255) / 256;
    if (grid > 148 * 8) grid = 148 * 8;
    sum_parts_bias_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(d_parts, n_parts, d_bias, n4, N / 4, d_out);
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_relu_dropout_backward(const float* d_out, const float* d_dy, int64_t n, float p, float* d_dx, void* stream) {
    if (!d_out || !d_dy || !d_dx || n < 4 || (n & 3) || !(p >= 0.f) || !(p < 1.f)) return set_error(IDL_EINVAL, "idl_relu_dropout_backward: bad argument%s", "");
    if (misaligned16(d_out) || misaligned16(d_dy) || misaligned16(d_dx))
        return set_error(IDL_EINVAL, "idl_relu_dropout_backward: misaligned buffer%s (out, dy and dx are read and written as float4)", "");
    long long grid = (n / 4 + 255) / 256;
    if (grid > 148 * 8) grid = 148 * 8;
    relu_dropout_bwd_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(d_out, d_dy, n / 4, 1.0f / (1.0f - p), d_dx);
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_pair_selection(const int64_t* d_pair_ids, int n, int64_t n_seqs, int32_t* d_sidx, int32_t* d_sel, void* stream) {
    if (!d_pair_ids || !d_sidx || !d_sel || n < 0 || n_seqs < 1) return set_error(IDL_EINVAL, "idl_pair_selection: bad argument%s", "");
    if (n == 0) return IDL_OK;
    pair_selection_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const long long*>(d_pair_ids), n, (long long)n_seqs, d_sidx,
                                                                            d_sel);
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_rmsprop_step(float* d_param, const float* d_grad, float* d_square_avg, int64_t n, float lr, float alpha, float eps, float weight_decay,
                     float grad_scale, void* stream) {
    if (!d_param || !d_grad || !d_square_avg || n < 0) return set_error(IDL_EINVAL, "idl_rmsprop_step: bad argument%s", "");
    if (n == 0) return IDL_OK;
    long long grid = (n + 255) / 256;
    if (grid > 148 * 8) grid = 148 * 8;
    rmsprop_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(d_param, d_grad, d_square_avg, n, lr, alpha, eps, weight_decay, grad_scale); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_rmsprop_allreduce_step(const uint64_t* h_grad_peers, const uint64_t* h_param_peers, uint64_t grad_multicast, uint64_t param_multicast,
                               float* d_square_avg, int64_t n_total, int rank, int world, float lr, float alpha, float eps, float weight_decay,
                               void* stream) {
    return allreduce_step_launch("idl_rmsprop_allreduce_step", "square_avg", h_grad_peers, h_param_peers, grad_multicast, param_multicast,
                                 StatePtrs{{d_square_avg, nullptr}}, n_total, rank, world, RmspropUpdate{lr, alpha, eps, weight_decay}, stream);
}

int idl_sgd_step(float* d_param, const float* d_grad, float* d_momentum_buf, int64_t n, float lr, float momentum, float weight_decay,
                 const int64_t* d_step, float grad_scale, void* stream) {
    if (!d_param || !d_grad || !d_momentum_buf || n < 0) return set_error(IDL_EINVAL, "idl_sgd_step: bad argument%s", "");
    if (bad_step(d_step)) return set_error(IDL_EINVAL, "idl_sgd_step: null / misaligned step counter%s (int64 in device memory)", "");
    return opt_step_launch(d_param, d_grad, StatePtrs{{d_momentum_buf, nullptr}}, n, grad_scale,
                           SgdUpdate{lr, momentum, weight_decay, reinterpret_cast<const long long*>(d_step), false}, stream);
}

int idl_adam_step(float* d_param, const float* d_grad, float* d_exp_avg, float* d_exp_avg_sq, int64_t n, float lr, double beta1, double beta2,
                  float eps, float weight_decay, const int64_t* d_step, float grad_scale, void* stream) {
    if (!d_param || !d_grad || !d_exp_avg || !d_exp_avg_sq || n < 0) return set_error(IDL_EINVAL, "idl_adam_step: bad argument%s", "");
    if (bad_step(d_step)) return set_error(IDL_EINVAL, "idl_adam_step: null / misaligned step counter%s (int64 in device memory)", "");
    return opt_step_launch(d_param, d_grad, StatePtrs{{d_exp_avg, d_exp_avg_sq}}, n, grad_scale,
                           AdamUpdate{lr, eps, weight_decay, beta1, beta2, reinterpret_cast<const long long*>(d_step), 0.f, 0.f, 0.f, 0.f, 0.f}, stream);
}

int idl_sgd_allreduce_step(const uint64_t* h_grad_peers, const uint64_t* h_param_peers, uint64_t grad_multicast, uint64_t param_multicast,
                           float* d_momentum_buf, int64_t n_total, int rank, int world, float lr, float momentum, float weight_decay,
                           const int64_t* d_step, void* stream) {
    if (bad_step(d_step)) return set_error(IDL_EINVAL, "idl_sgd_allreduce_step: null / misaligned step counter%s (int64 in device memory)", "");
    return allreduce_step_launch("idl_sgd_allreduce_step", "momentum_buffer", h_grad_peers, h_param_peers, grad_multicast, param_multicast,
                                 StatePtrs{{d_momentum_buf, nullptr}}, n_total, rank, world,
                                 SgdUpdate{lr, momentum, weight_decay, reinterpret_cast<const long long*>(d_step), false}, stream);
}

int idl_adam_allreduce_step(const uint64_t* h_grad_peers, const uint64_t* h_param_peers, uint64_t grad_multicast, uint64_t param_multicast,
                            float* d_exp_avg, float* d_exp_avg_sq, int64_t n_total, int rank, int world, float lr, double beta1, double beta2, float eps,
                            float weight_decay, const int64_t* d_step, void* stream) {
    if (bad_step(d_step)) return set_error(IDL_EINVAL, "idl_adam_allreduce_step: null / misaligned step counter%s (int64 in device memory)", "");
    return allreduce_step_launch("idl_adam_allreduce_step", "exp_avg / exp_avg_sq", h_grad_peers, h_param_peers, grad_multicast, param_multicast,
                                 StatePtrs{{d_exp_avg, d_exp_avg_sq}}, n_total, rank, world,
                                 AdamUpdate{lr, eps, weight_decay, beta1, beta2, reinterpret_cast<const long long*>(d_step), 0.f, 0.f, 0.f, 0.f, 0.f}, stream);
}

// ---- global-batch losses (see the kernels above) ----

// the `world` float buffers of a host peer table; false when one is null or not 4-byte aligned
static bool peer_floats(const uint64_t* h_peers, int world, PeerPtrs& out) {
    for (int r = 0; r < MAX_PEERS; ++r) out.p[r] = nullptr;
    for (int r = 0; r < world; ++r) {
        if (!h_peers[r] || (h_peers[r] & 3)) return false;
        out.p[r] = reinterpret_cast<float*>((uintptr_t)h_peers[r]);
    }
    return true;
}

// b rows per rank, world ranks, D columns: 1 <= world <= 16, b >= 1, and the [2B, D] / [2b, 2B] operands indexable with int rows
static bool bad_rows(int b, int world, int64_t width) { return world < 1 || world > MAX_PEERS || b < 1 || 2LL * b * world * width > INT32_MAX; }

int idl_iid_partial_s2(const float* d_z1, const float* d_z2, int B, int C, float* d_S2, void* stream) {
    if (!d_z1 || !d_z2 || !d_S2 || B < 1 || C < 1 || C > IID_MAXC)
        return set_error(IDL_EINVAL, "idl_iid_partial_s2: bad argument%s (B >= 1, 1 <= C <= 256)", "");
    const int nt = (C + IC_T - 1) / IC_T;
    iid_s2_kernel<<<nt * (nt + 1) / 2, IC_NT, 0, (cudaStream_t)stream>>>(d_z1, d_z2, B, C, nt, d_S2); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_iid_global_finish(const uint64_t* h_s2_peers, int world, const float* d_z1, const float* d_z2, int B, int C, float lamb, float eps,
                          float grad_scale, float loss_weight, const float* d_add, float add_weight, float* d_loss, float* d_dz1, float* d_dz2,
                          void* d_workspace, size_t workspace_bytes, void* stream) {
    if (!h_s2_peers || !d_z1 || !d_z2 || !d_workspace || world < 1 || world > MAX_PEERS || B < 1 || C < 1 || C > IID_MAXC)
        return set_error(IDL_EINVAL, "idl_iid_global_finish: bad argument%s (world 1..16, B >= 1, 1 <= C <= 256)", "");
    if (workspace_bytes < idl_iid_loss_workspace_bytes(C)) return set_error(IDL_EINVAL, "idl_iid_global_finish: workspace too small%s", "");
    PeerPtrs s2;
    if (!peer_floats(h_s2_peers, world, s2)) return set_error(IDL_EINVAL, "idl_iid_global_finish: null / misaligned peer pointer%s", "");
    cudaStream_t st = (cudaStream_t)stream;
    if (C <= IS_MAXC) {
        iid_global_small_kernel<<<1, IG_NT, 0, st>>>(s2, world, d_z1, d_z2, B, C, lamb, eps, grad_scale, loss_weight, d_add, add_weight, d_loss, d_dz1,
                                                     d_dz2); note_launch();
        IDL_CUDA_CHECK(cudaGetLastError());
        return IDL_OK;
    }
    float* S2 = reinterpret_cast<float*>(d_workspace);
    float* dS = S2 + (size_t)C * C;
    float* scratch = dS + (size_t)C * C;
    const bool grad = d_dz1 || d_dz2;
    iid_s2_sum_kernel<<<(C * C + 255) / 256, 256, 0, st>>>(s2, world, C * C, S2); note_launch();
    const int rc = idl_iid_joint_algebra(S2, C, lamb, eps, grad_scale, loss_weight, d_add, add_weight, d_loss, nullptr, grad ? dS : nullptr, scratch,
                                         stream);
    if (rc != IDL_OK || !grad) return rc;
    const int nt = (C + IC_T - 1) / IC_T;
    iid_dz_kernel<<<dim3((B + IC_BR - 1) / IC_BR, nt, 2), IC_NT, 0, st>>>(d_z1, d_z2, dS, B, C, d_dz1, d_dz2); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_nce_gather_rows(const uint64_t* h_fn_peers, int world, int b, int D, float* d_fn_all, void* stream) {
    if (!h_fn_peers || !d_fn_all || D < 1 || bad_rows(b, world, D))
        return set_error(IDL_EINVAL, "idl_nce_gather_rows: bad argument%s (world 1..16, b >= 1, D >= 1, 2 b world D < 2^31)", "");
    PeerPtrs fn;
    if (!peer_floats(h_fn_peers, world, fn)) return set_error(IDL_EINVAL, "idl_nce_gather_rows: null / misaligned peer pointer%s", "");
    const long long n = 2LL * b * world * D;
    long long grid = (n + 255) / 256;
    if (grid > 148 * 4) grid = 148 * 4;
    nce_gather_rows_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(fn, b, b * world, D, d_fn_all); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_nce_softmax_xent_rows(float* d_sim, int b, int rank, int world, float temperature, float grad_scale, float* d_rowloss, void* stream) {
    if (!d_sim || !d_rowloss || !(temperature > 0.f) || rank < 0 || rank >= world || bad_rows(b, world, 2LL * b * world))
        return set_error(IDL_EINVAL, "idl_nce_softmax_xent_rows: bad argument%s (world 1..16, 0 <= rank < world, b >= 1, 4 b^2 world^2 < 2^31)", "");
    const float inv_t = 1.0f / temperature;
    const int B = b * world;
    nce_rows_kernel<<<(2 * b + NCE_RB - 1) / NCE_RB, NCE_NT, 0, (cudaStream_t)stream>>>(d_sim, b, rank, B, inv_t, grad_scale * inv_t / (float)(2 * B),
                                                                                       d_rowloss); note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

int idl_nce_normalize_backward_global(const float* d_dfn_parts, int n_parts, const uint64_t* h_prod_peers, int world, const float* d_fn,
                                      const float* d_inv_norm, int b, int D, int rank, float* d_dh, float* d_loss, void* stream) {
    if (!d_dfn_parts || !h_prod_peers || !d_fn || !d_inv_norm || !d_dh || n_parts < 1 || D < 1 || D > 128 || rank < 0 || rank >= world ||
        bad_rows(b, world, D + 1))
        return set_error(IDL_EINVAL, "idl_nce_normalize_backward_global: bad argument%s (world 1..16, 0 <= rank < world, b >= 1, 1 <= D <= 128)", "");
    PeerPtrs prod;
    if (!peer_floats(h_prod_peers, world, prod)) return set_error(IDL_EINVAL, "idl_nce_normalize_backward_global: null / misaligned peer pointer%s", "");
    nce_normalize_backward_global_kernel<<<(2 * b + NCE_RB - 1) / NCE_RB, NCE_NT, 0, (cudaStream_t)stream>>>(d_dfn_parts, n_parts, prod, world, d_fn,
                                                                                                           d_inv_norm, b, D, rank, d_dh, d_loss);
    note_launch();
    IDL_CUDA_CHECK(cudaGetLastError());
    return IDL_OK;
}

}  // extern "C"
