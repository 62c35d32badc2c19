// lz_nn.cu -- fused elementwise epilogues around the network's convolutions (bf16, channels-last).
//
// The dense contraction itself (3x3 convolutions as implicit GEMMs) stays with PyTorch/cuDNN on the tensor
// cores (north_star); measured on B200 those run at ~90 % of the sustained bf16 peak, but PyTorch's eval-mode
// BatchNorm + ReLU + residual add around them are separate HBM-bound passes that cost more than the convs.
// A pre-activation residual block  x' = x + conv2(relu(bn2(conv1(relu(bn1(x))))))  needs, per conv, exactly
// one such pass if the passes are fused:
//     bn_relu      : a  = relu(scale * u + shift)
//     add_bn_relu  : x' = u + v ;  a = relu(scale * x' + shift)          (scale/shift of the NEXT block's bn1)
// Rows are (n, h, w) positions, C channels contiguous (NHWC); each thread handles 8 channels (16 B vectors).
// HBM-bound: 2 x 2 B/element for bn_relu, 4 x 2 B/element for add_bn_relu.
#include <cuda_bf16.h>

#include "lz_common.cuh"

namespace lzb {
namespace {

struct alignas(16) bf16x8 { __nv_bfloat162 v[4]; };

template <bool kAdd, bool kWriteSum>
__global__ void __launch_bounds__(256)
bn_relu_kernel(const bf16x8* __restrict__ u, const bf16x8* __restrict__ v, const float* __restrict__ scale,
               const float* __restrict__ shift, int64_t total_vec, int vec_per_row, bf16x8* __restrict__ out_sum,
               bf16x8* __restrict__ out_act) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec; i += (int64_t)gridDim.x * blockDim.x) {
        const int c0 = (int)(i % vec_per_row) * 8;
        bf16x8 a = u[i];
        bf16x8 s, r;
        bf16x8 b;
        if (kAdd) b = v[i];
        const float4 sc0 = *reinterpret_cast<const float4*>(scale + c0), sc1 = *reinterpret_cast<const float4*>(scale + c0 + 4);
        const float4 sh0 = *reinterpret_cast<const float4*>(shift + c0), sh1 = *reinterpret_cast<const float4*>(shift + c0 + 4);
        const float scv[8] = {sc0.x, sc0.y, sc0.z, sc0.w, sc1.x, sc1.y, sc1.z, sc1.w};
        const float shv[8] = {sh0.x, sh0.y, sh0.z, sh0.w, sh1.x, sh1.y, sh1.z, sh1.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float2 x = __bfloat1622float2(a.v[k]);
            if (kAdd) {
                const float2 y = __bfloat1622float2(b.v[k]);
                // the residual stream is stored in bf16 (as PyTorch's bf16 add does) and BN reads the stored value
                s.v[k] = __floats2bfloat162_rn(x.x + y.x, x.y + y.y);
                x = __bfloat1622float2(s.v[k]);
            }
            const float r0 = fmaxf(fmaf(x.x, scv[2 * k], shv[2 * k]), 0.0f);
            const float r1 = fmaxf(fmaf(x.y, scv[2 * k + 1], shv[2 * k + 1]), 0.0f);
            r.v[k] = __floats2bfloat162_rn(r0, r1);
        }
        if (kAdd && kWriteSum) out_sum[i] = s;
        out_act[i] = r;
    }
}

}  // namespace
}  // namespace lzb

using namespace lzb;

extern "C" int lzb_bn_relu_bf16(const void* u, const void* v, const float* scale, const float* shift, int64_t rows,
                                int32_t channels, void* out_sum, void* out_act, void* stream) {
    LZB_REQUIRE(rows >= 0 && channels > 0 && channels % 8 == 0, "channels must be a positive multiple of 8");
    if (rows == 0) return LZB_OK;
    LZB_REQUIRE(u && scale && shift && out_act, "null pointer");
    LZB_REQUIRE(((reinterpret_cast<uintptr_t>(u) | reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(out_sum) |
                  reinterpret_cast<uintptr_t>(out_act) | reinterpret_cast<uintptr_t>(scale) |
                  reinterpret_cast<uintptr_t>(shift)) & 15) == 0, "pointers must be 16-byte aligned");
    const int vec_per_row = channels / 8;
    const int64_t total = rows * vec_per_row;
    const int grid = thread_grid(total, 256);
    cudaStream_t s = (cudaStream_t)stream;
    const bf16x8* pu = reinterpret_cast<const bf16x8*>(u);
    const bf16x8* pv = reinterpret_cast<const bf16x8*>(v);
    bf16x8* ps = reinterpret_cast<bf16x8*>(out_sum);
    bf16x8* pa = reinterpret_cast<bf16x8*>(out_act);
    if (!v) bn_relu_kernel<false, false><<<grid, 256, 0, s>>>(pu, pv, scale, shift, total, vec_per_row, ps, pa);
    else if (out_sum) bn_relu_kernel<true, true><<<grid, 256, 0, s>>>(pu, pv, scale, shift, total, vec_per_row, ps, pa);
    else bn_relu_kernel<true, false><<<grid, 256, 0, s>>>(pu, pv, scale, shift, total, vec_per_row, ps, pa);
    return check_launch("bn_relu_kernel");
}

// ------------------------------------------------------------------------------------------------------
// Fused network heads (src/neural_network.py:98-151 + project_policy_logits_fast + bucket_logits_to_scalar).
// Input: pv = relu(bn(conv1x1([policy.conv1 ; value.conv1])(trunk)))  bf16 [n, 36, pc + vc] channels-last, i.e.
// the two heads' 1x1 convolutions run as ONE convolution; everything after it -- global pooling (mean / max /
// std), gpool_linear, bn2 + relu, the three 1-channel output convs, log-softmax, the value MLP, the bucket
// expectation and the masked softmax over the legal actions of the packed state -- is this one kernel
// (~30 PyTorch launches in the unfused path).
//
// A 256-thread block processes a TILE of kTile = 8 states: 512 blocks for a 4,096-leaf wave, all resident at once
// (3-4 per SM), so the latency of the small dense layers is hidden by other blocks.  Pooled features / hidden
// activations live in shared memory TRANSPOSED ([feature][state]) so that one broadcast 8/16-byte shared load
// feeds 2/4 FMAs; weights are pre-transposed (consecutive threads read consecutive addresses) and every weight
// element is used for kTile/groups states from a register.  fp32 math throughout.
// ------------------------------------------------------------------------------------------------------
namespace lzb {
namespace {

constexpr int kHeadsThreads = 256;
constexpr int kTile = 8;
constexpr int kMaxHeadCh = 64;     // policy_channels, value_channels <= 64
constexpr int kMaxMlp = 128;       // value_mlp_channels <= 128
constexpr int kMaxBins = 128;      // value buckets <= 128

struct HeadsParams {
    const __nv_bfloat16* pv; int64_t n; int pc, vc, mlp, bins;
    const float *wgl_t, *bn2_scale, *bn2_shift, *wout, *wfc1_t, *bfc1, *wfc2_t, *bfc2;
    const uint64_t* states; float *priors, *values, *log_heads, *value_logits;
};

__device__ __forceinline__ uint32_t to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
// C[8 states x 8 outputs] += A[8 x K] * B[K x 8] for one n-tile.  featT = features transposed in shared memory,
// [K][kTile] fp32 (A fragment: a0 = (row lane/4, k lane%4), a2 = (row lane/4, k lane%4 + 4); rows 8-15 are zero
// padding).  wfrag = this n-tile's packed B fragments: [k_step][lane] float2 = (B[k lane%4][n lane/4], B[k lane%4 + 4][..]).
// Result: c0 / c1 = C[row lane/4][col 2*(lane%4) (+1)].
__device__ __forceinline__ void mma_rows8(const float* __restrict__ wfrag, int ks_n, int K, const float* featT, int lane,
                                          float& c0, float& c1) {
    float c2 = 0.0f, c3 = 0.0f;
    const int kq = lane & 3, row = lane >> 2;
#pragma unroll 4
    for (int ks = 0; ks < ks_n; ++ks) {
        const float2 b = __ldg(reinterpret_cast<const float2*>(wfrag) + ks * 32 + lane);
        const int k0 = ks * 8 + kq;
        const uint32_t a0 = k0 < K ? to_tf32(featT[k0 * kTile + row]) : 0u;
        const uint32_t a2 = k0 + 4 < K ? to_tf32(featT[(k0 + 4) * kTile + row]) : 0u;
        asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
                     "{%0, %1, %2, %3};"
                     : "+f"(c0), "+f"(c1), "+f"(c2), "+f"(c3)
                     : "r"(a0), "r"(0u), "r"(a2), "r"(0u), "r"(__float_as_uint(b.x)), "r"(__float_as_uint(b.y)));
    }
}

__global__ void __launch_bounds__(kHeadsThreads, 4)
heads_tail_kernel(HeadsParams P) {
    __shared__ __align__(16) float poolT_p[3 * kMaxHeadCh][kTile];   // [feature][state]
    __shared__ __align__(16) float poolT_v[3 * kMaxHeadCh][kTile];
    __shared__ __align__(16) float g[kTile][kMaxHeadCh];
    __shared__ __align__(16) float hidT[kMaxMlp][kTile];
    __shared__ float vlog[kTile][kMaxBins + 1];
    __shared__ float lp[kTile][3][36];
    __shared__ __align__(16) float wpol[5][kMaxHeadCh];               // bn2 scale, bn2 shift, out_pos1, out_pos2, out_mark
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int pc = P.pc, vc = P.vc, c2 = pc + vc, mlp = P.mlp, bins = P.bins;
    for (int i = t; i < pc; i += kHeadsThreads) {
        wpol[0][i] = P.bn2_scale[i]; wpol[1][i] = P.bn2_shift[i];
        wpol[2][i] = P.wout[i]; wpol[3][i] = P.wout[pc + i]; wpol[4][i] = P.wout[2 * pc + i];
    }
    const int64_t num_tiles = (P.n + kTile - 1) / kTile;
    for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int64_t base = tile * kTile;
        const int ns = (int)min((int64_t)kTile, P.n - base);
        __syncthreads();
        // 1. global pooling per (state, channel): mean / max / std (biased variance + 1e-6)  neural_network.py:68-81
        //    thread -> (state, channel octet, half of the board): 18 independent 16-byte loads, one pass (max in fp32,
        //    and the sum and sum of squares of d = x - K in fp32); the two halves sit in adjacent lanes and meet by
        //    shuffle.  The shift K is the channel's value at cell 0, which both halves load: var = E[d^2] - E[d]^2
        //    then does not cancel on a channel that is nearly constant over the board (E[x^2] - E[x]^2 loses all of
        //    its bits there), and since d_0 = 0, E[d]^2 <= 36 var bounds the cancellation everywhere.  For bf16 x,
        //    x - K is exact unless the two magnitudes are more than 2^16 apart.
        {
            const int octets = c2 >> 3, items = kTile * octets * 2;
            for (int idx0 = 0; idx0 < items; idx0 += kHeadsThreads) {
                const int idx = idx0 + t;
                const bool valid = idx < items;
                const int hf = idx & 1, so = idx >> 1, s = valid ? so / octets : 0, o = valid ? so - s * octets : 0;
                float sm[8], sq[8], mx[8], k0[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) { sm[c] = 0.0f; sq[c] = 0.0f; mx[c] = -INFINITY; k0[c] = 0.0f; }
                if (valid && s < ns) {
                    const uint4* board = reinterpret_cast<const uint4*>(P.pv + (base + s) * 36 * c2 + o * 8);
                    const int stride = c2 >> 3;                    // uint4 per cell
                    const uint4 raw0 = __ldg(board);
                    const uint32_t w0[4] = {raw0.x, raw0.y, raw0.z, raw0.w};
#pragma unroll
                    for (int h = 0; h < 4; ++h) { k0[2 * h] = __uint_as_float(w0[h] << 16); k0[2 * h + 1] = __uint_as_float(w0[h] & 0xffff0000u); }
                    const uint4* src = board + hf * 18 * stride;
#pragma unroll
                    for (int cell = 0; cell < 18; ++cell) {
                        const uint4 raw = __ldg(src + cell * stride);
                        const uint32_t wv[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
                        for (int h = 0; h < 4; ++h) {
                            const float lo = __uint_as_float(wv[h] << 16), hi = __uint_as_float(wv[h] & 0xffff0000u);
                            const float dl = lo - k0[2 * h], dh = hi - k0[2 * h + 1];
                            sm[2 * h] += dl; sq[2 * h] = fmaf(dl, dl, sq[2 * h]); mx[2 * h] = fmaxf(mx[2 * h], lo);
                            sm[2 * h + 1] += dh; sq[2 * h + 1] = fmaf(dh, dh, sq[2 * h + 1]); mx[2 * h + 1] = fmaxf(mx[2 * h + 1], hi);
                        }
                    }
                }
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    sm[c] += __shfl_xor_sync(0xffffffffu, sm[c], 1);
                    sq[c] += __shfl_xor_sync(0xffffffffu, sq[c], 1);
                    mx[c] = fmaxf(mx[c], __shfl_xor_sync(0xffffffffu, mx[c], 1));
                }
                if (valid && hf == 0) {
                    const bool live = s < ns;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const int ch = o * 8 + c;
                        const float md = sm[c] * (1.0f / 36.0f);
                        const float var = fmaxf(fmaf(-md, md, sq[c] * (1.0f / 36.0f)), 0.0f);
                        const float r0 = live ? k0[c] + md : 0.0f, r1 = live ? mx[c] : 0.0f, r2 = live ? sqrtf(var + 1e-6f) : 1e-3f;
                        if (ch < pc) { poolT_p[ch][s] = r0; poolT_p[pc + ch][s] = r1; poolT_p[2 * pc + ch][s] = r2; }
                        else { const int cv = ch - pc; poolT_v[cv][s] = r0; poolT_v[vc + cv][s] = r1; poolT_v[2 * vc + cv][s] = r2; }
                    }
                }
            }
        }
        __syncthreads();
        // 2a / 2b / 3a: the three small dense layers on the tensor cores (mma.sync m16n8k8, TF32 inputs, fp32
        // accumulate): M = the tile's 8 states (rows 8-15 of the fragment are padding), N = outputs in tiles of 8
        // spread over the 8 warps, K in steps of 8.  Weights are pre-packed on the host in B-fragment order
        // ([n_tile][k_step][lane] float2, TF32-rounded), so each mma costs one coalesced 8-byte load per lane; the
        // A fragments come from the transposed feature tiles in shared memory (conflict-free).  This replaced a CUDA-core
        // version that was issue-bound at 21 k instructions per warp (ncu), 60 % of them in these three layers.
        // 2a. g = gpool_linear(pooled_p) (no bias)
        {
            const int K = 3 * pc, ks_n = (K + 7) >> 3, nt_n = (pc + 7) >> 3;
            for (int nt = warp; nt < nt_n; nt += kHeadsThreads / 32) {
                float c0 = 0.0f, c1 = 0.0f;
                mma_rows8(P.wgl_t + (size_t)nt * ks_n * 64, ks_n, K, &poolT_p[0][0], lane, c0, c1);
                const int j = nt * 8 + 2 * (lane & 3), srow = lane >> 2;
                if (j < pc) g[srow][j] = c0;
                if (j + 1 < pc) g[srow][j + 1] = c1;
            }
        }
        // 2b. hid = relu(fc1(pooled_v))
        {
            const int K = 3 * vc, ks_n = (K + 7) >> 3, nt_n = (mlp + 7) >> 3;
            for (int nt = warp; nt < nt_n; nt += kHeadsThreads / 32) {
                float c0 = 0.0f, c1 = 0.0f;
                mma_rows8(P.wfc1_t + (size_t)nt * ks_n * 64, ks_n, K, &poolT_v[0][0], lane, c0, c1);
                const int m = nt * 8 + 2 * (lane & 3), srow = lane >> 2;
                if (m < mlp) hidT[m][srow] = fmaxf(c0 + __ldg(P.bfc1 + m), 0.0f);
                if (m + 1 < mlp) hidT[m + 1][srow] = fmaxf(c1 + __ldg(P.bfc1 + m + 1), 0.0f);
            }
        }
        __syncthreads();
        // 3a. value logits = fc2(hid)
        {
            const int K = mlp, ks_n = (K + 7) >> 3, nt_n = (bins + 7) >> 3;
            for (int nt = warp; nt < nt_n; nt += kHeadsThreads / 32) {
                float c0 = 0.0f, c1 = 0.0f;
                mma_rows8(P.wfc2_t + (size_t)nt * ks_n * 64, ks_n, K, &hidT[0][0], lane, c0, c1);
                const int k = nt * 8 + 2 * (lane & 3), srow = lane >> 2;
                if (k < bins) vlog[srow][k] = c0 + __ldg(P.bfc2 + k);
                if (k + 1 < bins) vlog[srow][k + 1] = c1 + __ldg(P.bfc2 + k + 1);
            }
        }
        // 3b. policy: p2 = relu(bn2(p + g)); three 1-channel output convs -> raw logits (stored in lp).
        //     thread -> (state, cell, channel half); the two halves sit in adjacent lanes and meet by shuffle
        {
            const int half_ch = (pc + 1) >> 1;
            const bool vec = (pc % 16 == 0) && (c2 % 8 == 0);
            for (int idx0 = 0; idx0 < ns * 72; idx0 += kHeadsThreads) {
                const int idx = idx0 + t;
                const bool valid = idx < ns * 72;
                float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f;
                int s = 0, cell = 0;
                if (valid) {
                    const int item = idx >> 1, half = idx & 1;
                    s = item / 36; cell = item - s * 36;
                    const int ch0 = half * half_ch, ch1 = half ? pc : half_ch;
                    const __nv_bfloat16* src = P.pv + ((base + s) * 36 + cell) * c2;
                    if (vec) {
                        for (int ch = ch0; ch < ch1; ch += 8) {
                            const uint4 raw = *reinterpret_cast<const uint4*>(src + ch);
                            const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&raw);
                            float x[8];
#pragma unroll
                            for (int q = 0; q < 4; ++q) { const float2 f = __bfloat1622float2(h2[q]); x[2 * q] = f.x; x[2 * q + 1] = f.y; }
#pragma unroll
                            for (int q4 = 0; q4 < 2; ++q4) {
                                const float4 gg = *reinterpret_cast<const float4*>(&g[s][ch + 4 * q4]);
                                const float4 sc = *reinterpret_cast<const float4*>(&wpol[0][ch + 4 * q4]);
                                const float4 sh = *reinterpret_cast<const float4*>(&wpol[1][ch + 4 * q4]);
                                const float4 w0 = *reinterpret_cast<const float4*>(&wpol[2][ch + 4 * q4]);
                                const float4 w1 = *reinterpret_cast<const float4*>(&wpol[3][ch + 4 * q4]);
                                const float4 w2 = *reinterpret_cast<const float4*>(&wpol[4][ch + 4 * q4]);
                                const float gv[4] = {gg.x, gg.y, gg.z, gg.w}, scv[4] = {sc.x, sc.y, sc.z, sc.w};
                                const float shv[4] = {sh.x, sh.y, sh.z, sh.w}, w0v[4] = {w0.x, w0.y, w0.z, w0.w};
                                const float w1v[4] = {w1.x, w1.y, w1.z, w1.w}, w2v[4] = {w2.x, w2.y, w2.z, w2.w};
#pragma unroll
                                for (int q = 0; q < 4; ++q) {
                                    const float p2 = fmaxf(fmaf(scv[q], x[4 * q4 + q] + gv[q], shv[q]), 0.0f);
                                    a0 = fmaf(w0v[q], p2, a0); a1 = fmaf(w1v[q], p2, a1); a2 = fmaf(w2v[q], p2, a2);
                                }
                            }
                        }
                    } else {
                        for (int ch = ch0; ch < ch1; ++ch) {
                            const float p2 = fmaxf(fmaf(wpol[0][ch], __bfloat162float(src[ch]) + g[s][ch], wpol[1][ch]), 0.0f);
                            a0 = fmaf(wpol[2][ch], p2, a0); a1 = fmaf(wpol[3][ch], p2, a1); a2 = fmaf(wpol[4][ch], p2, a2);
                        }
                    }
                }
                // channel order of the sum: low half first, then the high half (fixed -> run-to-run deterministic)
                const float b0 = __shfl_xor_sync(0xffffffffu, a0, 1), b1 = __shfl_xor_sync(0xffffffffu, a1, 1);
                const float b2 = __shfl_xor_sync(0xffffffffu, a2, 1);
                if (valid && !(idx & 1)) { lp[s][0][cell] = a0 + b0; lp[s][1][cell] = a1 + b1; lp[s][2][cell] = a2 + b2; }
            }
        }
        __syncthreads();
        // 4. log-softmax of each (state, head) row over the 36 cells; value expectation per state
        for (int row = warp; row < ns * 3; row += kHeadsThreads / 32) {
            const int s = row / 3, h = row - s * 3;
            const float x0 = lp[s][h][lane], x1 = lane < 4 ? lp[s][h][32 + lane] : -INFINITY;
            float mx = fmaxf(x0, x1);
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            float se = expf(x0 - mx) + (lane < 4 ? expf(x1 - mx) : 0.0f);
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) se += __shfl_xor_sync(0xffffffffu, se, off);
            const float lse = mx + logf(se);
            lp[s][h][lane] = x0 - lse;
            if (lane < 4) lp[s][h][32 + lane] = x1 - lse;
            if (P.log_heads) {
                float* dst = P.log_heads + ((base + s) * 3 + h) * 36;
                dst[lane] = x0 - lse;
                if (lane < 4) dst[32 + lane] = x1 - lse;
            }
        }
        for (int s = warp; s < ns; s += kHeadsThreads / 32) {
            float mx = -INFINITY;
            for (int k = lane; k < bins; k += 32) mx = fmaxf(mx, vlog[s][k]);
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            float se = 0.0f, sc = 0.0f;
            const float step = bins > 1 ? 2.0f / (float)(bins - 1) : 0.0f;
            for (int k = lane; k < bins; k += 32) {
                const float e = expf(vlog[s][k] - mx);
                se += e; sc += e * (-1.0f + step * (float)k);
                if (P.value_logits) P.value_logits[(base + s) * bins + k] = vlog[s][k];
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                se += __shfl_xor_sync(0xffffffffu, se, off);
                sc += __shfl_xor_sync(0xffffffffu, sc, off);
            }
            if (lane == 0 && P.values) P.values[base + s] = sc / se;
        }
        __syncthreads();
        // 5. priors = softmax of the combined logits over the legal actions of the packed state (warp per state)
        if (P.priors && P.states) {
            for (int s = warp; s < ns; s += kHeadsThreads / 32) {
                const int64_t i = base + s;
                lz::State<int> st;
                lz::Packed pk;
                const ulonglong2* sp = reinterpret_cast<const ulonglong2*>(P.states + 4 * i);
                const ulonglong2 a = sp[0], b = sp[1];
                pk.w[0] = a.x; pk.w[1] = a.y; pk.w[2] = b.x; pk.w[3] = b.y;
                lz::unpack(pk, st);
                lz::Legal L;
                lz::legal_actions<int, true>(st, L, true);
                float logit[7], mx = -INFINITY;
#pragma unroll
                for (int k = 0; k < 7; ++k) {
                    const int ac = lane + 32 * k;
                    float v = -INFINITY;
                    if (ac < lz::kActionDim && lz::legal_test(L, ac)) {
                        if (ac < 36) v = lp[s][0][ac];
                        else if (ac < 180) {
                            const int from = (ac - 36) >> 2, d = (ac - 36) & 3;
                            v = lp[s][1][from] + lp[s][0][from + (d == 0 ? -6 : d == 1 ? 6 : d == 2 ? -1 : 1)];
                        } else if (ac < 216) v = lp[s][2][ac - 180];
                        else v = 0.0f;
                    }
                    logit[k] = v; mx = fmaxf(mx, v);
                }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
                const bool ok = mx > -INFINITY && mx < INFINITY;
                float e[7], sum = 0.0f;
#pragma unroll
                for (int k = 0; k < 7; ++k) { e[k] = (ok && logit[k] > -INFINITY) ? expf(logit[k] - mx) : 0.0f; sum += e[k]; }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
#pragma unroll
                for (int k = 0; k < 7; ++k) {
                    const int ac = lane + 32 * k;
                    if (ac < lz::kActionDim) P.priors[i * lz::kActionDim + ac] = ok ? e[k] / sum : 0.0f;
                }
            }
        }
    }
}

}  // namespace
}  // namespace lzb

extern "C" int lzb_heads_tail(const void* pv, int64_t n, int32_t pc, int32_t vc, int32_t mlp, int32_t bins,
                              const float* wgl_t, const float* bn2_scale, const float* bn2_shift, const float* wout,
                              const float* wfc1_t, const float* bfc1, const float* wfc2_t, const float* bfc2,
                              const uint64_t* states, float* priors, float* values, float* log_heads,
                              float* value_logits, void* stream) {
    LZB_REQUIRE(n >= 0, "bad batch");
    LZB_REQUIRE(pc >= 1 && pc <= lzb::kMaxHeadCh && vc >= 1 && vc <= lzb::kMaxHeadCh, "head channels must be in [1, 64]");
    LZB_REQUIRE(mlp >= 1 && mlp <= lzb::kMaxMlp && bins >= 2 && bins <= lzb::kMaxBins, "value MLP / bins too large");
    if (n == 0) return LZB_OK;
    LZB_REQUIRE(pv && wgl_t && bn2_scale && bn2_shift && wout && wfc1_t && bfc1 && wfc2_t && bfc2, "null weights");
    LZB_REQUIRE(!priors || states, "priors need the packed states");
    LZB_REQUIRE((pc + vc) % 8 == 0 && (reinterpret_cast<uintptr_t>(pv) & 15) == 0, "pv: channel count a multiple of 8, 16-byte aligned");
    lzb::HeadsParams P;
    P.pv = reinterpret_cast<const __nv_bfloat16*>(pv); P.n = n; P.pc = pc; P.vc = vc; P.mlp = mlp; P.bins = bins;
    P.wgl_t = wgl_t; P.bn2_scale = bn2_scale; P.bn2_shift = bn2_shift; P.wout = wout; P.wfc1_t = wfc1_t; P.bfc1 = bfc1;
    P.wfc2_t = wfc2_t; P.bfc2 = bfc2; P.states = states; P.priors = priors; P.values = values;
    P.log_heads = log_heads; P.value_logits = value_logits;
    const int64_t tiles = (n + lzb::kTile - 1) / lzb::kTile;
    const int64_t blocks = tiles < (int64_t)lzb::kNumSMs * 4 ? tiles : (int64_t)lzb::kNumSMs * 4;
    lzb::heads_tail_kernel<<<(int)blocks, lzb::kHeadsThreads, 0, (cudaStream_t)stream>>>(P);
    return lzb::check_launch("heads_tail_kernel");
}
