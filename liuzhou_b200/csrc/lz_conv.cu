// lz_conv.cu -- the network's 3x3 / 1x1 convolutions as hand-written tcgen05 implicit GEMMs (sm_100a) with the
// whole pre-activation-ResNet epilogue fused in (replaces cuDNN conv + our bn_relu pass; src/neural_network.py:83-96).
// The fused trunk kernel (lz_trunk.cu) runs a net of up to 10 blocks in one launch; this per-layer path runs deeper nets.
//
// One launch = one convolution layer over the whole wave batch:
//     D[rows = n*36, 128] = sum over taps (ky,kx) of  A_tap[rows, Cin] * W_tap[Cin, 128]        (bf16 x bf16 -> fp32)
// * A operand: all taps are served from shared-memory-resident padded boards.  A CTA tile is 3 WHOLE boards kept in a
//   padded row space,
//       row(b, y, x) = b * 42 + (y + 1) * 6 + x,     y = -1 .. 5   (y = -1: a zero row above every board),
//   and a tap (dy, dx) is an MMA whose A descriptor simply STARTS 6 * (dy + 1) rows into that buffer: the tensor core
//   applies the 128-byte swizzle on absolute shared-memory address bits, so a descriptor may start on any 128-byte row
//   (measured, tools/probe/umma_shift_probe.cu: base_offset = 0 works for every row shift).  The x shift cannot share
//   rows (no pad column: that would cost 1/7 of the MMA rows again), so there is one copy per dx, each written by ONE
//   tiled TMA load whose box starts at x = dx, y = -1: the out-of-bounds column / row arrive as zeros.  A tile therefore
//   loads 3 copies instead of 9 taps (83 KB instead of 288 KB of real bytes per CTA), the rows b * 42 + 36 .. 41 of the
//   accumulator are junk (the price: 108 useful rows of 128), rows 126 .. 135 of every copy are a zero block written once.
//   The three dx copies are the A pipeline stages (the producer runs one tile ahead).
// * B operand: a ring of weight stages (one tap each); a CTA pair (cta_group::2, cluster of 2) splits Cout, so each CTA
//   loads its 64-cout half of every tap.
// * MMA: tcgen05.mma.cta_group::2.kind::f16, M = 256 (128 rows per CTA), N = 128, K = 16; fp32 accumulators in
//   TMEM, double buffered (2 x 128 columns) so the epilogue of tile i overlaps the MMAs of tile i+1.
// * Persistent: up to 74 clusters walk the pair tiles round-robin.  Warp roles per CTA: warp 0 = TMA producer,
//   warp 1 = TMEM allocator + (leader CTA) MMA issuer, warps 2-9 = epilogue (TMEM lane quarter x column half).
// * Epilogue (per row, fp32): v = acc + bias[c] (+ residual[row][c]); optional ReLU; out1 = bf16(v);
//   out2 = bf16(relu(scale[c] * float(out1) + shift[c])).  With BatchNorm folded this covers
//       conv1 of a block : out1 = relu(bn2(conv1(a)))                      (bias, relu)
//       conv2 of a block : out1 = x + conv2(h) ; out2 = relu(bn1_next(out1)) (residual, both outputs)
//       stem             : out1 = relu(stem_bn(conv(x))) ; out2 = relu(bn1_0(out1)).
// Algorithmic work per launch (C = 128): 2 * rows * 128 * 1152 FLOP; bytes: rows * 256 B read + rows * 256 B per
// output (+ residual).
#include <cuda.h>
#include <cuda_bf16.h>

#include "lz_common.cuh"
#include "lz_tc.cuh"

namespace lzb {
namespace {
using namespace tc;

constexpr int kConvThreads = 320;                // warp 0 producer, warp 1 MMA, warps 2-9 epilogue
constexpr int kCout = 128;
constexpr int kKC = 64;                          // channels per 128 B swizzle row
constexpr uint32_t kWSlotBytes = (kCout / 2) * kKC * 2;   // 8 KB: 64 couts (this CTA's half) x 64 cin
constexpr int kAccStages = 2;
constexpr uint32_t kTmemCols = kAccStages * kCout;        // 256 fp32 columns

struct ConvParams {
    const float* bias;                 // [128] or null
    const __nv_bfloat16* residual;     // [rows,128] or null
    const float* scale;                // [128] (out2) or null
    const float* shift;
    __nv_bfloat16* out1;               // [rows,128] or null
    __nv_bfloat16* out2;               // [rows,128] or null
    int relu1;
    int images;                        // n
};

constexpr int kBoards = 3;                               // boards per CTA tile
constexpr int kBoardRows = 42;                           // padded rows per board
constexpr int kBoxRows = kBoards * kBoardRows;           // 126 rows written by one TMA box
constexpr int kBufRows = 136;                            // rows per chunk buffer: 126 loaded + 6 zero + 4 spare
constexpr uint32_t kPChunkBytes = kBufRows * 128;        // 17,408 B = 17 x 1024
constexpr uint32_t kPBoxBytes = kBoxRows * 128;          // 16,128 B per TMA load
constexpr int kWStages = 4;

template <int TAPS, int KCH>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kConvThreads, 1)
conv_pad_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, const ConvParams P) {
    constexpr int NDX = TAPS == 9 ? 3 : 1, NDY = TAPS == 9 ? 3 : 1;
    constexpr uint32_t kACopyBytes = KCH * kPChunkBytes;          // one dx copy: 34,816 B (KCH = 2)
    constexpr uint32_t kWStageBytes = KCH * kWSlotBytes;          // one tap's weights (this CTA's half of Cout): 16 KB
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t a_smem = base;
    const uint32_t w_smem = a_smem + NDX * kACopyBytes;
    const uint32_t bar0 = w_smem + kWStages * kWStageBytes;
    const uint32_t afull_bar = bar0;                              // [NDX]      leader: copy landed (both CTAs' bytes)
    const uint32_t aempty_bar = afull_bar + 8 * NDX;              // [NDX]      both  : the MMAs that read the copy are done
    const uint32_t wfull_bar = aempty_bar + 8 * NDX;              // [kWStages] leader
    const uint32_t wempty_bar = wfull_bar + 8 * kWStages;         // [kWStages] both
    const uint32_t tfull_bar = wempty_bar + 8 * kWStages;         // [kAccStages] both
    const uint32_t tempty_bar = tfull_bar + 8 * kAccStages;       // [kAccStages] leader
    const uint32_t tmem_slot = tempty_bar + 8 * kAccStages;
    const uint32_t vec_smem = (tmem_slot + 16 + 15u) & ~15u;
    const uint32_t stage_smem = vec_smem + 3 * kCout * 4;
    uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
    float* vec = reinterpret_cast<float*>(gen + (vec_smem - base));
    volatile uint32_t* tmem_slot_p = reinterpret_cast<volatile uint32_t*>(gen + (tmem_slot - base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
    const int64_t pair_tiles = (P.images + 2 * kBoards - 1) / (2 * kBoards);

    if (threadIdx.x == 0) {
        prefetch_tmap(&tmA);
        prefetch_tmap(&tmW);
        for (int i = 0; i < NDX; ++i) { mbar_init(afull_bar + 8 * i, 1); mbar_init(aempty_bar + 8 * i, 1); }
        for (int i = 0; i < kWStages; ++i) { mbar_init(wfull_bar + 8 * i, 1); mbar_init(wempty_bar + 8 * i, 1); }
        for (int i = 0; i < kAccStages; ++i) { mbar_init(tfull_bar + 8 * i, 1); mbar_init(tempty_bar + 8 * i, 16); }
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    for (int i = threadIdx.x; i < kCout; i += kConvThreads) {
        vec[i] = P.bias ? P.bias[i] : 0.0f;
        vec[kCout + i] = P.scale ? P.scale[i] : 1.0f;
        vec[2 * kCout + i] = P.shift ? P.shift[i] : 0.0f;
    }
    // the zero block below the last board of every chunk buffer (rows 126 .. 135): written once, never touched by TMA
    {
        constexpr int kZero16 = (kBufRows - kBoxRows) * 128 / 16;           // 80 x 16 B per chunk buffer
        for (int i = threadIdx.x; i < NDX * KCH * kZero16; i += kConvThreads) {
            const int buf = i / kZero16, off = i - buf * kZero16;
            *reinterpret_cast<uint4*>(gen + (a_smem - base) + buf * kPChunkBytes + kPBoxBytes + off * 16) = make_uint4(0u, 0u, 0u, 0u);
        }
    }
    fence_proxy_async();           // generic-proxy writes (the zero blocks) -> visible to the tensor core's async proxy
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_p;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");

    if (warp == 0) {
        // ===================== TMA producer (both CTAs) =====================
        const uint32_t afull_leader = mapa_rank(afull_bar, 0), wfull_leader = mapa_rank(wfull_bar, 0);
        uint32_t wst = 0, wph = 0, aph = 0;
        for (int64_t pt = cluster_id; pt < pair_tiles; pt += num_clusters) {
            const int board0 = (int)(2 * pt + rank) * kBoards;
#pragma unroll
            for (int dxi = 0; dxi < NDX; ++dxi) {
                mbar_wait(aempty_bar + 8 * dxi, aph ^ 1);
                if (elect_one()) {
                    if (leader) mbar_arrive_expect_tx(afull_bar + 8 * dxi, 2 * KCH * kPBoxBytes);
#pragma unroll
                    for (int kc = 0; kc < KCH; ++kc)     // box (64 ch, 6 x, 7 y, 3 boards) at x = dx, y = -1: zeros outside
                        tma_tile4d_2sm(a_smem + dxi * kACopyBytes + kc * kPChunkBytes, &tmA, afull_leader + 8 * dxi,
                                       kc * kKC, TAPS == 9 ? dxi - 1 : 0, -1, board0);
                }
                __syncwarp();
#pragma unroll
                for (int dyi = 0; dyi < NDY; ++dyi) {
                    const int tap = TAPS == 9 ? dyi * 3 + dxi : 0;
                    mbar_wait(wempty_bar + 8 * wst, wph ^ 1);
                    if (elect_one()) {
                        if (leader) mbar_arrive_expect_tx(wfull_bar + 8 * wst, 2 * kWStageBytes);
#pragma unroll
                        for (int kc = 0; kc < KCH; ++kc)
                            tma_tile2d_2sm(w_smem + wst * kWStageBytes + kc * kWSlotBytes, &tmW, wfull_leader + 8 * wst,
                                           kc * kKC, tap * kCout + (int)rank * (kCout / 2));
                    }
                    __syncwarp();
                    if (++wst == kWStages) { wst = 0; wph ^= 1; }
                }
            }
            aph ^= 1;
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA) =====================
        if (leader) {
            uint32_t wst = 0, wph = 0, aph = 0, acc = 0, acc_phase = 0;
            for (int64_t pt = cluster_id; pt < pair_tiles; pt += num_clusters) {
                mbar_wait(tempty_bar + 8 * acc, acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * kCout;
#pragma unroll
                for (int dxi = 0; dxi < NDX; ++dxi) {
                    mbar_wait(afull_bar + 8 * dxi, aph);
                    tc_fence_after();
#pragma unroll
                    for (int dyi = 0; dyi < NDY; ++dyi) {
                        mbar_wait(wfull_bar + 8 * wst, wph);
                        tc_fence_after();
                        if (elect_one()) {
                            // tap (dy, dx): rows [6 (dy + 1), 6 (dy + 1) + 128) of copy dx  (1x1: dy = 0)
                            const uint32_t shift = (uint32_t)(TAPS == 9 ? dyi * 6 : 6) * 128u;
#pragma unroll
                            for (int kc = 0; kc < KCH; ++kc) {
                                const uint64_t adesc = umma_desc_sw128(a_smem + dxi * kACopyBytes + kc * kPChunkBytes + shift);
                                const uint64_t bdesc = umma_desc_sw128(w_smem + wst * kWStageBytes + kc * kWSlotBytes);
#pragma unroll
                                for (int k = 0; k < kKC / 16; ++k)
                                    umma_2sm(d_tmem, adesc + 2 * k, bdesc + 2 * k, (uint32_t)((dxi | dyi | kc | k) != 0));
                            }
                            umma_commit_2sm(wempty_bar + 8 * wst, 3);
                            if (dyi == NDY - 1) umma_commit_2sm(aempty_bar + 8 * dxi, 3);      // the copy is free in both CTAs
                            if (dyi == NDY - 1 && dxi == NDX - 1) umma_commit_2sm(tfull_bar + 8 * acc, 3);
                        }
                        __syncwarp();
                        if (++wst == kWStages) { wst = 0; wph ^= 1; }
                    }
                }
                aph ^= 1;
                if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===================== epilogue: warps 2..9 =====================
        // TMEM lane quarter = warp % 4 (hardware rule), column half = (warp - 2) / 4: each warp owns 32 rows x 64
        // channels of the tile.  Per 32-column chunk: TMEM -> registers (lane = row) -> fp32 staging tile in shared
        // memory (XOR-swizzled 16 B slots, conflict-free both ways) -> re-read so that 4 consecutive lanes own 32
        // consecutive channels of one row: residual loads and both output stores are then full 32 B sectors,
        // 8 rows per instruction.  The residual is prefetched into registers BEFORE waiting for the accumulator.
        // Accumulator row i = b * 42 + y * 6 + x of the tile <-> global pixel row (board0 + b) * 36 + y * 6 + x,
        // rows with i % 42 >= 36 (the pad row between boards), i >= 126 or a board beyond the batch are junk: skipped
        const int q = warp & 3, half = (warp - 2) >> 2;
        const uint32_t tempty_leader = mapa_rank(tempty_bar, 0);
        uint32_t acc = 0, acc_phase = 0;
        float4* stg = reinterpret_cast<float4*>(gen + (stage_smem - base)) + (warp - 2) * (32 * 8);
        const int sub = lane & 3, rsub = lane >> 2;
        const bool relu1 = P.relu1 != 0;
        int rem4[4], b4[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int i = q * 32 + rsub + 8 * k;
            b4[k] = i / kBoardRows;
            rem4[k] = i - b4[k] * kBoardRows;
        }
        for (int64_t pt = cluster_id; pt < pair_tiles; pt += num_clusters) {
            const int board0 = (int)(2 * pt + rank) * kBoards;
            int64_t goff[4];                                 // global row of this lane's 4 rows, or -1
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const bool ok = b4[k] < kBoards && rem4[k] < 36 && board0 + b4[k] < P.images;
                goff[k] = ok ? (int64_t)(board0 + b4[k]) * 36 + rem4[k] : -1;
            }
            uint4 resv[2][4];
            if (P.residual) {
#pragma unroll
                for (int jj = 0; jj < 2; ++jj)
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        resv[jj][k] = goff[k] >= 0 ? __ldg(reinterpret_cast<const uint4*>(P.residual) +
                                                          ((goff[k] * kCout + half * 64 + jj * 32 + sub * 8) >> 3))
                                                   : make_uint4(0u, 0u, 0u, 0u);
            }
            mbar_wait(tfull_bar + 8 * acc, acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * kCout + half * 64;
            uint32_t v[2][32];
            tmem_ld32(taddr, v[0]);
            tmem_ld32(taddr + 32, v[1]);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(tempty_leader + 8 * acc);
            if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) {
                const int c0 = half * 64 + jj * 32 + sub * 8;
                const float4 b0 = *reinterpret_cast<const float4*>(vec + c0), b1 = *reinterpret_cast<const float4*>(vec + c0 + 4);
                const float4 s0 = *reinterpret_cast<const float4*>(vec + kCout + c0), s1 = *reinterpret_cast<const float4*>(vec + kCout + c0 + 4);
                const float4 t0 = *reinterpret_cast<const float4*>(vec + 2 * kCout + c0), t1 = *reinterpret_cast<const float4*>(vec + 2 * kCout + c0 + 4);
                const float2 bias2[4] = {make_float2(b0.x, b0.y), make_float2(b0.z, b0.w), make_float2(b1.x, b1.y), make_float2(b1.z, b1.w)};
                const float2 scale2[4] = {make_float2(s0.x, s0.y), make_float2(s0.z, s0.w), make_float2(s1.x, s1.y), make_float2(s1.z, s1.w)};
                const float2 shift2[4] = {make_float2(t0.x, t0.y), make_float2(t0.z, t0.w), make_float2(t1.x, t1.y), make_float2(t1.z, t1.w)};
                __syncwarp();
#pragma unroll
                for (int f = 0; f < 8; ++f)
                    stg[lane * 8 + (f ^ (lane & 7))] = make_float4(__uint_as_float(v[jj][4 * f]), __uint_as_float(v[jj][4 * f + 1]),
                                                                   __uint_as_float(v[jj][4 * f + 2]), __uint_as_float(v[jj][4 * f + 3]));
                __syncwarp();
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (goff[k] < 0) continue;
                    const int r = rsub + 8 * k;
                    const float4 x0 = stg[r * 8 + ((2 * sub) ^ (r & 7))], x1 = stg[r * 8 + ((2 * sub + 1) ^ (r & 7))];
                    float2 x[4] = {make_float2(x0.x, x0.y), make_float2(x0.z, x0.w), make_float2(x1.x, x1.y), make_float2(x1.z, x1.w)};
                    const int64_t off = (goff[k] * kCout + c0) >> 3;
                    if (P.residual) {
                        const uint32_t* rw = reinterpret_cast<const uint32_t*>(&resv[jj][k]);
#pragma unroll
                        for (int h = 0; h < 4; ++h)
                            x[h] = __fadd2_rn(x[h], make_float2(__uint_as_float(rw[h] << 16), __uint_as_float(rw[h] & 0xffff0000u)));
                    }
                    uint32_t p1[4], p2[4];
#pragma unroll
                    for (int h = 0; h < 4; ++h) {
                        float2 f = __fadd2_rn(x[h], bias2[h]);
                        if (relu1) { f.x = fmaxf(f.x, 0.0f); f.y = fmaxf(f.y, 0.0f); }
                        p1[h] = pack_bf16(f.x, f.y);
                        const float2 sv = make_float2(__uint_as_float(p1[h] << 16), __uint_as_float(p1[h] & 0xffff0000u));
                        const float2 g = __ffma2_rn(scale2[h], sv, shift2[h]);
                        p2[h] = pack_bf16(fmaxf(g.x, 0.0f), fmaxf(g.y, 0.0f));
                    }
                    if (P.out1) reinterpret_cast<uint4*>(P.out1)[off] = make_uint4(p1[0], p1[1], p1[2], p1[3]);
                    if (P.out2) reinterpret_cast<uint4*>(P.out2)[off] = make_uint4(p2[0], p2[1], p2[2], p2[3]);
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

// ---- host side ----------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
bool driver_entry(const char* name, void** fn) {
    cudaDriverEntryPointQueryResult st;
    return cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &st) == cudaSuccess && st == cudaDriverEntryPointSuccess &&
           *fn != nullptr;
}

template <int TAPS, int KCH>
int launch_conv_pad(const void* x, const void* w, const ConvParams& P, cudaStream_t stream) {
    static EncodeTiledFn encode_tiled = nullptr;
    if (!encode_tiled && !driver_entry("cuTensorMapEncodeTiled", reinterpret_cast<void**>(&encode_tiled))) {
        set_error("lzb_conv: cuTensorMapEncodeTiled unavailable");
        return LZB_ERR_CUDA;
    }
    constexpr int cin = KCH * kKC;
    alignas(64) CUtensorMap tmA, tmW;
    {   // activations (C, W, H, N) bf16 NHWC; box = 64 channels x 6 x 7 x 3 boards: one padded copy of a CTA tile
        const cuuint64_t dim[4] = {(cuuint64_t)cin, 6, 6, (cuuint64_t)P.images};
        const cuuint64_t stride[3] = {(cuuint64_t)cin * 2, (cuuint64_t)cin * 2 * 6, (cuuint64_t)cin * 2 * 36};
        const cuuint32_t box[4] = {kKC, 6, 7, kBoards};
        const cuuint32_t estr[4] = {1, 1, 1, 1};
        const CUresult rc = encode_tiled(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x), dim, stride, box, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (rc != CUDA_SUCCESS) { set_error("lzb_conv: cuTensorMapEncodeTiled (activations) failed (%d)", (int)rc); return LZB_ERR_CUDA; }
    }
    {   // weights: [tap * 128 + cout][cin] bf16
        const cuuint64_t dim[2] = {(cuuint64_t)cin, (cuuint64_t)TAPS * kCout};
        const cuuint64_t stride[1] = {(cuuint64_t)cin * 2};
        const cuuint32_t box[2] = {kKC, kCout / 2};
        const cuuint32_t estr[2] = {1, 1};
        const CUresult rc = encode_tiled(&tmW, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(w), dim, stride, box, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (rc != CUDA_SUCCESS) { set_error("lzb_conv: cuTensorMapEncodeTiled (weights) failed (%d)", (int)rc); return LZB_ERR_CUDA; }
    }
    constexpr int NDX = TAPS == 9 ? 3 : 1;
    constexpr size_t smem = 1024 + (size_t)NDX * KCH * kPChunkBytes + (size_t)kWStages * KCH * kWSlotBytes +
                            8 * (2 * NDX + 2 * kWStages + 2 * kAccStages) + 32 + 3 * kCout * sizeof(float) + 8 * 32 * 128 + 512;
    static int sm_count[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { set_error("lzb_conv: bad current device"); return LZB_ERR_CUDA; }
    if (sm_count[dev] == 0) {
        if (cudaFuncSetAttribute(conv_pad_kernel<TAPS, KCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            set_error("lzb_conv: cannot raise dynamic shared memory to %zu", smem);
            return LZB_ERR_CUDA;
        }
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 2) n = kNumSMs;
        sm_count[dev] = n;
    }
    const int64_t pair_tiles = (P.images + 2 * kBoards - 1) / (2 * kBoards);
    const int clusters = (int)(pair_tiles < sm_count[dev] / 2 ? pair_tiles : sm_count[dev] / 2);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * clusters);
    cfg.blockDim = dim3(kConvThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, conv_pad_kernel<TAPS, KCH>, tmA, tmW, P) != cudaSuccess) return check_launch("conv_pad_kernel");
    return check_launch("conv_pad_kernel");
}

}  // namespace
}  // namespace lzb

// x bf16 [n,6,6,cin] (NHWC), w bf16 [taps][128][cin], outputs bf16 [n,6,6,128]; n must be a multiple of 64.
extern "C" int lzb_conv_bf16(const void* x, const void* w, int64_t n, int32_t cin, int32_t taps, const float* bias,
                             const void* residual, const float* scale, const float* shift, int32_t relu1, void* out1,
                             void* out2, void* stream) {
    LZB_REQUIRE(n > 0 && n % 64 == 0, "batch must be a positive multiple of 64 (256-row tile pairs)");
    LZB_REQUIRE((cin == 128 && (taps == 9 || taps == 1)) || (cin == 64 && taps == 9),
                "supported: cin = 128 with taps = 9 (3x3, pad 1) or 1 (1x1); cin = 64 with taps = 9");
    LZB_REQUIRE(x && w && (out1 || out2), "null pointer");
    LZB_REQUIRE(!out2 || (scale && shift), "out2 needs scale / shift");
    LZB_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(residual) |
                  reinterpret_cast<uintptr_t>(out1) | reinterpret_cast<uintptr_t>(out2)) & 15) == 0, "pointers must be 16-byte aligned");
    lzb::ConvParams P;
    P.bias = bias; P.residual = reinterpret_cast<const __nv_bfloat16*>(residual); P.scale = scale; P.shift = shift;
    P.out1 = reinterpret_cast<__nv_bfloat16*>(out1); P.out2 = reinterpret_cast<__nv_bfloat16*>(out2);
    P.relu1 = relu1; P.images = (int)n;
    if (cin == 64) return lzb::launch_conv_pad<9, 1>(x, w, P, (cudaStream_t)stream);
    if (taps == 9) return lzb::launch_conv_pad<9, 2>(x, w, P, (cudaStream_t)stream);
    return lzb::launch_conv_pad<1, 2>(x, w, P, (cudaStream_t)stream);
}
