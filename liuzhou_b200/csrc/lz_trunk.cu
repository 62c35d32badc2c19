// lz_trunk.cu -- the WHOLE convolutional trunk of ChessNet (stem conv + 2 x blocks 3x3 convs + the heads' 1x1 conv,
// src/neural_network.py:83-96,213-259) as ONE persistent tcgen05 kernel: activations never leave the SM.
//
// Why this is possible: a convolution only mixes pixels of the same board, and a CTA tile here is 3 WHOLE boards (6 per
// CTA pair), so layer l + 1 of a tile depends on nothing but layer l of the same tile -- no grid-wide synchronisation
// between layers.  The per-layer kernels (lz_conv.cu) spend more time moving activations (L2 -> SM operand loads, the
// epilogue's global stores / residual loads, DRAM spill of the 113 MB working set) than in the tensor core
// (profiles/r02_conv_decompose_*.txt, profiles/r02_conv_pad_ncu_full.csv); here a tile's activations stay in shared
// memory / TMEM through all 22 layers and only the weights stream (L2-resident, 5.9 MB for the whole net).
//
// Data flow of one tile (CTA pair, cta_group::2: M = 256 = 2 x 128 accumulator rows, N = 128, K = 16 per MMA):
//   * A operand = the previous layer's activations as bf16 "padded boards" in shared memory: row(b, y, x) = b * 42 +
//     (y + 1) * 6 + x (a zero row above every board), three copies pre-shifted in x (dx = -1, 0, +1, zero column where
//     the neighbour is off the board); a tap (dy, dx) is an MMA whose A descriptor starts 6 (dy + 1) rows into copy dx
//     (the tensor core swizzles on absolute address bits, so a descriptor may start on any 128-byte row:
//     tools/probe/umma_shift_probe.cu).  The stem's copies come from global memory by TMA (zeros out of bounds); every
//     other layer's copies are written by the epilogue of the layer before it.
//   * accumulators in TMEM: acc_h (stem, conv1, heads conv) and acc_x = the RESIDUAL STREAM in fp32: conv2's MMAs
//     accumulate straight onto it (x' = x + conv2(h) is done by the tensor core, never rounded to bf16).
//   * epilogue warps (8): TMEM -> registers -> bias / BatchNorm / ReLU -> bf16 -> the three shifted copies in shared
//     memory (swizzled 16-byte stores), 64 channels at a time: the next layer's MMAs on channels 0-63 start while the
//     epilogue still produces channels 64-127 (K-chunk pipelining).
//   * weights: one tap (this CTA's 64 couts x 128 cin, 16 KB) per pipeline stage, streamed by TMA through a kWStages
//     ring across layer and tile boundaries.
// Per layer and tile: 72 MMAs (36 for the stem, 8 for the 1x1 heads conv); junk accumulator rows (the pad row between
// boards, 20 of 128) are the price of serving all taps from one resident tile.
#include <cuda.h>

#include "lz_common.cuh"
#include "lz_tc.cuh"

namespace lzb {
namespace {
using namespace tc;

constexpr int kTrunkThreads = 320;                     // warp 0 producer, warp 1 MMA, warps 2-9 epilogue
constexpr int kBoards = 3;                             // boards per CTA tile
constexpr int kBoardRows = 42;                         // padded rows per board
constexpr int kBoxRows = kBoards * kBoardRows;         // 126
constexpr int kBufRows = 136;                          // rows per chunk buffer (126 + 6 zero + 4 spare)
constexpr uint32_t kChunkBytes = kBufRows * 128;       // 17,408: [rows][64 ch] bf16, SWIZZLE_128B
constexpr uint32_t kBoxBytes = kBoxRows * 128;         // 16,128 per TMA box
constexpr uint32_t kCopyBytes = 2 * kChunkBytes;       // one dx copy, 128 channels
constexpr int kCopyBufs = 4;                           // ring of copy buffers shared by the two tiles in flight
constexpr uint32_t kWStageBytes = 2 * 64 * 64 * 2;     // 16 KB: one tap, this CTA's 64 couts x 128 cin (two 64-channel slices)
constexpr int kWStages = 5;
constexpr uint32_t kAccH = 0, kAccX = 128;             // TMEM column offsets inside a slot's 256 columns
constexpr uint32_t kTrunkTmemCols = 512;               // 2 slots x (acc_h + acc_x)

struct TrunkParams {
    __nv_bfloat16* out;        // [images * 36][128] : relu(heads conv + bias), the input of heads_tail_kernel
    int images;
    int blocks;                // residual blocks; layers = 2 * blocks + 2
};

// Per-layer epilogue parameters in CONSTANT memory (warp-uniform reads through the constant cache: no shared-memory
// traffic -- thread-side shared-memory accesses are starved while the tensor core streams its operands).  Compact layout:
// stem: bias | scale | shift (384); conv1 of block i: bias (128); conv2 of block i: scale | shift (256); heads: bias (128).
constexpr int kMaxBlocks = 10;
constexpr int kTableFloats = 384 + kMaxBlocks * (128 + 256) + 128;      // 4,352 floats = 17 KB
__constant__ float c_trunk_table[kTableFloats];      // refreshed from device memory in stream order before every launch
__host__ __device__ __forceinline__ int table_offset(int l, int layers) {   // first float of layer l
    if (l == 0) return 0;
    if (l == layers - 1) return 384 + (layers - 2) / 2 * 384;
    const int i = (l - 1) >> 1;
    return 384 + i * 384 + ((l & 1) ? 0 : 128);
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void mbar_arrive_n(uint32_t bar, uint32_t n) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(n) : "memory");
}

// Job order of a cluster: its pair tiles k = 0 .. ntiles-1 are taken two at a time (slots 0 / 1); a round runs
// layer 0 of slot 0, layer 0 of slot 1, layer 1 of slot 0, ...: while the tensor core works on one slot, the epilogue
// warps turn the other slot's accumulator into its next operand.  Operand copies are numbered in consumption order
// (3 per job, 1 for the 1x1 heads layer) and live in ring buffer number (copy index % 4).
struct Sched {
    int layers;
    __device__ __forceinline__ int ncopies(int l) const { return l == layers - 1 ? 1 : 3; }
    // copies of a round with ns slots that precede job (l, s)
    __device__ __forceinline__ int before(int l, int s, int ns) const {
        return l < layers - 1 ? ns * 3 * l + 3 * s : ns * 3 * (layers - 1) + s;
    }
    __device__ __forceinline__ int round_total(int ns) const { return ns * (3 * (layers - 1) + 1); }
};

// One cluster = one MMA pair (2 CTAs, set at launch); rank 0 is the pair's leader.
__global__ void __launch_bounds__(kTrunkThreads, 1)
trunk_kernel(const __grid_constant__ CUtensorMap tmIn, const __grid_constant__ CUtensorMap tmW0,
             const __grid_constant__ CUtensorMap tmW1, const TrunkParams P) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t a_smem = base;                                    // kCopyBufs copy buffers x 2 chunks
    const uint32_t w_smem = a_smem + kCopyBufs * kCopyBytes;         // weight ring
    const uint32_t bar0 = w_smem + kWStages * kWStageBytes;
    const uint32_t full_bar = bar0;                                  // [4] leader: copy buffer written (16 arrivals, or TMA)
    const uint32_t empty_bar = full_bar + 8 * kCopyBufs;             // [4] both  : the MMAs that read the buffer are done
    const uint32_t wfull_bar = empty_bar + 8 * kCopyBufs;            // [kWStages] leader
    const uint32_t wempty_bar = wfull_bar + 8 * kWStages;            // [kWStages] both
    const uint32_t accfull_bar = wempty_bar + 8 * kWStages;          // [2] both  : a slot's accumulator is complete
    const uint32_t epidone_bar = accfull_bar + 16;                   // [2] leader: a slot's last accumulator drained (16 arrivals)
    const uint32_t tmem_slot = epidone_bar + 16;
    uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
    volatile uint32_t* tmem_slot_p = reinterpret_cast<volatile uint32_t*>(gen + (tmem_slot - base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Copy hand-off epilogue -> MMA thread.  The operand copies are written with st.shared by the CTA whose OWN tensor
    // core reads them (cta_group::2: every CTA's A rows come from its own shared memory), so what has to hold is that the
    // stores were performed and fenced into the async proxy before the arrive leaves the SM: fence.proxy.async +
    // an arrive with the default (release, CTA-scope) semantics = MEMBAR.ALL.CTA.  (release.cluster / acquire.cluster
    // would cost MEMBAR.ALL.GPU + CCTL.IVALL: ~1,000 cycles per copy, 3 copies per job.)
    const uint32_t rank = cluster_ctarank();                         // rank in the MMA pair
    const bool leader = rank == 0;
    const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
    const int64_t pair_tiles = (P.images + 2 * kBoards - 1) / (2 * kBoards);
    const int ntiles = (int)((pair_tiles - cluster_id + num_clusters - 1) / num_clusters);
    const int rounds = (ntiles + 1) / 2;
    Sched sch;
    sch.layers = 2 * P.blocks + 2;
    const int layers = sch.layers;
    // Tap order (copy order, and dy order inside a copy) is the same for every cluster: it fixes the fp32 summation
    // order of every board, so a board's result does not depend on where in the batch it sits (compacted and
    // full-batch searches must agree bit for bit).

    if (threadIdx.x == 0) {
        prefetch_tmap(&tmIn); prefetch_tmap(&tmW0); prefetch_tmap(&tmW1);
        for (int i = 0; i < kCopyBufs; ++i) { mbar_init(full_bar + 8 * i, 16); mbar_init(empty_bar + 8 * i, 1); }
        for (int i = 0; i < kWStages; ++i) { mbar_init(wfull_bar + 8 * i, 1); mbar_init(wempty_bar + 8 * i, 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(accfull_bar + 8 * i, 1); mbar_init(epidone_bar + 8 * i, 16); }
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTrunkTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    // the copy buffers start out all zero: pad rows are never written afterwards, pad columns are rewritten with zeros
    for (uint32_t i = threadIdx.x; i < kCopyBufs * kCopyBytes / 16; i += kTrunkThreads)
        *reinterpret_cast<uint4*>(gen + (a_smem - base) + i * 16) = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_p;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");

    if (warp == 0) {
        // ===================== TMA producer (both CTAs): stem input copies + every weight tap, in MMA order =============
        const uint32_t full_leader = mapa_rank(full_bar, 0), wfull_leader = mapa_rank(wfull_bar, 0);
        uint32_t wst = 0, wph = 0;
        int g_round = 0;                                             // copies before this round
        for (int r = 0; r < rounds; ++r) {
            const int ns = ntiles - 2 * r >= 2 ? 2 : 1;
            for (int l = 0; l < layers; ++l) {
                const int taps = l == layers - 1 ? 1 : 9;
                for (int s = 0; s < ns; ++s) {
                    if (l == 0) {                                    // the stem's three copies come from global memory
                        const int64_t pt = cluster_id + (int64_t)(2 * r + s) * num_clusters;
                        const int board0 = (int)(2 * pt + rank) * kBoards;
                        const int g0 = g_round + sch.before(0, s, ns);
                        for (int c = 0; c < 3; ++c) {
                            const int g = g0 + c, buf = g & 3;
                            mbar_wait(empty_bar + 8 * buf, (((uint32_t)g >> 2) & 1u) ^ 1u);
                            if (elect_one()) {
                                if (leader) {                        // 16 arrivals expected: 1 with the byte count + 15 plain
                                    mbar_arrive_expect_tx(full_bar + 8 * buf, 2 * kBoxBytes);
                                    mbar_arrive_n(full_bar + 8 * buf, 15);
                                }
                                tma_tile4d_2sm(a_smem + buf * kCopyBytes, &tmIn, full_leader + 8 * buf, 0, c - 1, -1, board0);
                            }
                            __syncwarp();
                        }
                    }
                    const int tap_base = l == 0 ? 0 : (l - 1) * 9;
                    for (int t = 0; t < taps; ++t) {
                        // MMA order: copy-major, dy-minor; tap index in the weight tensor = (dy + 1) * 3 + (dx + 1)
                        const int tap = taps == 9 ? (t % 3) * 3 + t / 3 : 0;
                        mbar_wait(wempty_bar + 8 * wst, wph ^ 1);
                        if (elect_one()) {
                            const uint32_t dstw = w_smem + wst * kWStageBytes;
                            if (l == 0) {
                                if (leader) mbar_arrive_expect_tx(wfull_bar + 8 * wst, 2 * 8192);
                                tma_tile2d_2sm(dstw, &tmW0, wfull_leader + 8 * wst, 0, tap * 128 + (int)rank * 64);
                            } else {
                                if (leader) mbar_arrive_expect_tx(wfull_bar + 8 * wst, 2 * kWStageBytes);
                                tma_tile2d_2sm(dstw, &tmW1, wfull_leader + 8 * wst, 0, (tap_base + tap) * 128 + (int)rank * 64);
                                tma_tile2d_2sm(dstw + 8192, &tmW1, wfull_leader + 8 * wst, 64, (tap_base + tap) * 128 + (int)rank * 64);
                            }
                        }
                        __syncwarp();
                        if (++wst == (uint32_t)kWStages) { wst = 0; wph ^= 1; }
                    }
                }
            }
            g_round += sch.round_total(ns);
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA) =====================
        if (leader) {
            uint32_t wst = 0, wph = 0;
            uint32_t acc_tile_ph[2] = {0, 0};
            int g = 0;                                               // next copy to consume
            for (int r = 0; r < rounds; ++r) {
                const int ns = ntiles - 2 * r >= 2 ? 2 : 1;
                for (int l = 0; l < layers; ++l) {
                    const int kch = l == 0 ? 1 : 2;
                    const bool conv2 = l >= 2 && l < layers - 1 && (l & 1) == 0;     // accumulates onto the residual stream
                    for (int s = 0; s < ns; ++s) {
                        if (l == 0) {                                // acc_h of this slot's previous tile has been drained
                            mbar_wait(epidone_bar + 8 * s, acc_tile_ph[s] ^ 1);
                            acc_tile_ph[s] ^= 1;
                        }
                        const uint32_t d_tmem = tmem_base + (uint32_t)s * 256u + (conv2 ? kAccX : kAccH);
                        const int nc = sch.ncopies(l);
                        for (int c = 0; c < nc; ++c, ++g) {
                            const int buf = g & 3;
                            mbar_wait(full_bar + 8 * buf, ((uint32_t)g >> 2) & 1u);
                            tc_fence_after();
                            for (int d = 0; d < nc; ++d) {            // nc = 3: three dy taps per copy; heads conv: one tap (dy = 0)
                                const int dyi = nc == 3 ? d : 1;
                                mbar_wait(wfull_bar + 8 * wst, wph);
                                tc_fence_after();
                                if (elect_one()) {
                                    const bool first_tap = c == 0 && d == 0;
                                    const bool last_tap = c == nc - 1 && d == nc - 1;
#pragma unroll
                                    for (int kc = 0; kc < 2; ++kc) {
                                        if (kc < kch) {
                                            const uint64_t adesc = umma_desc_sw128(a_smem + buf * kCopyBytes + kc * kChunkBytes +
                                                                                   (uint32_t)(dyi * 6) * 128u);
                                            const uint64_t bdesc = umma_desc_sw128(w_smem + wst * kWStageBytes + kc * 8192);
                                            // the stem's operand has 11 real channels in a 64-channel row: channels 16..63
                                            // are zero in the input AND in the packed weights, so only the first K = 16
                                            // step contributes (9 MMAs instead of 36 for the layer)
#pragma unroll
                                            for (int k = 0; k < 4; ++k)
                                                if (k == 0 || l != 0)
                                                    umma_2sm(d_tmem, adesc + 2 * k, bdesc + 2 * k,
                                                             (uint32_t)(conv2 || !first_tap || (kc | k) != 0));
                                        }
                                    }
                                    umma_commit_2sm(wempty_bar + 8 * wst, 3);                    // both CTAs hold this stage
                                    if (d == nc - 1) umma_commit_2sm(empty_bar + 8 * buf, 3);    // copy consumed
                                    if (last_tap) umma_commit_2sm(accfull_bar + 8 * s, 3);
                                }
                                __syncwarp();
                                if (++wst == (uint32_t)kWStages) { wst = 0; wph ^= 1; }
                            }
                        }
                    }
                }
            }
        }
    } else {
        // ===================== epilogue: warps 2..9 =====================
        // thread <-> accumulator row i = q * 32 + lane (TMEM lane quarter q = warp % 4) and 64 of the 128 columns
        // (col_half = (warp - 2) / 4), handled 32 at a time.  Row i = b * 42 + y * 6 + x; i % 42 >= 36 or b = 3: junk.
        const int q = warp & 3, col_half = (warp - 2) >> 2;
        const int i_row = q * 32 + lane;
        const int b = i_row / kBoardRows, rem = i_row - b * kBoardRows;
        const bool row_ok = b < kBoards && rem < 36;
        const int y = rem / 6, x = rem - y * 6;
        // position of this pixel in copy dx: copy dx holds pixel (y, x' + dx) at (y, x'); the column x' that has no source
        // (its neighbour is off the board) is written with zeros by the thread that wraps onto it
        uint32_t rowoff[3], swz[3];
        bool zero[3];
#pragma unroll
        for (int dxi = 0; dxi < 3; ++dxi) {
            const int xs = x - (dxi - 1);
            zero[dxi] = xs < 0 || xs > 5;
            const int xp = (xs + 6) % 6;
            const int rho = b * kBoardRows + (y + 1) * 6 + xp;
            rowoff[dxi] = (uint32_t)rho * 128u;
            swz[dxi] = (uint32_t)(rho & 7);
        }
        const uint32_t full_leader = mapa_rank(full_bar, 0), epidone_leader = mapa_rank(epidone_bar, 0);
        uint32_t acc_ph[2] = {0, 0};
        int g_round = 0;
        for (int r = 0; r < rounds; ++r) {
            const int ns = ntiles - 2 * r >= 2 ? 2 : 1;
            for (int l = 0; l < layers; ++l) {
                const bool last = l == layers - 1;
                const bool conv2 = l >= 2 && !last && (l & 1) == 0;
                const bool stem = l == 0;
                for (int s = 0; s < ns; ++s) {
                    const float* tp = c_trunk_table + table_offset(l, layers);   // constant bank, warp-uniform addresses
                    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)s * 256u;
                    const uint32_t acc_col = conv2 ? kAccX : kAccH;
                    const int64_t pt = cluster_id + (int64_t)(2 * r + s) * num_clusters;
                    const int board0 = (int)(2 * pt + rank) * kBoards;
                    mbar_wait(accfull_bar + 8 * s, acc_ph[s]);
                    acc_ph[s] ^= 1;
                    tc_fence_after();
                    // 1. the whole accumulator row segment (64 channels) -> registers -> bias / BatchNorm / ReLU -> bf16, ONCE:
                    //    after this the accumulator is dead, so the slot's next MMAs may overwrite it at any time
                    uint32_t pk[2][16];
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        const int c0 = col_half * 64 + hh * 32;        // first of 32 output channels (chunk kc = col_half)
                        uint32_t v[32];
                        tmem_ld32(lane_addr + acc_col + (uint32_t)c0, v);
                        tmem_ld_wait();
                        // stem: bias | scale | shift; conv1 / heads: bias; conv2: scale | shift
                        const float4* vb = reinterpret_cast<const float4*>(tp + c0);
                        const float4* vs = reinterpret_cast<const float4*>(tp + (stem ? 128 : 0) + c0);
                        const float4* vt = reinterpret_cast<const float4*>(tp + (stem ? 256 : 128) + c0);
                        if (stem) {
                            // x0 = relu(conv + bias) -> residual stream (fp32, TMEM); a0 = relu(scale * x0 + shift)
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const float4 bb = vb[j];
                                v[4 * j] = __float_as_uint(fmaxf(__uint_as_float(v[4 * j]) + bb.x, 0.0f));
                                v[4 * j + 1] = __float_as_uint(fmaxf(__uint_as_float(v[4 * j + 1]) + bb.y, 0.0f));
                                v[4 * j + 2] = __float_as_uint(fmaxf(__uint_as_float(v[4 * j + 2]) + bb.z, 0.0f));
                                v[4 * j + 3] = __float_as_uint(fmaxf(__uint_as_float(v[4 * j + 3]) + bb.w, 0.0f));
                            }
                            tmem_st32(lane_addr + kAccX + (uint32_t)c0, v);
                        }
                        if (stem || conv2) {
                            // conv2: the accumulator IS x' = x + conv2(h); a' = relu(scale * x' + shift)
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const float4 ss = vs[j], tt = vt[j];
                                pk[hh][2 * j] = pack_bf16(fmaxf(fmaf(ss.x, __uint_as_float(v[4 * j]), tt.x), 0.0f),
                                                          fmaxf(fmaf(ss.y, __uint_as_float(v[4 * j + 1]), tt.y), 0.0f));
                                pk[hh][2 * j + 1] = pack_bf16(fmaxf(fmaf(ss.z, __uint_as_float(v[4 * j + 2]), tt.z), 0.0f),
                                                              fmaxf(fmaf(ss.w, __uint_as_float(v[4 * j + 3]), tt.w), 0.0f));
                            }
                        } else {
                            // conv1 / heads conv: relu(acc + bias)
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const float4 bb = vb[j];
                                pk[hh][2 * j] = pack_bf16(fmaxf(__uint_as_float(v[4 * j]) + bb.x, 0.0f),
                                                          fmaxf(__uint_as_float(v[4 * j + 1]) + bb.y, 0.0f));
                                pk[hh][2 * j + 1] = pack_bf16(fmaxf(__uint_as_float(v[4 * j + 2]) + bb.z, 0.0f),
                                                              fmaxf(__uint_as_float(v[4 * j + 3]) + bb.w, 0.0f));
                            }
                        }
                    }
                    if (stem) tmem_st_wait();
                    // 2. the operand copies of this slot's NEXT layer, in ring order, as their buffers become free -- or,
                    //    after the last layer, the rows of the output tensor
                    if (last) {
                        if (row_ok && board0 + b < P.images) {
#pragma unroll
                            for (int hh = 0; hh < 2; ++hh) {
                                uint4* o = reinterpret_cast<uint4*>(P.out + ((int64_t)(board0 + b) * 36 + rem) * 128 + col_half * 64 + hh * 32);
#pragma unroll
                                for (int t = 0; t < 4; ++t)
                                    o[t] = make_uint4(pk[hh][4 * t], pk[hh][4 * t + 1], pk[hh][4 * t + 2], pk[hh][4 * t + 3]);
                            }
                        }
                    } else {
                        const int nc = sch.ncopies(l + 1);
                        const int g0 = g_round + sch.before(l + 1, s, ns);
                        for (int c = 0; c < nc; ++c) {
                            const int dxi = nc == 3 ? c : 1;
                            const int g = g0 + c, buf = g & 3;
                            mbar_wait(empty_bar + 8 * buf, (((uint32_t)g >> 2) & 1u) ^ 1u);      // its previous readers are done
                            if (row_ok) {
                                // copy dx index is a loop variable: select this thread's row offset / swizzle / zero flag
                                const uint32_t ro = dxi == 0 ? rowoff[0] : dxi == 1 ? rowoff[1] : rowoff[2];
                                const uint32_t sw = dxi == 0 ? swz[0] : dxi == 1 ? swz[1] : swz[2];
                                const bool zr = dxi == 0 ? zero[0] : dxi == 1 ? zero[1] : zero[2];
                                const uint32_t rowaddr = a_smem + buf * kCopyBytes + (uint32_t)col_half * kChunkBytes + ro;
#pragma unroll
                                for (int hh = 0; hh < 2; ++hh)
#pragma unroll
                                    for (int t = 0; t < 4; ++t) {
                                        const uint32_t c16 = (uint32_t)(hh * 4 + t) ^ sw;
                                        if (zr) st_shared_v4(rowaddr + c16 * 16, 0u, 0u, 0u, 0u);
                                        else st_shared_v4(rowaddr + c16 * 16, pk[hh][4 * t], pk[hh][4 * t + 1], pk[hh][4 * t + 2], pk[hh][4 * t + 3]);
                                    }
                            }
                            fence_proxy_async();          // generic-proxy stores -> visible to the tensor core (async proxy)
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive_remote(full_leader + 8 * buf);
                        }
                    }
                    if (last) {                           // acc_h has been read: this slot's next tile may overwrite it
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_remote(epidone_leader + 8 * s);
                    }
                }
            }
            g_round += sch.round_total(ns);
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTrunkTmemCols) : "memory");
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace
}  // namespace lzb

// planes bf16 [n,6,6,64] (channel-padded input), w_stem bf16 [9][128][64], w_trunk bf16 [2*blocks*9 + 1][128][128]
// (conv1_0, conv2_0, ..., conv2_{blocks-1}, heads 1x1; BatchNorm folded where it follows a conv), params f32 (DEVICE
// memory, compact: stem bias | scale | shift (384), then per block conv1 bias (128) + conv2 scale | shift (256), then the
// heads conv bias (128)), out bf16 [n,6,6,128] = relu(heads conv + bias).  blocks <= 10.
extern "C" int lzb_trunk_bf16(const void* planes, int64_t n, const void* w_stem, const void* w_trunk, const float* params,
                              int32_t blocks, void* out, void* stream) {
    using namespace lzb;
    LZB_REQUIRE(n > 0 && n < (1ll << 30), "bad batch size");
    LZB_REQUIRE(blocks >= 1 && blocks <= kMaxBlocks, "blocks must be in [1, 10]");
    LZB_REQUIRE(planes && w_stem && w_trunk && params && out, "null pointer");
    LZB_REQUIRE(((reinterpret_cast<uintptr_t>(planes) | reinterpret_cast<uintptr_t>(w_stem) | reinterpret_cast<uintptr_t>(w_trunk) |
                  reinterpret_cast<uintptr_t>(out)) & 15) == 0, "pointers must be 16-byte aligned");
    static EncodeTiledFn encode_tiled = nullptr;
    if (!encode_tiled) {
        cudaDriverEntryPointQueryResult st;
        void* fn = nullptr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &st) != cudaSuccess ||
            st != cudaDriverEntryPointSuccess || !fn) {
            set_error("lzb_trunk: cuTensorMapEncodeTiled unavailable");
            return LZB_ERR_CUDA;
        }
        encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
    }
    alignas(64) CUtensorMap tmIn, tmW0, tmW1;
    {
        const cuuint64_t dim[4] = {64, 6, 6, (cuuint64_t)n};
        const cuuint64_t stride[3] = {128, 128 * 6, 128 * 36};
        const cuuint32_t box[4] = {64, 6, 7, (cuuint32_t)kBoards};
        const cuuint32_t estr[4] = {1, 1, 1, 1};
        const CUresult rc = encode_tiled(&tmIn, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(planes), dim, stride, box,
                                         estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (rc != CUDA_SUCCESS) { set_error("lzb_trunk: tensor map (planes) failed (%d)", (int)rc); return LZB_ERR_CUDA; }
    }
    for (int which = 0; which < 2; ++which) {
        const cuuint64_t cin = which == 0 ? 64 : 128;
        const cuuint64_t rows = which == 0 ? 9 * 128 : ((cuuint64_t)blocks * 18 + 1) * 128;
        const cuuint64_t dim[2] = {cin, rows};
        const cuuint64_t stride[1] = {cin * 2};
        const cuuint32_t box[2] = {64, 64};
        const cuuint32_t estr[2] = {1, 1};
        const CUresult rc = encode_tiled(which == 0 ? &tmW0 : &tmW1, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                                         const_cast<void*>(which == 0 ? w_stem : w_trunk), dim, stride, box, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (rc != CUDA_SUCCESS) { set_error("lzb_trunk: tensor map (weights %d) failed (%d)", which, (int)rc); return LZB_ERR_CUDA; }
    }
    constexpr size_t smem = 1024 + (size_t)kCopyBufs * kCopyBytes + (size_t)kWStages * kWStageBytes +
                            8 * (2 * kCopyBufs + 2 * kWStages + 4) + 32 + 256;
    // the dynamic shared memory opt-in and the SM count are per DEVICE (a process may drive several GPUs)
    static int max_clusters[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { set_error("lzb_trunk: bad current device"); return LZB_ERR_CUDA; }
    if (max_clusters[dev] == 0) {
        if (cudaFuncSetAttribute(trunk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            set_error("lzb_trunk: cannot raise dynamic shared memory to %zu", smem);
            return LZB_ERR_CUDA;
        }
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 2) sms = kNumSMs;
        max_clusters[dev] = sms / 2;
    }
    TrunkParams P;
    P.out = reinterpret_cast<__nv_bfloat16*>(out); P.images = (int)n; P.blocks = blocks;
    // the parameter table goes to constant memory in stream order (device -> constant copy; a memcpy node under capture),
    // so every launch -- also a graph replay after an in-place weight refresh, or another network on this stream -- sees
    // its own current parameters
    if (cudaMemcpyToSymbolAsync(c_trunk_table, params, sizeof(float) * (size_t)(384 + blocks * 384 + 128), 0,
                                cudaMemcpyDeviceToDevice, (cudaStream_t)stream) != cudaSuccess) {
        set_error("lzb_trunk: parameter table upload failed: %s", cudaGetErrorString(cudaGetLastError()));
        return LZB_ERR_CUDA;
    }
    const int64_t pair_tiles = (n + 2 * kBoards - 1) / (2 * kBoards);
    const int clusters = (int)(pair_tiles < max_clusters[dev] ? pair_tiles : max_clusters[dev]);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * clusters);
    cfg.blockDim = dim3(kTrunkThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    (void)cudaLaunchKernelEx(&cfg, trunk_kernel, tmIn, tmW0, tmW1, P);
    return check_launch("trunk_kernel");
}
