// lz_actor.cu -- device-side game bookkeeping of the refilling self-play actor (liuzhou_b200/actor.py).
//
// Every live slot records one 336-B fixed row per ply (liuzhou_b200/compact.py: compact_rows_fixed layout) into its own
// game arena; when a game ends, its rows get their value targets and are appended to a linear output buffer together
// with one game record.  Two launches per ply, no host synchronisation, deterministic output order.
#include "lz_common.cuh"

using namespace lz;

namespace lzb {
namespace {

constexpr int kRowWords = 42;              // compact.FIXED_ROW_WORDS
constexpr int kRowVecs = kRowWords / 2;    // 16-byte vectors per row
constexpr int kPolicySlots = 64;
constexpr int kEmitThreads = 256;          // slots per emit block
constexpr uint32_t kNaN = 0x7FC00000u;     // the value words of a row whose game has not ended yet

__device__ __forceinline__ Packed load_state(const uint64_t* p, int64_t i) {
    const ulonglong2* v = reinterpret_cast<const ulonglong2*>(p + 4 * i);
    const ulonglong2 a = v[0], b = v[1];
    Packed r;
    r.w[0] = a.x; r.w[1] = a.y; r.w[2] = b.x; r.w[3] = b.y;
    return r;
}

// One warp per slot.  Lane l owns actions l, 32 + l, ..., so the policy row is read coalesced; ranks among the legal and
// the illegal actions come from ballots.  The policy slot order is compact._legal_order: legal actions ascending, then
// illegal ones ascending (non-zero only when the row is not representable, which the flags word then says).
__global__ void __launch_bounds__(kThreads)
actor_record_kernel(const uint64_t* __restrict__ states, const uint8_t* __restrict__ active,
                    const float* __restrict__ policy, const int64_t* __restrict__ chosen, int64_t G, int32_t max_plies,
                    int32_t* __restrict__ nrows, int64_t* __restrict__ arena, int8_t* __restrict__ signs,
                    int16_t* __restrict__ actions, unsigned long long* __restrict__ ctl) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t g = warp; g < G; g += nwarps) {
        if (!active[g]) continue;
        const int r = nrows[g];
        if (r >= max_plies) {                              // cannot happen under the finish rules; never silent
            if (lane == 0) atomicOr(&ctl[3], 2ull);
            continue;
        }
        State<int> s;
        unpack(load_state(states, g), s);
        Legal L;
        legal_actions<int, false>(s, L, true);             // encode_actions_fast semantics (no game-over check)
        uint64_t w[4];
        legal_to_words(L, w);
        const int nlegal = popc64(w[0]) + popc64(w[1]) + popc64(w[2]) + popc64(w[3]);
        const int64_t row = g * (int64_t)max_plies + r;
        int64_t* out = arena + row * kRowWords;
        float* pol_out = reinterpret_cast<float*>(out + 8);
        const float* pol = policy + g * kActionDim;
        bool off_legal = false;
        int legal_before = 0;
#pragma unroll
        for (int c = 0; c < 7; ++c) {
            const int a = 32 * c + lane;
            const bool in = a < kActionDim;
            const bool lg = in && ((w[a >> 6] >> (a & 63)) & 1);
            const uint32_t m = __ballot_sync(0xffffffffu, lg);
            const int rank_l = legal_before + __popc(m & ((1u << lane) - 1u));
            legal_before += __popc(m);
            if (in) {
                const float v = pol[a];
                const int pos = lg ? rank_l : nlegal + (a - rank_l);
                if (pos < kPolicySlots) pol_out[pos] = v;
                off_legal |= !lg && v != 0.0f;
            }
        }
        const bool bad_policy = __any_sync(0xffffffffu, off_legal);
        if (lane == 0) {
            const bool black = s.player == 1;
            const bool phase_ok = s.phase >= 1 && s.phase <= 7;
            const uint64_t phase_bits = phase_ok ? (uint64_t)s.phase : 1ull;   // argmax of an all-zero phase one-hot + 1
            out[0] = (black ? s.black : s.white) | (phase_bits << 36);
            out[1] = black ? s.white : s.black;
            out[2] = black ? s.mb : s.mw;
            out[3] = black ? s.mw : s.mb;
            out[4] = (int64_t)w[0]; out[5] = (int64_t)w[1]; out[6] = (int64_t)w[2]; out[7] = (int64_t)w[3];
            out[40] = (int64_t)(((uint64_t)kNaN << 32) | kNaN);
            out[41] = (bad_policy || nlegal > kPolicySlots || !phase_ok) ? 1 : 0;
            signs[row] = black ? (int8_t)1 : (int8_t)-1;
            actions[row] = (int16_t)chosen[g];
            nrows[g] = r + 1;
        }
    }
}

// Sum of (x, y) over the block; every thread gets the totals.
__device__ __forceinline__ void block_sum2(long long& x, long long& y, long long* sh) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        x += __shfl_xor_sync(0xffffffffu, x, o);
        y += __shfl_xor_sync(0xffffffffu, y, o);
    }
    __syncthreads();
    if (lane == 0) { sh[2 * wid] = x; sh[2 * wid + 1] = y; }
    __syncthreads();
    x = y = 0;
    for (int i = 0; i < kEmitThreads / 32; ++i) { x += sh[2 * i]; y += sh[2 * i + 1]; }
}

// Exclusive prefix of (x, y) over the block in thread order.
__device__ __forceinline__ void block_exclusive_scan2(long long& x, long long& y, long long* sh) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    long long ix = x, iy = y;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long tx = __shfl_up_sync(0xffffffffu, ix, o), ty = __shfl_up_sync(0xffffffffu, iy, o);
        if (lane >= o) { ix += tx; iy += ty; }
    }
    __syncthreads();
    if (lane == 31) { sh[2 * wid] = ix; sh[2 * wid + 1] = iy; }
    __syncthreads();
    long long bx = 0, by = 0;
    for (int i = 0; i < wid; ++i) { bx += sh[2 * i]; by += sh[2 * i + 1]; }
    x = bx + ix - x;
    y = by + iy - y;
}

// Block b owns slots [256 b, 256 b + 256).  Offsets are a stable scan over the finished flags in slot order: every block
// sums the slots before its range itself (G flags, a few KB from L2), scans its own range, and copies its games.  The
// last block to finish advances the cursors and clears the row counters of the finished slots.
__global__ void __launch_bounds__(kEmitThreads)
actor_emit_kernel(const uint8_t* __restrict__ finished, const float* __restrict__ result,
                  const float* __restrict__ soft, const uint64_t* __restrict__ states, int64_t G, int32_t max_plies,
                  int32_t* __restrict__ nrows, const int64_t* __restrict__ arena, const int8_t* __restrict__ signs,
                  const int16_t* __restrict__ actions, int64_t* __restrict__ out_rows,
                  int16_t* __restrict__ out_actions, int64_t* __restrict__ records, int64_t capacity,
                  unsigned long long* __restrict__ ctl, int64_t step) {
    __shared__ long long sh[2 * (kEmitThreads / 32)];
    __shared__ int s_slot[kEmitThreads];
    __shared__ long long s_row[kEmitThreads];
    __shared__ int s_count;
    __shared__ bool s_last;
    const int tid = threadIdx.x;
    const int64_t lo = (int64_t)blockIdx.x * kEmitThreads;
    long long before_g = 0, before_r = 0, tot_g = 0, tot_r = 0;
    for (int64_t i = tid; i < G; i += kEmitThreads) {
        const long long f = finished[i] ? 1 : 0, l = f ? nrows[i] : 0;
        tot_g += f; tot_r += l;
        if (i < lo) { before_g += f; before_r += l; }
    }
    block_sum2(before_g, before_r, sh);
    block_sum2(tot_g, tot_r, sh);
    const int64_t slot = lo + tid;
    const bool fin = slot < G && finished[slot];
    long long rank_g = fin ? 1 : 0, rank_r = fin ? nrows[slot] : 0;
    block_exclusive_scan2(rank_g, rank_r, sh);
    if (fin) { s_slot[rank_g] = (int)slot; s_row[rank_g] = before_r + rank_r; }
    if (tid == kEmitThreads - 1) s_count = (int)rank_g + (fin ? 1 : 0);
    __syncthreads();
    const long long row_cursor = (long long)ctl[0], game_cursor = (long long)ctl[1], serial0 = (long long)ctl[2];
    const int count = s_count;
    uint32_t flags = 0;
    for (int k = 0; k < count; ++k) {
        const int g = s_slot[k];
        const int len = nrows[g];
        const long long r0 = row_cursor + s_row[k];
        const long long gi = game_cursor + before_g + k;
        if (r0 + len > capacity || gi >= capacity) {       // writes nothing past the end; the drain raises
            if (tid == 0) atomicOr(&ctl[3], 1ull);
            continue;
        }
        const float res = result[g], sv = soft[g];
        const uint4* src = reinterpret_cast<const uint4*>(arena + (int64_t)g * max_plies * kRowWords);
        uint4* dst = reinterpret_cast<uint4*>(out_rows + r0 * kRowWords);
        for (int e = tid; e < len * kRowVecs; e += kEmitThreads) {
            uint4 v = src[e];
            if (e % kRowVecs == kRowVecs - 1) {              // words 40 (value | soft) and 41 (flags)
                const int p = e / kRowVecs;
                const float sg = (float)signs[(int64_t)g * max_plies + p];
                v.x = __float_as_uint(sg * res);
                v.y = __float_as_uint(sg * sv);
                flags |= v.z;
            }
            dst[e] = v;
        }
        for (int p = tid; p < len; p += kEmitThreads) out_actions[r0 + p] = actions[(int64_t)g * max_plies + p];
        if (tid == 0) {
            const Packed st = load_state(states, g);
            const int delta = popc64(st.w[0] & kFull) - popc64(st.w[1] & kFull);
            int64_t* rec = records + gi * 8;
            rec[0] = serial0 + before_g + k;
            rec[1] = g;
            rec[2] = len;
            rec[3] = r0;
            rec[4] = step;
            rec[5] = delta;
            rec[6] = (int64_t)(((uint64_t)__float_as_uint(sv) << 32) | __float_as_uint(res));
            rec[7] = 0;
            atomicAdd(&ctl[res > 0.0f ? 6 : res < 0.0f ? 7 : 8], 1ull);
            atomicAdd(&ctl[9 + min(max(delta + 18, 0), 36)], 1ull);
        }
    }
    if (flags) atomicOr(&ctl[4], (unsigned long long)flags);
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&ctl[5], 1ull) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int64_t i = tid; i < G; i += kEmitThreads)
        if (finished[i]) nrows[i] = 0;
    if (tid == 0) {
        ctl[0] += (unsigned long long)tot_r;
        ctl[1] += (unsigned long long)tot_g;
        ctl[2] += (unsigned long long)tot_g;
        ctl[5] = 0;
    }
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace
}  // namespace lzb

using namespace lzb;

extern "C" int lzb_actor_record(const uint64_t* states, const uint8_t* active, const float* policy, const int64_t* chosen,
                                int64_t G, int32_t max_plies, int32_t* nrows, int64_t* arena, int8_t* signs,
                                int16_t* actions, uint64_t* ctl, void* stream) {
    LZB_REQUIRE(G >= 0 && max_plies > 0, "bad shape");
    if (G == 0) return LZB_OK;
    LZB_REQUIRE(states && active && policy && chosen && nrows && arena && signs && actions && ctl, "null pointer");
    LZB_REQUIRE(aligned16(states), "states must be 16-byte aligned");
    actor_record_kernel<<<warp_grid(G), kThreads, 0, (cudaStream_t)stream>>>(
        states, active, policy, chosen, G, max_plies, nrows, arena, signs, actions,
        reinterpret_cast<unsigned long long*>(ctl));
    return check_launch("actor_record_kernel");
}

extern "C" int lzb_actor_emit(const uint8_t* finished, const float* result, const float* soft, const uint64_t* states,
                              int64_t G, int32_t max_plies, int32_t* nrows, const int64_t* arena, const int8_t* signs,
                              const int16_t* actions, int64_t* out_rows, int16_t* out_actions, int64_t* records,
                              int64_t capacity, uint64_t* ctl, int64_t step, void* stream) {
    LZB_REQUIRE(G >= 0 && max_plies > 0 && capacity >= 0, "bad shape");
    if (G == 0) return LZB_OK;
    LZB_REQUIRE(finished && result && soft && states && nrows && arena && signs && actions && out_rows && out_actions &&
                records && ctl, "null pointer");
    LZB_REQUIRE(aligned16(states) && aligned16(arena) && aligned16(out_rows), "states, arena and out_rows must be 16-byte aligned");
    const int64_t blocks = (G + kEmitThreads - 1) / kEmitThreads;
    LZB_REQUIRE(blocks < (1 << 30), "too many slots");
    actor_emit_kernel<<<(int)blocks, kEmitThreads, 0, (cudaStream_t)stream>>>(
        finished, result, soft, states, G, max_plies, nrows, arena, signs, actions, out_rows, out_actions, records,
        capacity, reinterpret_cast<unsigned long long*>(ctl), step);
    return check_launch("actor_emit_kernel");
}
