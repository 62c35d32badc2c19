// lz_tree.cu -- device-resident full-tree MCTS: selection (PUCT descent, virtual loss), expansion (legal-move
// generation + atomic phase transitions on bitboards + node allocation from a bump arena) and player-aware
// backup, one warp per game tree.
//
// Semantics = the reference's portable tree search (/root/reference/v1/cpp/portable_mcts.cpp:483-939):
//   select : while expanded & has children & !terminal: argmax_a q + c*P*sqrt(max(1,N_parent))/(1+N_child),
//            q = 0 if N_child == 0 else mean(child) negated iff child.player != node.player; ties -> lowest action
//   expand : children for all legal actions (scalar-engine rules) in ascending action index,
//            prior = p[a] / sum_legal p (uniform if the sum is <= 0), child.terminal = IsGameOver(child)
//   backup : visit += 1, value_sum += v up the path, v negated when parent.player != node.player
// Arithmetic is fp64 with the reference's operation order (fp64 priors / value sums, int32 visits), so that
// visit counts are bit-identical for identical network outputs.
//
// HBM layout (structure of arrays over a node arena; the children of a node are contiguous, so a warp reads
// N / W / P / info of all siblings with coalesced loads):
//   visit i32[cap] | value_sum f64[cap] | prior f64[cap] | info u32[cap] | first_child i32[cap] |
//   parent i32[cap] | state u64[cap][4]
// Nodes 0..T-1 are the roots; the rest is handed out by an atomic bump pointer (one atomicAdd per expansion).
// A tree is only ever touched by its own warp, so N / W updates need no atomics and results are
// deterministic regardless of scheduling.
#include "lz_common.cuh"

using namespace lz;

namespace lzb {
namespace {

constexpr int32_t kFlagArena = 1, kFlagIllegalAdvance = 2, kFlagBadNetwork = 4;   // sticky bits of counters[1]
constexpr uint32_t kInfoActionMask = 0xFFu;
constexpr uint32_t kInfoTerminal = 1u << 16;
constexpr uint32_t kInfoExpanded = 1u << 17;
constexpr uint32_t kInfoNoLegal = 1u << 18;
constexpr uint32_t kInfoWhite = 1u << 19;
constexpr uint32_t kInfoPending = 1u << 20;
constexpr uint32_t kInfoInactive = 1u << 21;
__device__ __forceinline__ int info_nchild(uint32_t inf) { return (int)((inf >> 8) & 0xFFu); }

__device__ __forceinline__ Packed load_packed(const uint64_t* p, int64_t i) {
    const ulonglong2* v = reinterpret_cast<const ulonglong2*>(p + 4 * i);
    const ulonglong2 a = v[0], b = v[1];
    Packed r; r.w[0] = a.x; r.w[1] = a.y; r.w[2] = b.x; r.w[3] = b.y;
    return r;
}
__device__ __forceinline__ void store_packed(uint64_t* p, int64_t i, const Packed& s) {
    ulonglong2* v = reinterpret_cast<ulonglong2*>(p + 4 * i);
    v[0] = make_ulonglong2(s.w[0], s.w[1]);
    v[1] = make_ulonglong2(s.w[2], s.w[3]);
}

// TerminalValue, portable_mcts.cpp:267-273
__device__ __forceinline__ double terminal_value(const State<int>& s) {
    const int w = winner(s);
    return w == 0 ? 0.0 : (w == s.player ? 1.0 : -1.0);
}

__global__ void __launch_bounds__(kThreads)
tree_init_kernel(lzb_tree A, const uint64_t* __restrict__ roots, const uint8_t* __restrict__ active) {
    const int64_t T = A.num_trees;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (int64_t)gridDim.x * blockDim.x) {
        const Packed p = load_packed(roots, t);
        State<int> s;
        unpack(p, s);
        store_packed(A.state, t, p);
        A.visit[t] = 0; A.value_sum[t] = 0.0; A.prior[t] = 1.0; A.first_child[t] = -1; A.parent[t] = -1;
        uint32_t inf = 0xFFu;
        if (game_over(s)) inf |= kInfoTerminal;                       // Node::terminal = IsGameOver (:414)
        if (s.player == -1) inf |= kInfoWhite;
        if (active && !active[t]) inf |= kInfoInactive;
        A.info[t] = inf;
        A.root_value[t] = 0.0;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        A.counters[0] = (int32_t)T; A.counters[1] = 0; A.counters[2] = 0; A.counters[3] = 0;
        A.counters[4] = 0; A.counters[5] = 0;      // [4] sibling records scanned by select, [5] levels descended
        A.counters[6] = 0x7fffffff;                // [6] arena index of the FIRST failed allocation (nothing above it is valid)
    }
}

// Backup, portable_mcts.cpp:876-892 (one lane walks the parent chain)
__device__ __forceinline__ void backup_path(const lzb_tree& A, int node, double v) {
    while (true) {
        A.visit[node] += 1;
        A.value_sum[node] = __dadd_rn(A.value_sum[node], v);
        const int p = A.parent[node];
        if (p < 0) break;
        if ((A.info[p] ^ A.info[node]) & kInfoWhite) v = -v;
        node = p;
    }
}
// The same backup with the path known up front (recorded during the descent): lane j owns the node at depth j, so
// the whole chain is ONE round trip to HBM instead of one per level.  The value flips sign once per colour change
// between a node and its parent, i.e. node j receives +v iff it has the leaf's colour -- the parity of the colour
// changes between j and the leaf.  Each node gets exactly the fp64 add the sequential walk would do (bit-identical).
constexpr int kPathLanes = 32;                 // deeper paths fall back to the parent walk
constexpr int kPathStride = kPathLanes + 2;    // [0,32) nodes | [32] depth (-1: use the parent walk) | [33] colour bits
__device__ __forceinline__ void backup_recorded(const lzb_tree& A, int lane, int path_node, uint32_t white_mask, int depth,
                                                double v) {
    if (lane <= depth) {
        const bool same = ((white_mask >> lane) & 1u) == ((white_mask >> depth) & 1u);
        A.visit[path_node] += 1;
        A.value_sum[path_node] = __dadd_rn(A.value_sum[path_node], same ? v : -v);
    }
}

// Virtual loss for K > 1 leaves per tree per wave: every node on the path gets +1 visit; its value sum moves
// by `vl` AGAINST the player who chose it, so q seen from the parent always drops.  sign = +1 apply, -1 revert.
__device__ __forceinline__ void virtual_loss_path(const lzb_tree& A, int node, double vl, int sign) {
    while (true) {
        const int p = A.parent[node];
        A.visit[node] += sign;
        if (p >= 0) {
            const bool same = !((A.info[p] ^ A.info[node]) & kInfoWhite);
            A.value_sum[node] = __dadd_rn(A.value_sum[node], (same ? -vl : vl) * (double)sign);
        }
        if (p < 0) break;
        node = p;
    }
}

// One state -> bf16 channels-last planes padded to 64 channels ([36 cells][64 ch] = 288 x 16 B), written by a warp.
// kPadToo = false writes only channels 0..15 (two of the eight 16-byte groups of a cell): channels 16..63 are zero padding
// that nothing ever changes in a buffer that starts out zero (InferenceNet.new_input), and 3/4 of the 4.6 KB per leaf.
template <bool kPadToo>
__device__ __forceinline__ void encode_c64_row(const Packed& p, uint4* __restrict__ out, int lane) {
    State<int> s;
    unpack(p, s);
    const bool black = s.player == 1;
    const uint64_t p0 = black ? s.black : s.white, p1 = black ? s.white : s.black;
    const uint64_t p2 = black ? s.mb : s.mw, p3 = black ? s.mw : s.mb;
    const int phase_plane = 3 + s.phase;
    constexpr int kGroups = kPadToo ? 8 : 2;
    for (int e = lane; e < 36 * kGroups; e += 32) {
        const int cell = e / kGroups, oct = e - cell * kGroups;
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        if (oct == 0) {                                          // planes 0..7: the four bitboards + phases 1..4
            const uint32_t b0 = (uint32_t)(p0 >> cell) & 1u, b1 = (uint32_t)(p1 >> cell) & 1u;
            const uint32_t b2 = (uint32_t)(p2 >> cell) & 1u, b3 = (uint32_t)(p3 >> cell) & 1u;
            w[0] = b0 * 0x00003F80u | b1 * 0x3F800000u;          // bf16 1.0 in the low / high half
            w[1] = b2 * 0x00003F80u | b3 * 0x3F800000u;
            w[2] = (phase_plane == 4 ? 0x00003F80u : 0u) | (phase_plane == 5 ? 0x3F800000u : 0u);
            w[3] = (phase_plane == 6 ? 0x00003F80u : 0u) | (phase_plane == 7 ? 0x3F800000u : 0u);
        } else if (oct == 1) {                                   // planes 8..10: phases 5..7; 11..15: zero
            w[0] = (phase_plane == 8 ? 0x00003F80u : 0u) | (phase_plane == 9 ? 0x3F800000u : 0u);
            w[1] = phase_plane == 10 ? 0x00003F80u : 0u;
        }
        out[cell * 8 + oct] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// status codes written per leaf slot
constexpr int kLeafEval = 0;       // needs a network evaluation, then expand (+ backup)
constexpr int kLeafDone = 1;       // terminal / inactive: nothing to evaluate (backup already done)
constexpr int kLeafDuplicate = 2;  // K > 1 only: same leaf already pending in this wave (simulation dropped)

// The K descents of one tree, by one warp (SelectLeaves / SelectPath / SelectChild, portable_mcts.cpp:515-552,832-874).
__device__ __forceinline__ void select_tree(const lzb_tree& A, int64_t t, int K, double c_puct, double vl,
                                            int32_t* __restrict__ leaf_node, int32_t* __restrict__ leaf_status,
                                            uint64_t* __restrict__ leaf_states, int32_t* __restrict__ leaf_path,
                                            int roots_only, uint4* __restrict__ enc_out, int lane) {
    {
        // leaf-batch rows of this tree: identity, or (waves only) the compacted row A.tree_rows[t]; a negative row
        // means the tree takes no part in this wave (finished game): nothing is read or written for it
        int64_t base = t;
        if (A.tree_rows && !roots_only) {
            const int r = A.tree_rows[t];
            if (r < 0) return;
            base = r;
        }
        for (int k = 0; k < K; ++k) {
            const int64_t slot = base * K + k;
            int node = (int)t;
            uint32_t inf = A.info[node];
            // SelectLeaves :519-521; PrepareRoots (:483-513) only ever evaluates an unexpanded root -- a root that
            // kept its subtree through advance_roots is left alone
            if ((inf & (kInfoTerminal | kInfoInactive)) || (roots_only && (inf & kInfoExpanded))) {
                if (lane == 0) { leaf_node[slot] = -1; leaf_status[slot] = kLeafDone; }
                continue;
            }
            // SelectPath :862-874.  One dependent HBM round trip per level: the sibling scan also fetches each
            // child's first_child / info / visit, so the next level needs nothing else from the chosen child.
            int fc = A.first_child[node], nv = A.visit[node];
            int depth = 0, path_node = lane == 0 ? node : -1, scanned = 0;
            bool path_white = lane == 0 && (inf & kInfoWhite);
            while ((inf & kInfoExpanded) && info_nchild(inf) > 0 && !(inf & kInfoTerminal)) {
                const int n = info_nchild(inf);
                scanned += n;
                const uint32_t node_white = inf & kInfoWhite;
                double best = -INFINITY;
                int best_i = 0x7fffffff, b_vc = 0, b_fc = -1;
                uint32_t b_inf = 0;
                const double sqrt_total = sqrt((double)(nv > 1 ? nv : 1));
                for (int i = lane; i < n; i += 32) {                 // SelectChild :832-860
                    const int c = fc + i;
                    const int vc = A.visit[c];
                    const uint32_t ci = A.info[c];
                    const int cfc = A.first_child[c];
                    const double pr = A.prior[c];
                    const double ws = A.value_sum[c];               // loaded whether or not vc > 0: ONE round trip per level
                    double q = 0.0;
                    if (vc > 0) {
                        q = __ddiv_rn(ws, (double)vc);
                        if ((ci & kInfoWhite) != node_white) q = -q;
                    }
                    const double u = __ddiv_rn(__dmul_rn(__dmul_rn(c_puct, pr), sqrt_total), (double)(1 + vc));
                    const double score = __dadd_rn(q, u);
                    if (score > best || (score == best && i < best_i)) { best = score; best_i = i; b_vc = vc; b_fc = cfc; b_inf = ci; }
                }
                {
                    // warp argmax (ties -> lowest child index) with three redux.sync instead of five shuffle rounds: the
                    // score as an order-preserving 64-bit key, maximised high word first, then the lowest index among
                    // the lanes that hold the maximum.  -0.0 == +0.0 in the reference's comparison: canonicalised.
                    const double sc = best == 0.0 ? 0.0 : best;
                    const unsigned long long bits = (unsigned long long)__double_as_longlong(sc);
                    const unsigned long long key = bits ^ ((bits >> 63) ? ~0ull : 0x8000000000000000ull);
                    const uint32_t khi = (uint32_t)(key >> 32), klo = (uint32_t)key;
                    const bool has = best_i != 0x7fffffff;
                    const uint32_t mhi = __reduce_max_sync(0xffffffffu, has ? khi : 0u);
                    const bool c1 = has && khi == mhi;
                    const uint32_t mlo = __reduce_max_sync(0xffffffffu, c1 ? klo : 0u);
                    const bool c2 = c1 && klo == mlo;
                    best_i = (int)__reduce_min_sync(0xffffffffu, c2 ? (uint32_t)best_i : 0x7fffffffu);
                }
                if (best_i == 0x7fffffff) break;                     // child == nullptr
                const int owner = best_i & 31;                       // that lane's local best IS the global best
                node = fc + best_i;
                inf = __shfl_sync(0xffffffffu, b_inf, owner);
                nv = __shfl_sync(0xffffffffu, b_vc, owner);
                fc = __shfl_sync(0xffffffffu, b_fc, owner);
                ++depth;
                if (depth < kPathLanes && lane == depth) { path_node = node; path_white = (inf & kInfoWhite) != 0; }
            }
            const bool recorded = depth < kPathLanes;
            if (lane == 0 && depth > 0) { atomicAdd(&A.counters[4], scanned); atomicAdd(&A.counters[5], depth); }
            const uint32_t white_mask = __ballot_sync(0xffffffffu, path_white);
            int status;
            if (inf & kInfoTerminal) {                               // :527-532
                double tv = 0.0;
                if (lane == 0) {
                    State<int> s;
                    unpack(load_packed(A.state, node), s);
                    tv = (inf & kInfoNoLegal) ? -1.0 : terminal_value(s);
                    atomicAdd(&A.counters[3], 1);
                }
                tv = __shfl_sync(0xffffffffu, tv, 0);
                if (recorded) backup_recorded(A, lane, path_node, white_mask, depth, tv);
                else if (lane == 0) backup_path(A, node, tv);
                status = kLeafDone;
            } else if ((inf & kInfoExpanded) && info_nchild(inf) == 0) {   // :533-538
                if (lane == 0) A.info[node] = inf | kInfoTerminal | kInfoNoLegal;
                if (recorded) backup_recorded(A, lane, path_node, white_mask, depth, -1.0);
                else if (lane == 0) backup_path(A, node, -1.0);
                status = kLeafDone;
            } else if (inf & kInfoPending) {
                status = kLeafDuplicate;
            } else {
                status = kLeafEval;
                Packed leaf;
                leaf.w[0] = leaf.w[1] = leaf.w[2] = leaf.w[3] = 0;
                if (lane == 0) {
                    A.info[node] = inf | kInfoPending;
                    leaf = load_packed(A.state, node);
                    store_packed(leaf_states, slot, leaf);
                    if (K > 1 && vl > 0.0) virtual_loss_path(A, node, vl, +1);
                }
                if (enc_out) {      // the network input of this leaf, written here instead of by a separate launch
#pragma unroll
                    for (int k = 0; k < 4; ++k) leaf.w[k] = __shfl_sync(0xffffffffu, leaf.w[k], 0);
                    encode_c64_row<false>(leaf, enc_out + slot * 288, lane);
                }
                if (leaf_path) {                                     // the path travels to the expand / backup kernel
                    leaf_path[slot * kPathStride + lane] = path_node;
                    if (lane == 0) {
                        leaf_path[slot * kPathStride + kPathLanes] = recorded ? depth : -1;
                        leaf_path[slot * kPathStride + kPathLanes + 1] = (int32_t)white_mask;
                    }
                }
            }
            if (lane == 0) { leaf_node[slot] = status == kLeafEval ? node : -1; leaf_status[slot] = status; }
            __syncwarp();
        }
    }
}

__global__ void __launch_bounds__(kThreads, 4)      // 4 x 8 warps per SM: all 4,096 trees of a wave resident at once
tree_select_kernel(lzb_tree A, int K, double c_puct, double vl, int32_t* __restrict__ leaf_node,
                   int32_t* __restrict__ leaf_status, uint64_t* __restrict__ leaf_states, int32_t* __restrict__ leaf_path,
                   int roots_only, uint4* __restrict__ enc_out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t t = warp; t < A.num_trees; t += nwarps)
        select_tree(A, t, K, c_puct, vl, leaf_node, leaf_status, leaf_states, leaf_path, roots_only, enc_out, lane);
}

// Both expand kernels ask for 3 blocks of 8 warps per SM; tree_expand_select_kernel says why.
constexpr int kExpandMinBlocks = 3;

// Expand (portable_mcts.cpp:894-939) + Backup for every evaluated leaf slot of a tree, sequentially in slot
// order (deterministic).  priors f32[slots,220] dense over the 220-d action space, values f32[slots].
// (spri = this warp's 220-float staging row in shared memory)
__device__ __forceinline__ void expand_tree(const lzb_tree& A, int64_t t, int K, const int32_t* __restrict__ leaf_node,
                                            const int32_t* __restrict__ leaf_status, const float* __restrict__ priors,
                                            const float* __restrict__ values, int do_backup, double vl,
                                            const int32_t* __restrict__ leaf_path, float* spri, int lane) {
    {
        int64_t base = t;
        if (A.tree_rows && do_backup) {           // waves use the compacted rows; the root step (no backup) never does
            const int r = A.tree_rows[t];
            if (r < 0) return;
            base = r;
        }
        for (int k = 0; k < K; ++k) {
            const int64_t slot = base * K + k;
            // Everything whose address depends only on the slot is requested in ONE round trip, before the status is
            // looked at (all of it is valid memory for any slot): status, node, value, this lane's 7 prior entries, the
            // descent's path.  The second round trip fetches what hangs off the node / the path.
            const int st = leaf_status[slot];
            const int node_raw = leaf_node[slot];
            const float value_f = values[slot];
            float pv_reg[7];
#pragma unroll
            for (int j = 0; j < 7; ++j) {
                const int a = lane + 32 * j;
                pv_reg[j] = a < kActionDim ? priors[slot * kActionDim + a] : 0.0f;
            }
            int path_node = -1, path_depth = -1;
            uint32_t path_white = 0;
            if (do_backup && leaf_path) {
                path_node = leaf_path[slot * kPathStride + lane];
                path_depth = leaf_path[slot * kPathStride + kPathLanes];
                path_white = (uint32_t)leaf_path[slot * kPathStride + kPathLanes + 1];
            }
            if (st != kLeafEval) continue;
            const int node = node_raw;
            // statistics of the path nodes for the backup at the end: only this warp touches this tree, so they cannot
            // change in between -- except through this warp's own virtual-loss bookkeeping (K > 1), which re-reads
            const bool pre_backup = do_backup && path_depth >= 0 && !(K > 1 && vl > 0.0);
            int pre_visit = 0;
            double pre_sum = 0.0;
            if (pre_backup && lane <= path_depth) { pre_visit = A.visit[path_node]; pre_sum = A.value_sum[path_node]; }
            State<int> s;
            unpack(load_packed(A.state, node), s);
            Legal L;
            legal_actions<int, true>(s, L, true);
            const int n = legal_count(L);
            double value = (double)value_f;
            const uint32_t inf = A.info[node] & ~kInfoPending;
            if (lane == 0 && K > 1 && vl > 0.0) virtual_loss_path(A, node, vl, -1);
            __syncwarp();
            // CompletePending / Expand throw on a non-finite value or a negative / non-finite prior
            // (portable_mcts.cpp: "model value is NaN or Inf", "model prior is negative, NaN, or Inf"); here: sticky
            // flag, the leaf stays unexpanded and nothing is backed up, so the tree statistics stay clean
            bool bad = !isfinite(value);
            if (n > 0) {                          // the prior row is staged in shared memory once, checked, then used
#pragma unroll
                for (int j = 0; j < 7; ++j) {
                    const int a = lane + 32 * j;
                    if (a < kActionDim) {
                        const float pv = pv_reg[j];
                        spri[a] = pv;
                        if (legal_test(L, a) && (!(pv >= 0.0f) || isinf(pv))) bad = true;
                    }
                }
            }
            __syncwarp();                         // staging writes visible to lane 0's sequential sum below
            bad = __any_sync(0xffffffffu, bad);
            if (bad) {
                if (lane == 0) { A.info[node] = inf; atomicOr(&A.counters[1], kFlagBadNetwork); }
                __syncwarp();
                continue;
            }
            if (n == 0) {                                             // :900-907
                const bool over = game_over(s);
                value = over ? terminal_value(s) : -1.0;
                if (lane == 0) {
                    A.info[node] = inf | kInfoExpanded | kInfoTerminal | (over ? 0u : kInfoNoLegal);
                    if (node < A.num_trees) A.root_value[node] = value;
                }
            } else {
                // prior_sum accumulated sequentially in ascending action order, in fp64 (:909-918).  Lane i holds the
                // i-th legal action and its prior (needed for its child anyway); the values reach the adder by shuffle,
                // so the dependent chain is one fp64 add per action instead of bit scan + shared-memory load + add.
                // Every lane runs the same additions: no broadcast of the result.
                int fc = 0;
                if (lane == 0) fc = atomicAdd(&A.counters[0], n);   // requested first: its round trip runs under the sum
                uint64_t lw[4];
                legal_to_words(L, lw);
                double prior_sum = 0.0;
                int act0 = -1, act1 = -1, act2 = -1;               // this lane's actions of rounds 0..2 (n <= 72 < 96)
                for (int r = 0; r * 32 < n; ++r) {
                    const int i = r * 32 + lane;
                    const int a = i < n ? legal_kth_words(lw, i) : -1;
                    if (r == 0) act0 = a; else if (r == 1) act1 = a; else if (r == 2) act2 = a;
                    const float pv = a >= 0 ? spri[a] : 0.0f;
                    const int m = n - r * 32 < 32 ? n - r * 32 : 32;
                    for (int j0 = 0; j0 < m; j0 += 8) {            // eight shuffles in flight, then the eight ordered adds
                        float v[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) v[j] = __shfl_sync(0xffffffffu, pv, (j0 + j) & 31);
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            if (j0 + j < m) prior_sum = __dadd_rn(prior_sum, (double)v[j]);
                    }
                }
                if (lane == 0) {
                    // the bump pointer only grows: after the first failure every later allocation fails too, so
                    // [num_trees, first failed index) is exactly the set of valid nodes (advance_roots relies on it)
                    if ((int64_t)fc + n > A.capacity) { atomicOr(&A.counters[1], 1); atomicMin(&A.counters[6], fc); fc = -1; }
                    else atomicAdd(&A.counters[2], 1);
                }
                fc = __shfl_sync(0xffffffffu, fc, 0);
                if (fc >= 0) {
                    const bool uniform = !(prior_sum > 0.0) || isinf(prior_sum);      // :919
                    for (int i = lane, r = 0; i < n; i += 32, ++r) {   // child i <-> i-th legal action in ascending index order
                        {
                            const int a = r == 0 ? act0 : r == 1 ? act1 : r == 2 ? act2 : legal_kth_words(lw, i);
                            const int c = fc + i;
                            State<int> cs = s;
                            apply_index<int, true>(cs, a);      // a comes from this state's legal set
                            store_packed(A.state, c, pack(cs));
                            A.visit[c] = 0; A.value_sum[c] = 0.0;
                            A.prior[c] = uniform ? __ddiv_rn(1.0, (double)n) : __ddiv_rn((double)spri[a], prior_sum);
                            A.first_child[c] = -1; A.parent[c] = node;
                            uint32_t ci = (uint32_t)a;
                            if (game_over(cs)) ci |= kInfoTerminal;
                            if (cs.player == -1) ci |= kInfoWhite;
                            A.info[c] = ci;
                        }
                    }
                    if (lane == 0) {
                        A.first_child[node] = fc;
                        A.info[node] = (inf & ~(0xFFu << 8)) | ((uint32_t)n << 8) | kInfoExpanded;
                        if (node < A.num_trees) A.root_value[node] = value;      // Node::initial_value
                    }
                } else if (lane == 0) {
                    A.info[node] = inf;      // arena exhausted: leave the leaf unexpanded, flag is reported to the host
                }
            }
            __syncwarp();
            if (do_backup) {
                if (pre_backup) {                 // backup_recorded with the statistics fetched at the top: stores only
                    if (lane <= path_depth) {
                        const bool same = ((path_white >> lane) & 1u) == ((path_white >> path_depth) & 1u);
                        A.visit[path_node] = pre_visit + 1;
                        A.value_sum[path_node] = __dadd_rn(pre_sum, same ? value : -value);
                    }
                } else if (path_depth >= 0) backup_recorded(A, lane, path_node, path_white, path_depth, value);
                else if (lane == 0) backup_path(A, node, value);
            }
            __syncwarp();
        }
    }
}

__global__ void __launch_bounds__(kThreads, kExpandMinBlocks)
tree_expand_kernel(lzb_tree A, int K, const int32_t* __restrict__ leaf_node, const int32_t* __restrict__ leaf_status,
                   const float* __restrict__ priors, const float* __restrict__ values, int do_backup, double vl,
                   const int32_t* __restrict__ leaf_path) {
    __shared__ float s_pri[kWarpsPerBlock][kActionDim];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + w;
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t t = warp; t < A.num_trees; t += nwarps)
        expand_tree(A, t, K, leaf_node, leaf_status, priors, values, do_backup, vl, leaf_path, s_pri[w], lane);
}

// Expand + backup of wave w FOLLOWED BY the descent of wave w + 1, tree by tree: the trees are independent, so the two
// latency chains of a warp run back to back without a grid-wide barrier between them, and a simulation wave needs one
// tree kernel instead of two (select -> network -> expand becomes network -> expand+select).  The warp's own writes
// (children, statistics along the path) are ordered before its reads by __syncwarp().
// 4,096 trees are 4,096 warps = 27.7 per SM; 3 blocks of 8 warps (80 registers) keep only 24 resident, so 13 % of the
// blocks wait for a second round and the kernel lasts two latency chains.
__global__ void __launch_bounds__(kThreads, kExpandMinBlocks)
tree_expand_select_kernel(lzb_tree A, int K, int32_t* __restrict__ leaf_node, int32_t* __restrict__ leaf_status,
                          const float* __restrict__ priors, const float* __restrict__ values, double c_puct, double vl,
                          uint64_t* __restrict__ leaf_states, int32_t* __restrict__ leaf_path, uint4* __restrict__ enc_out) {
    __shared__ float s_pri[kWarpsPerBlock][kActionDim];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + w;
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t t = warp; t < A.num_trees; t += nwarps) {
        expand_tree(A, t, K, leaf_node, leaf_status, priors, values, 1, vl, leaf_path, s_pri[w], lane);
        __syncwarp();
        select_tree(A, t, K, c_puct, vl, leaf_node, leaf_status, leaf_states, leaf_path, 0, enc_out, lane);
    }
}

// AdvanceRoots (portable_mcts.cpp:739-768): the child reached by the played action becomes the root and keeps its whole
// subtree (visit counts, value sums, priors, states); everything else of the old tree is dropped.  The reference
// moves a unique_ptr; here the kept subtree is copied into a scratch arena (children blocks stay
// contiguous, one atomicAdd on the scratch bump pointer per block), which is then copied back over the arena prefix --
// a copying collector, so the arena never accumulates dead nodes over a game.  Three passes: (1) one warp per tree
// finds the child that becomes the root and writes the new root; (2) one thread per old NODE decides whether it is kept
// and reserves its children block; (3) one thread per old node copies itself to its new place.  Nothing walks a tree,
// so the cost does not depend on the size of the largest kept subtree.
//   action < 0 or inactive tree : the tree is kept as it is (reference: early return), i.e. copied with its own root
//   reset_mask[t]               : the tree is replaced by a fresh unexpanded root for reset_states[t] (a new game)
//   action not among the root's children : counters[1] |= 2 (the reference throws), tree kept
//   scratch exhausted           : counters[1] |= 1, the affected node is kept as an unexpanded leaf

__global__ void tree_advance_begin_kernel(lzb_tree A, lzb_tree B) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        B.counters[0] = (int32_t)A.num_trees; B.counters[1] = A.counters[1];
        B.counters[2] = A.counters[2]; B.counters[3] = A.counters[3];
        B.counters[4] = A.counters[4]; B.counters[5] = A.counters[5];
        B.counters[6] = 0x7fffffff;
    }
}

__device__ __forceinline__ void copy_node(const lzb_tree& A, int s, const lzb_tree& B, int d, uint32_t info, int parent) {
    B.visit[d] = A.visit[s]; B.value_sum[d] = A.value_sum[s]; B.prior[d] = A.prior[s];
    B.info[d] = info; B.first_child[d] = -1; B.parent[d] = parent;
    store_packed(B.state, d, load_packed(A.state, s));
}

__global__ void __launch_bounds__(kThreads)
tree_advance_kernel(lzb_tree A, lzb_tree B, const int32_t* __restrict__ actions, const uint64_t* __restrict__ reset_states,
                    const uint8_t* __restrict__ reset_mask, int32_t* __restrict__ src_root_out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t t = warp; t < A.num_trees; t += nwarps) {
        const uint32_t root_inf = A.info[t];
        if (reset_mask && reset_mask[t]) {                              // a new game starts in this slot
            if (lane == 0) {
                const Packed p = load_packed(reset_states, t);
                State<int> s;
                unpack(p, s);
                store_packed(B.state, t, p);
                B.visit[t] = 0; B.value_sum[t] = 0.0; B.prior[t] = 1.0; B.first_child[t] = -1; B.parent[t] = -1;
                uint32_t inf = 0xFFu;
                if (game_over(s)) inf |= kInfoTerminal;
                if (s.player == -1) inf |= kInfoWhite;
                B.info[t] = inf;
                B.root_value[t] = 0.0;
                src_root_out[t] = -1;                                       // every node of the old tree is dropped
            }
            continue;
        }
        int src_root = (int)t;
        const int a = actions[t];
        if (!(root_inf & kInfoInactive) && a >= 0) {
            const int n = (root_inf & kInfoExpanded) ? info_nchild(root_inf) : 0;
            const int fc = A.first_child[t];
            int found = -1;
            for (int base = 0; base < n && found < 0; base += 32) {
                const int i = base + lane;
                const bool hit = i < n && (int)(A.info[fc + i] & kInfoActionMask) == a;
                const uint32_t m = __ballot_sync(0xffffffffu, hit);
                if (m) found = base + __ffs(m) - 1;
            }
            if (found >= 0) src_root = fc + found;
            else if (lane == 0) atomicOr(&B.counters[1], kFlagIllegalAdvance);
        }
        const uint32_t src_inf = A.info[src_root];
        if (lane == 0) {
            const uint32_t inf = ((src_inf & ~(kInfoActionMask | kInfoPending | kInfoInactive)) | 0xFFu) | (root_inf & kInfoInactive);
            copy_node(A, src_root, B, (int)t, inf, -1);
            B.root_value[t] = src_root == (int)t ? A.root_value[t] : 0.0;
        }
        if (lane == 0) src_root_out[t] = src_root;
    }
}

// Pass 2 (one THREAD per old node): is the node kept?  It walks its parent chain to the depth-1 ancestor x and the tree t
// (a handful of dependent loads, all 10-20 M nodes in flight at once instead of one latency chain per tree); it is kept
// iff the whole tree is kept (src_root[t] == t) or x is the child that becomes the root.  A kept node with children
// reserves its children block in the new arena (one atomicAdd) and publishes it in remap[]:
//   remap[i] = -2 dropped | -1 kept, no children block | >= 0 first index of its children block in the new arena.
constexpr int kDropped = -2, kNoBlock = -1;

// nodes [0, valid_top) have been written: the bump pointer, cut at the first failed allocation and the capacity
__device__ __forceinline__ int64_t valid_top(const lzb_tree& A) {
    return min(min((int64_t)A.counters[0], (int64_t)A.counters[6]), A.capacity);
}

__device__ __forceinline__ bool node_kept(const lzb_tree& A, const int32_t* __restrict__ src_root, int i, int& tree_out) {
    const int T = (int)A.num_trees;
    int x = i, p = A.parent[x];
    while (p >= T) { x = p; p = A.parent[x]; }
    tree_out = p;
    const int sr = src_root[p];
    return sr == p || sr == x;
}

__global__ void __launch_bounds__(256)
tree_advance_mark_kernel(lzb_tree A, lzb_tree B, const int32_t* __restrict__ src_root, int32_t* __restrict__ remap) {
    const int64_t top = valid_top(A);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int T = (int)A.num_trees;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < top; i += stride) {
        bool kept;
        if (i < T) kept = src_root[i] == (int)i;                        // an old root survives only if its tree is kept whole
        else { int t; kept = node_kept(A, src_root, (int)i, t); }
        int r = kDropped;
        if (kept) {
            const uint32_t inf = A.info[i];
            const int n = (inf & kInfoExpanded) ? info_nchild(inf) : 0;
            r = kNoBlock;
            if (n > 0) {
                const int fc = atomicAdd(&B.counters[0], n);
                if ((int64_t)fc + n > B.capacity) { atomicOr(&B.counters[1], kFlagArena); atomicMin(&B.counters[6], fc); }   // stays a leaf
                else r = fc;
            }
        }
        remap[i] = r;
    }
}

// Pass 3 (one thread per old node): a kept node copies itself to  remap[parent] + (its position among its siblings)
// with its parent's and its children's new indices; the node that becomes the root only hands its block to slot t.
__global__ void __launch_bounds__(256)
tree_advance_copy_kernel(lzb_tree A, lzb_tree B, const int32_t* __restrict__ src_root, const int32_t* __restrict__ remap) {
    const int64_t top = valid_top(A);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int T = (int)A.num_trees;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < top; i += stride) {
        const int r = remap[i];
        if (r == kDropped) continue;
        if (i < T) {                                   // root of a tree that is kept as it is (already copied by pass 1)
            B.first_child[i] = r;
            if (r == kNoBlock && (A.info[i] & kInfoExpanded) && info_nchild(A.info[i]) > 0)
                B.info[i] = B.info[i] & ~(kInfoExpanded | (0xFFu << 8));
            continue;
        }
        int t;
        node_kept(A, src_root, (int)i, t);
        const int sr = src_root[t];
        uint32_t inf = A.info[i] & ~kInfoPending;
        if (r == kNoBlock && (inf & kInfoExpanded) && info_nchild(inf) > 0) inf &= ~(kInfoExpanded | (0xFFu << 8));   // arena full
        if ((int)i == sr) {                            // the new root itself lives in slot t (pass 1); just link its block
            B.first_child[t] = r;
            if (r == kNoBlock && (A.info[i] & kInfoExpanded) && info_nchild(A.info[i]) > 0)
                B.info[t] = B.info[t] & ~(kInfoExpanded | (0xFFu << 8));
            continue;
        }
        const int p = A.parent[i];
        const int pblock = remap[p];
        if (pblock < 0) continue;                      // the parent lost its block (arena full): unreachable, drop
        int p_new;
        if (p == sr) p_new = t;
        else if (p < T) p_new = p;
        else { const int gp = A.parent[p]; p_new = remap[gp] + (p - A.first_child[gp]); }
        const int d = pblock + ((int)i - A.first_child[p]);
        copy_node(A, (int)i, B, d, inf, p_new);
        B.first_child[d] = r;                          // -1 (kNoBlock) or the children block
    }
}

// scratch prefix [0, counters[0]) -> arena (the scratch never holds more nodes than the arena did)
__global__ void __launch_bounds__(256)
tree_copy_back_kernel(lzb_tree B, lzb_tree A) {
    const int64_t n = min(valid_top(B), A.capacity);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t i = tid; i < n; i += stride) {
        A.visit[i] = B.visit[i]; A.value_sum[i] = B.value_sum[i]; A.prior[i] = B.prior[i];
        A.info[i] = B.info[i]; A.first_child[i] = B.first_child[i]; A.parent[i] = B.parent[i];
    }
    const ulonglong2* bs = reinterpret_cast<const ulonglong2*>(B.state);
    ulonglong2* as = reinterpret_cast<ulonglong2*>(A.state);
    for (int64_t i = tid; i < 2 * n; i += stride) as[i] = bs[i];
    for (int64_t i = tid; i < A.num_trees; i += stride) A.root_value[i] = B.root_value[i];
    if (tid < 7) A.counters[tid] = tid == 0 ? (int32_t)n : tid == 6 ? 0x7fffffff : B.counters[tid];
}

// RootOutputs (portable_mcts.cpp:664-737) + RootPriors (:592-624)
__global__ void __launch_bounds__(kThreads)
tree_root_outputs_kernel(lzb_tree A, int32_t* __restrict__ visits, float* __restrict__ qvalues,
                         float* __restrict__ root_values, uint8_t* __restrict__ legal, uint8_t* __restrict__ terminal,
                         float* __restrict__ priors) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t t = warp; t < A.num_trees; t += nwarps) {
        const uint32_t inf = A.info[t];
        const int n = (inf & kInfoExpanded) ? info_nchild(inf) : 0;
        const int fc = A.first_child[t];
        for (int a = lane; a < kActionDim; a += 32) {
            const int64_t o = t * kActionDim + a;
            if (visits) visits[o] = 0;
            if (qvalues) qvalues[o] = 0.0f;
            if (legal) legal[o] = 0;
            if (priors) priors[o] = 0.0f;
        }
        __syncwarp();
        for (int i = lane; i < n; i += 32) {
            const int c = fc + i;
            const uint32_t ci = A.info[c];
            const int64_t o = t * kActionDim + (int)(ci & kInfoActionMask);
            const int vc = A.visit[c];
            if (visits) visits[o] = vc;
            if (legal) legal[o] = 1;
            if (priors) priors[o] = (float)A.prior[c];
            if (qvalues && vc > 0) {
                double q = __ddiv_rn(A.value_sum[c], (double)vc);
                if ((ci ^ inf) & kInfoWhite) q = -q;
                qvalues[o] = (float)q;
            }
        }
        if (lane == 0) {
            if (terminal) terminal[t] = ((inf & kInfoTerminal) || n == 0) ? 1 : 0;
            if (root_values) {
                const int nv = A.visit[t];
                double v;
                if (nv > 0) v = __ddiv_rn(A.value_sum[t], (double)nv);
                else if (inf & kInfoNoLegal) v = -1.0;
                else if (inf & kInfoTerminal) {
                    State<int> s;
                    unpack(load_packed(A.state, t), s);
                    v = (inf & kInfoExpanded) ? A.root_value[t] : terminal_value(s);
                } else v = A.root_value[t];
                root_values[t] = (float)v;
            }
        }
    }
}

// SetRootPriors (portable_mcts.cpp:626-662): prior_c = p[action_c] / sum_children p (fp64, child order)
__global__ void __launch_bounds__(kThreads)
tree_set_root_priors_kernel(lzb_tree A, const float* __restrict__ priors) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t t = warp; t < A.num_trees; t += nwarps) {
        const uint32_t inf = A.info[t];
        const int n = (inf & kInfoExpanded) ? info_nchild(inf) : 0;
        if ((inf & (kInfoTerminal | kInfoInactive)) || n == 0) continue;
        const int fc = A.first_child[t];
        double sum = 0.0;
        if (lane == 0)
            for (int i = 0; i < n; ++i)
                sum = __dadd_rn(sum, (double)priors[t * kActionDim + (int)(A.info[fc + i] & kInfoActionMask)]);
        sum = __shfl_sync(0xffffffffu, sum, 0);
        if (!(sum > 0.0) || isinf(sum)) continue;                     // the reference throws; we keep the old priors
        for (int i = lane; i < n; i += 32)
            A.prior[fc + i] = __ddiv_rn((double)priors[t * kActionDim + (int)(A.info[fc + i] & kInfoActionMask)], sum);
    }
}

// Model input planes straight from packed states (EncodeModelInput :241-265 == encoding.cpp:26-79).
// layout 0: f32 [n,11,6,6] (NCHW);  layout 1: bf16 channels-last, i.e. physical [n,6,6,11].
template <int kLayout>
__global__ void __launch_bounds__(kThreads)
encode_inputs_kernel(const uint64_t* __restrict__ states, int64_t n, void* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t i = warp; i < n; i += nwarps) {
        State<int> s;
        unpack(load_packed(states, i), s);
        const bool black = s.player == 1;
        const uint64_t p0 = black ? s.black : s.white, p1 = black ? s.white : s.black;
        const uint64_t p2 = black ? s.mb : s.mw, p3 = black ? s.mw : s.mb;
        const int phase_plane = 3 + s.phase;
        for (int e = lane; e < 396; e += 32) {
            int plane, cell;
            if (kLayout == 0) { plane = e / 36; cell = e - plane * 36; }
            else { cell = e / 11; plane = e - cell * 11; }
            const uint64_t bits = plane == 0 ? p0 : plane == 1 ? p1 : plane == 2 ? p2 : p3;
            const bool on = plane < 4 ? ((bits >> cell) & 1) : (plane == phase_plane);
            if (kLayout == 0) reinterpret_cast<float*>(out)[i * 396 + e] = on ? 1.0f : 0.0f;
            else reinterpret_cast<uint16_t*>(out)[i * 396 + e] = on ? (uint16_t)0x3F80 : (uint16_t)0;   // bf16 1.0
        }
    }
}

// layout 2: bf16 channels-last padded to 64 channels (physical [n,6,6,64], channels 11..63 zero): the K = 64 input of
// our tcgen05 stem convolution (csrc/lz_conv.cu); 16-byte stores, 8 channels each.
__global__ void __launch_bounds__(kThreads)
encode_inputs_c64_kernel(const uint64_t* __restrict__ states, int64_t n, uint4* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t i = warp; i < n; i += nwarps) encode_c64_row<true>(load_packed(states, i), out + i * 288, lane);
}

// Policy heads -> dense priors over the legal actions of each leaf (masked softmax, fp32) and bucketed value
// head -> scalar (expectation over linspace(-1, 1, bins)): fuses project_policy_logits_fast.cpp:16-164 with
// neural_network.py:201-210 and takes the legal set from the packed state (scalar-engine semantics).
__global__ void __launch_bounds__(kThreads)
heads_to_priors_kernel(const uint64_t* __restrict__ states, int64_t n, const float* __restrict__ log_p1,
                       const float* __restrict__ log_p2, const float* __restrict__ log_pmc,
                       const float* __restrict__ value_logits, int bins, float* __restrict__ priors,
                       float* __restrict__ values) {
    __shared__ float heads[kWarpsPerBlock][3][36];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + w;
    const int64_t nwarps = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t i = warp; i < n; i += nwarps) {
        State<int> s;
        unpack(load_packed(states, i), s);
        Legal L;
        legal_actions<int, true>(s, L, true);
        __syncwarp();
        for (int c = lane; c < 36; c += 32) {
            heads[w][0][c] = log_p1[i * 36 + c]; heads[w][1][c] = log_p2[i * 36 + c]; heads[w][2][c] = log_pmc[i * 36 + c];
        }
        __syncwarp();
        float logit[7], mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < 7; ++k) {
            const int a = lane + 32 * k;
            float v = -INFINITY;
            if (a < kActionDim && legal_test(L, a)) {
                if (a < 36) v = heads[w][0][a];
                else if (a < 180) {
                    const int from = (a - 36) >> 2, d = (a - 36) & 3;
                    v = heads[w][1][from] + heads[w][0][from + (d == 0 ? -6 : d == 1 ? 6 : d == 2 ? -1 : 1)];
                } else if (a < 216) v = heads[w][2][a - 180];
                else v = 0.0f;
            }
            logit[k] = v;
            mx = fmaxf(mx, v);
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
            const int a = lane + 32 * k;
            if (a < kActionDim) priors[i * kActionDim + a] = ok ? e[k] / sum : 0.0f;
        }
        // value = sum softmax(logits) * linspace(-1, 1, bins)
        float vmx = -INFINITY;
        for (int b = lane; b < bins; b += 32) vmx = fmaxf(vmx, value_logits[i * bins + b]);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) vmx = fmaxf(vmx, __shfl_xor_sync(0xffffffffu, vmx, off));
        float se = 0.0f, sc = 0.0f;
        const float step = bins > 1 ? 2.0f / (float)(bins - 1) : 0.0f;
        for (int b = lane; b < bins; b += 32) {
            const float ev = expf(value_logits[i * bins + b] - vmx);
            se += ev; sc += ev * (-1.0f + step * (float)b);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            se += __shfl_xor_sync(0xffffffffu, se, off);
            sc += __shfl_xor_sync(0xffffffffu, sc, off);
        }
        if (lane == 0) values[i] = sc / se;
    }
}

}  // namespace
}  // namespace lzb

using namespace lzb;

static int check_tree(const lzb_tree* t) {
    LZB_REQUIRE(t && t->visit && t->value_sum && t->prior && t->info && t->first_child && t->parent && t->state &&
                t->counters && t->root_value, "tree arena has null arrays");
    LZB_REQUIRE(t->num_trees > 0 && t->capacity >= t->num_trees && t->capacity < (1LL << 31), "bad tree sizes");
    return LZB_OK;
}

extern "C" int lzb_tree_init_roots(const lzb_tree* tree, const uint64_t* root_states, const uint8_t* active, void* stream) {
    int rc = check_tree(tree);
    if (rc) return rc;
    LZB_REQUIRE(root_states, "null root states");
    tree_init_kernel<<<thread_grid(tree->num_trees), kThreads, 0, (cudaStream_t)stream>>>(*tree, root_states, active);
    return check_launch("tree_init_kernel");
}

extern "C" int lzb_tree_select(const lzb_tree* tree, int32_t K, double c_puct, double virtual_loss, int32_t* leaf_node,
                               int32_t* leaf_status, uint64_t* leaf_states, int32_t* leaf_path, int32_t roots_only,
                               void* inputs_c64, void* stream) {
    int rc = check_tree(tree);
    if (rc) return rc;
    LZB_REQUIRE(K >= 1 && K <= 64, "leaves per tree per wave must be in [1, 64]");
    LZB_REQUIRE(c_puct >= 0.0 && c_puct == c_puct, "exploration_weight must be finite and non-negative");
    LZB_REQUIRE(leaf_node && leaf_status && leaf_states, "null output");
    LZB_REQUIRE(!roots_only || K == 1, "prepare_roots uses one slot per tree");
    LZB_REQUIRE((reinterpret_cast<uintptr_t>(inputs_c64) & 15) == 0, "inputs must be 16-byte aligned");
    tree_select_kernel<<<warp_grid(tree->num_trees), kThreads, 0, (cudaStream_t)stream>>>(
        *tree, K, c_puct, roots_only ? 0.0 : virtual_loss, leaf_node, leaf_status, leaf_states, roots_only ? nullptr : leaf_path,
        roots_only ? 1 : 0, reinterpret_cast<uint4*>(inputs_c64));
    return check_launch("tree_select_kernel");
}

extern "C" int lzb_tree_advance_roots(const lzb_tree* tree, const lzb_tree* scratch, const int32_t* actions,
                                      const uint64_t* reset_states, const uint8_t* reset_mask, int32_t* work,
                                      void* stream) {
    int rc = check_tree(tree);
    if (rc) return rc;
    rc = check_tree(scratch);
    if (rc) return rc;
    LZB_REQUIRE(scratch->num_trees == tree->num_trees && scratch->capacity >= tree->num_trees, "scratch arena mismatch");
    LZB_REQUIRE(scratch->visit != tree->visit && scratch->state != tree->state, "scratch arena must not alias the tree");
    LZB_REQUIRE(actions && work, "null actions / work array");
    LZB_REQUIRE((reset_states == nullptr) == (reset_mask == nullptr), "reset_states and reset_mask go together");
    cudaStream_t st = (cudaStream_t)stream;
    tree_advance_begin_kernel<<<1, 32, 0, st>>>(*tree, *scratch);
    int32_t* src_root = work;                          // [num_trees]
    int32_t* remap = work + tree->num_trees;           // [capacity]
    tree_advance_kernel<<<warp_grid(tree->num_trees), kThreads, 0, st>>>(*tree, *scratch, actions, reset_states, reset_mask,
                                                                        src_root);
    tree_advance_mark_kernel<<<148 * 8, 256, 0, st>>>(*tree, *scratch, src_root, remap);
    tree_advance_copy_kernel<<<148 * 8, 256, 0, st>>>(*tree, *scratch, src_root, remap);
    tree_copy_back_kernel<<<148 * 8, 256, 0, st>>>(*scratch, *tree);
    return check_launch("tree_advance_kernel");
}

extern "C" int lzb_tree_expand_backup(const lzb_tree* tree, int32_t K, const int32_t* leaf_node,
                                      const int32_t* leaf_status, const float* priors, const float* values,
                                      int32_t do_backup, double virtual_loss, const int32_t* leaf_path, void* stream) {
    int rc = check_tree(tree);
    if (rc) return rc;
    LZB_REQUIRE(K >= 1 && K <= 64, "leaves per tree per wave must be in [1, 64]");
    LZB_REQUIRE(leaf_node && leaf_status && priors && values, "null input");
    tree_expand_kernel<<<warp_grid(tree->num_trees), kThreads, 0, (cudaStream_t)stream>>>(
        *tree, K, leaf_node, leaf_status, priors, values, do_backup, virtual_loss, leaf_path);
    return check_launch("tree_expand_kernel");
}

extern "C" int lzb_tree_expand_select(const lzb_tree* tree, int32_t K, int32_t* leaf_node, int32_t* leaf_status,
                                      const float* priors, const float* values, double c_puct, double virtual_loss,
                                      uint64_t* leaf_states, int32_t* leaf_path, void* inputs_c64, void* stream) {
    int rc = check_tree(tree);
    if (rc) return rc;
    LZB_REQUIRE(K >= 1 && K <= 64, "leaves per tree per wave must be in [1, 64]");
    LZB_REQUIRE(c_puct >= 0.0 && c_puct == c_puct, "exploration_weight must be finite and non-negative");
    LZB_REQUIRE(leaf_node && leaf_status && priors && values && leaf_states && leaf_path, "null pointer");
    LZB_REQUIRE((reinterpret_cast<uintptr_t>(inputs_c64) & 15) == 0, "inputs must be 16-byte aligned");
    tree_expand_select_kernel<<<warp_grid(tree->num_trees), kThreads, 0, (cudaStream_t)stream>>>(
        *tree, K, leaf_node, leaf_status, priors, values, c_puct, virtual_loss, leaf_states, leaf_path,
        reinterpret_cast<uint4*>(inputs_c64));
    return check_launch("tree_expand_select_kernel");
}

extern "C" int lzb_tree_root_outputs(const lzb_tree* tree, int32_t* visits, float* qvalues, float* root_values,
                                     uint8_t* legal, uint8_t* terminal, float* priors, void* stream) {
    int rc = check_tree(tree);
    if (rc) return rc;
    tree_root_outputs_kernel<<<warp_grid(tree->num_trees), kThreads, 0, (cudaStream_t)stream>>>(
        *tree, visits, qvalues, root_values, legal, terminal, priors);
    return check_launch("tree_root_outputs_kernel");
}

extern "C" int lzb_tree_set_root_priors(const lzb_tree* tree, const float* priors, void* stream) {
    int rc = check_tree(tree);
    if (rc) return rc;
    LZB_REQUIRE(priors, "null priors");
    tree_set_root_priors_kernel<<<warp_grid(tree->num_trees), kThreads, 0, (cudaStream_t)stream>>>(*tree, priors);
    return check_launch("tree_set_root_priors_kernel");
}

extern "C" int lzb_encode_inputs_packed(const uint64_t* states, int64_t n, int32_t layout, void* out, void* stream) {
    LZB_REQUIRE(n >= 0 && (layout == 0 || layout == 1 || layout == 2), "bad arguments");
    if (n == 0) return LZB_OK;
    LZB_REQUIRE(states && out, "null pointer");
    if (layout == 2) {
        LZB_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "out must be 16-byte aligned");
        encode_inputs_c64_kernel<<<warp_grid(n), kThreads, 0, (cudaStream_t)stream>>>(states, n, reinterpret_cast<uint4*>(out));
        return check_launch("encode_inputs_c64_kernel");
    }
    if (layout == 0) encode_inputs_kernel<0><<<warp_grid(n), kThreads, 0, (cudaStream_t)stream>>>(states, n, out);
    else encode_inputs_kernel<1><<<warp_grid(n), kThreads, 0, (cudaStream_t)stream>>>(states, n, out);
    return check_launch("encode_inputs_kernel");
}

extern "C" int lzb_heads_to_priors(const uint64_t* states, int64_t n, const float* log_p1, const float* log_p2,
                                   const float* log_pmc, const float* value_logits, int32_t bins, float* priors,
                                   float* values, void* stream) {
    LZB_REQUIRE(n >= 0 && bins >= 1, "bad arguments");
    if (n == 0) return LZB_OK;
    LZB_REQUIRE(states && log_p1 && log_p2 && log_pmc && value_logits && priors && values, "null pointer");
    heads_to_priors_kernel<<<warp_grid(n), kThreads, 0, (cudaStream_t)stream>>>(states, n, log_p1, log_p2, log_pmc,
                                                                               value_logits, bins, priors, values);
    return check_launch("heads_to_priors_kernel");
}
