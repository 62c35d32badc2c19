/*
 * liuzhou_b200.h -- C ABI of libliuzhou_b200.so: hand-written sm_100a kernels for the Liuzhou Chess
 * (六洲棋) batched-MCTS self-play hot path.
 *
 * Drop-in boundary: every entry point below replaces one function of the reference's `v0_core` torch
 * extension (pybind11 module, /root/reference/v0/src/bindings/module.cpp:874-1482) or one step of its
 * v1 wave loop; the Python shim `liuzhou_b200.v0_core` presents them under the reference's names,
 * argument order and dtypes.  See INTEGRATION.md for the binding a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers + sizes, no torch types; all data pointers are DEVICE pointers on the current
 *     device unless the parameter is named h_*;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); launches are
 *     asynchronous on it; no global mutable state, re-entrant from several host threads;
 *   - return value: 0 = LZB_OK, negative = error (lzb_last_error() gives a thread-local message);
 *     the Python shim raises RuntimeError like TORCH_CHECK does in the reference;
 *   - reference tensor layout ("SoA of bytes", v1/python/mcts_gpu.py:40-55): board int8[B,36]
 *     (+1 black, -1 white, 0 empty), marks_black / marks_white bool(uint8)[B,36], nine int64[B] scalars;
 *   - native layout: one game state = 4 x uint64 (32 B) packed bitboards, see lzb_pack_states.
 */
#ifndef LIUZHOU_B200_H
#define LIUZHOU_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define LZB_API __attribute__((visibility("default")))
#else
#define LZB_API
#endif

#define LZB_OK 0
#define LZB_ERR_INVALID_ARGUMENT (-1)
#define LZB_ERR_CUDA (-2)
#define LZB_ERR_CAPACITY (-3)

#define LZB_ACTION_DIM 220
#define LZB_STATE_WORDS 4 /* uint64 words per packed state */

/* Reference tensor layout of a state batch (12 tensors). move_count / moves_since_capture may be NULL
 * where the reference op does not take them (encode_actions_fast, states_to_model_input). */
typedef struct {
    const int8_t *board;          /* [B,36] */
    const uint8_t *marks_black;   /* [B,36] */
    const uint8_t *marks_white;   /* [B,36] */
    const int64_t *phase, *current_player;
    const int64_t *pending_marks_required, *pending_marks_remaining;
    const int64_t *pending_captures_required, *pending_captures_remaining;
    const int64_t *forced_removals_done, *move_count, *moves_since_capture;
} lzb_states_in;

typedef struct {
    int8_t *board;
    uint8_t *marks_black, *marks_white;
    int64_t *phase, *current_player;
    int64_t *pending_marks_required, *pending_marks_remaining;
    int64_t *pending_captures_required, *pending_captures_remaining;
    int64_t *forced_removals_done, *move_count, *moves_since_capture;
} lzb_states_out;

LZB_API const char *lzb_last_error(void);
/* ABI / build identification: returns e.g. "liuzhou_b200 0.1 sm_100a". */
LZB_API const char *lzb_version(void);
/* Number of kernels this library has launched in this process (bench.py's gpu_launches). */
LZB_API uint64_t lzb_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * (a2) legal mask -- replaces v0_core.encode_actions_fast
 *      reference: v0/src/game/fast_legal_mask_cuda.cu:282-404 (kernel), :406-485 (launcher),
 *                 binding module.cpp:1294-1310.
 * mask u8[B,T], metadata i32[B,T,4] with T = sum of the four dims; fully written (no pre-fill needed).
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_encode_actions_fast(const lzb_states_in *st, int64_t B, int64_t placement_dim, int64_t movement_dim,
                            int64_t selection_dim, int64_t auxiliary_dim, uint8_t *mask, int32_t *metadata,
                            void *stream);

/* ------------------------------------------------------------------------------------------------
 * (a4) apply move -- replaces v0_core.batch_apply_moves / batch_apply_moves_inplace
 *      reference: v0/src/game/fast_apply_moves_cuda.cu:548-744 / :746-917, binding module.cpp:1311-1327.
 * action_codes i32[N,4] = (kind, primary, secondary, extra) rows as emitted in `metadata`;
 * parent_indices / slot_indices i64[N].  Illegal actions are silent no-ops exactly like the reference
 * CUDA kernel (move_count still advances for every kind except placement).
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_batch_apply_moves(const lzb_states_in *parents, int64_t B, const int32_t *action_codes,
                          const int64_t *parent_indices, int64_t N, const lzb_states_out *children, void *stream);
LZB_API int lzb_batch_apply_moves_inplace(const lzb_states_out *states, int64_t B, const int32_t *action_codes,
                                  const int64_t *slot_indices, int64_t N, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (a6) states_to_model_input -- v0/src/net/encoding.cpp:26-79, binding module.cpp:1286-1293.
 * out f32[B,11,6,6].
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_states_to_model_input(const lzb_states_in *st, int64_t B, float *out, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (a7) project_policy_logits_fast -- v0/src/net/project_policy_logits_fast.cpp:16-164,
 *      binding module.cpp:1328-1338.  fp32 heads [B,36]; legal_mask u8[B,220];
 *      probs f32[B,220], masked_logits f32[B,220].
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_project_policy_logits_fast(const float *log_p1, const float *log_p2, const float *log_pmc,
                                   const uint8_t *legal_mask, int64_t B, float *probs, float *masked_logits,
                                   void *stream);

/* ------------------------------------------------------------------------------------------------
 * (a9) root-PUCT -- replaces v0_core.root_puct_allocate_visits
 *      reference: v0/src/mcts/root_puct_fused.cu:12-183, binding module.cpp:1349-1356.
 * priors / leaf_values f32[R,M], valid_mask u8[R,M] -> visits f32[R,M], value_sum f32[R,M],
 * root_values f32[R].  One warp per root, N/W/P in registers, warp-shuffle argmax (ties -> lowest index).
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_root_puct_allocate_visits(const float *priors, const float *leaf_values, const uint8_t *valid_mask,
                                  int64_t R, int64_t M, int64_t num_simulations, float exploration_weight,
                                  float *visits, float *value_sum, float *root_values, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (a8) root_pack_sparse_actions -- module.cpp:258-363.  Two calls because the output shapes (R, M, N)
 * are data dependent (the reference syncs on `.item()` at :310 as well):
 *   1. lzb_root_pack_count: row_counts i64[B], terminal_mask u8[B], root_rank i64[B] (index among valid
 *      roots), flat_offset i64[B] (exclusive prefix of counts over valid roots), summary i64[3] = {R, M, N};
 *   2. host reads `summary`, allocates, then lzb_root_pack_fill writes the padded [R,M] matrices and the
 *      flat [N] child list.
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_root_pack_count(const uint8_t *legal_mask, int64_t B, int64_t A, int64_t *row_counts, uint8_t *terminal_mask,
                        int64_t *root_rank, int64_t *flat_offset, int64_t *summary, void *stream);
LZB_API int lzb_root_pack_fill(const uint8_t *legal_mask, const float *probs, const int32_t *metadata, int64_t B, int64_t A,
                       const int64_t *row_counts, const int64_t *root_rank, const int64_t *flat_offset, int64_t R,
                       int64_t M, int64_t *valid_root_indices, int64_t *counts, uint8_t *valid_mask,
                       int64_t *legal_index_mat, float *priors_mat, int32_t *action_code_mat, int64_t *flat_indices,
                       int32_t *action_codes_all, int64_t *parent_indices_all, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (a10) root_finalize_from_visits (sample_moves = false) -- module.cpp:441-535.
 * Outputs cover all `batch_size` rows (rows that are not valid roots get zeros / -1 / false).
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_root_finalize_from_visits(const int64_t *legal_index_mat, const int32_t *action_code_mat,
                                  const uint8_t *valid_mask, const float *visits, const float *value_sum,
                                  const int64_t *valid_root_indices, int64_t R, int64_t M, int64_t batch_size,
                                  int64_t total_action_dim, const float *root_temperatures, float *policy_dense,
                                  int64_t *chosen_action_indices, int32_t *chosen_action_codes,
                                  uint8_t *chosen_valid_mask, float *root_value, void *stream);

/* (a10) root_sparse_writeback -- module.cpp:365-439: scatter an externally supplied legal policy f32[R,M] (x valid_mask)
 * and the column picked per root (local_picks i64[R]) back to dense rows; same output convention as above. */
LZB_API int lzb_root_sparse_writeback(const int64_t *legal_index_mat, const int32_t *action_code_mat,
                                      const uint8_t *valid_mask, const float *legal_policy, const int64_t *local_picks,
                                      const int64_t *valid_root_indices, int64_t R, int64_t M, int64_t batch_size,
                                      int64_t total_action_dim, float *policy_dense, int64_t *chosen_action_indices,
                                      int32_t *chosen_action_codes, uint8_t *chosen_valid_mask, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (a14) self_play_step_inplace -- module.cpp:632-871.  Mutates the 12 state tensors, plies, done.
 * Output buffers must hold K entries; *num_finalized (device i64) receives F.  Order of the F entries:
 * immediate-done slots in active order, then finished-by-move slots in active order (as the reference).
 * scratch: K * 16 bytes.
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_self_play_step_inplace(const lzb_states_out *states, int64_t B, int64_t *plies, uint8_t *done,
                               const int64_t *active_idx, const int32_t *chosen_action_codes,
                               const uint8_t *terminal_mask, const uint8_t *chosen_valid_mask, int64_t K,
                               int64_t max_game_plies, float soft_value_k, int64_t *finalize_slots,
                               float *result_from_black, float *soft_value_from_black, int64_t *num_finalized,
                               void *scratch, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (a15) finalize_trajectory_inplace -- module.cpp:547-630.
 * final_slots / final_counts hold F entries; summary i64[4] = {kept, black wins, white wins, draws}.
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_finalize_trajectory_inplace(float *value_targets, float *soft_value_targets, const int8_t *player_signs,
                                    const int64_t *step_index_matrix, int64_t G, int64_t T, const int64_t *step_counts,
                                    const int64_t *slots, const float *result_from_black,
                                    const float *soft_value_from_black, int64_t F, int64_t *final_slots,
                                    int64_t *final_counts, int64_t *summary, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Native packed layout (a1): state i = packed[4*i .. 4*i+3]
 *   w0 = black(36 bits) | meta << 36, w1 = white, w2 = marks_black, w3 = marks_white
 *   meta = phase:3 | white_to_move:1 | forced:2 | pm_req:2 | pm_rem:2 | pc_req:2 | pc_rem:2 |
 *          move_count:8 | moves_since_capture:6
 * Replaces v0::TensorStateBatch conversions (v0/src/game/tensor_state_batch.cpp) at the boundary.
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_pack_states(const lzb_states_in *st, int64_t B, uint64_t *packed, void *stream);
LZB_API int lzb_unpack_states(const uint64_t *packed, int64_t B, const lzb_states_out *st, void *stream);
LZB_API int lzb_init_states(uint64_t *packed, int64_t B, void *stream);

/* Native legal mask: 220-bit masks as 4 x uint64 per state (bit a of word a/64) + legal counts i32[B].
 * scalar_semantics != 0 -> v0::GenerateAllLegalMoves (empty on game over), else encode_actions_fast. */
LZB_API int lzb_legal_masks_packed(const uint64_t *packed, int64_t B, int scalar_semantics, uint64_t *mask_words,
                           int32_t *counts, void *stream);
/* Native apply by 220-d action index: children[i] = apply(parents[parent_indices[i]], actions[i]);
 * parent_indices may be NULL (identity). In place if children == parents and parent_indices == NULL. */
LZB_API int lzb_apply_actions_packed(const uint64_t *parents, const int64_t *parent_indices, const int32_t *actions, int64_t N,
                             uint64_t *children, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Config-2 workload: uniform-random playouts on the scalar-engine rules, counter-based RNG
 * pick = mulhi32(mix64(mix64(seed ^ game*K) + ply) >> 32, n)   (same function in oracle/lz_oracle.c).
 * lzb_playout_run advances every unfinished game by up to `max_steps` plies inside one launch (state
 * lives in registers); result i8[B]: 2 = running, else result_from_black (+1, -1, 0).
 * plies i32[B] counts plies played; hash u64[B] chains mix64(hash ^ state_hash) per ply (optional).
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_playout_run(uint64_t *packed, int32_t *plies, int8_t *result, uint64_t *hash, int64_t B, uint64_t seed,
                    uint64_t game_offset, int32_t max_steps, int32_t max_game_plies, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (a12/a13) Device-resident full-tree MCTS -- replaces the reference's CPU `PortableTreeBatch`
 *      (v1/cpp/portable_mcts.cpp:437-977; protocol prepare_roots -> complete_pending -> select_leaves ->
 *      ... -> root_outputs, bound at :1069-1112) and the v0 `MCTSCore` virtual-loss batching
 *      (v0/src/mcts/mcts_core.cpp:252-268,640-701).
 * Node arena (structure of arrays, `capacity` nodes; nodes [0, num_trees) are the roots):
 *   visit i32 | value_sum f64 | prior f64 | info u32 (action:8 | nchild:8 | flags) | first_child i32 |
 *   parent i32 | state u64[4] | root_value f64[num_trees] | counters i32[8] = {top, sticky flags
 *   (see lzb_tree_advance_roots), expansions, terminal hits, sibling records scanned by select, levels descended,
 *   arena index of the first failed allocation (INT32_MAX if none: nodes above it were never written), reserved}.
 * One warp per tree; K leaves per tree per wave (K = 1 reproduces the reference exactly).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t *visit;
    double *value_sum;
    double *prior;
    uint32_t *info;
    int32_t *first_child;
    int32_t *parent;
    uint64_t *state;
    double *root_value;
    int32_t *counters;
    int64_t capacity;
    int64_t num_trees;
    /* optional i32[num_trees] (NULL = identity): leaf-batch row of tree t in the simulation waves (slots
     * tree_rows[t]*K .. +K-1 of leaf_node / leaf_status / leaf_states / leaf_path / inputs / priors / values);
     * tree_rows[t] < 0 = the tree sits this wave out (a finished game).  The live trees' leaves then form a dense prefix
     * of the batch, so the network runs on ceil64(live) rows instead of num_trees.  prepare_roots and the root expansion
     * (do_backup = 0) always use row t. */
    const int32_t *tree_rows;
} lzb_tree;

/* Reset the arena to `num_trees` unexpanded roots (PortableTreeBatch ctor, :443-459). active u8[T] or NULL. */
LZB_API int lzb_tree_init_roots(const lzb_tree *tree, const uint64_t *root_states, const uint8_t *active, void *stream);
/* select_leaves (:515-552) or, with roots_only = 1, prepare_roots (:483-513).  Per slot (tree*K + k): leaf_node i32
 * (-1 if none), leaf_status i32 (0 = evaluate, 1 = terminal/inactive, already backed up, 2 = duplicate of a pending leaf),
 * leaf_states u64[.,4].
 * leaf_path i32[slots][LZB_TREE_PATH_STRIDE] (optional, may be NULL): the descent's node path ([0,32) node per depth,
 * [32] depth or -1 if deeper than 32, [33] colour bits) so that lzb_tree_expand_backup can back up the whole path in
 * one memory round trip instead of walking the parent chain.
 * roots_only = 1 (requires K = 1; leaf_path and virtual_loss are ignored, and exploration_weight has no effect because
 * nothing is descended): one slot per tree; only an UNEXPANDED, non-terminal, active root becomes a pending leaf
 * (status 0) -- a root that kept its subtree through lzb_tree_advance_roots is left alone (status 1).
 * inputs_c64 (optional, may be NULL; 16-byte aligned): bf16 [slots,6,6,64] channels-last; the kernel also writes the
 * network input of every status-0 slot, the planes of lzb_encode_inputs_packed layout 2, which saves a separate
 * encoding launch per simulation wave.  Only channels 0..15 of those rows are written: channels 16..63 must already be
 * zero (the caller zero-fills the buffer once), and the rows of all other slots are left untouched. */
#define LZB_TREE_PATH_STRIDE 34
LZB_API int lzb_tree_select(const lzb_tree *tree, int32_t K, double exploration_weight, double virtual_loss,
                            int32_t *leaf_node, int32_t *leaf_status, uint64_t *leaf_states, int32_t *leaf_path,
                            int32_t roots_only, void *inputs_c64, void *stream);
/* advance_roots (:739-768) + the start of new games, with subtree reuse: for every tree the child reached by
 * actions[t] (i32, an action index in [0,220)) becomes the root and keeps its subtree; actions[t] < 0 or an inactive
 * tree keeps the tree unchanged; reset_mask[t] != 0 (optional, with reset_states u64[T,4]) replaces the tree by a
 * fresh unexpanded root.  The kept subtrees are compacted into `scratch` (a second arena with its own arrays,
 * capacity >= the nodes kept) by node-parallel passes and copied back, so the arena holds no dead nodes afterwards.
 * work: i32[num_trees + capacity] temporary (new root per tree, children-block remap per old node).
 * Sticky flags in counters[1]: 1 arena/scratch exhausted (the node is kept as an unexpanded leaf), 2 action is not a
 * child of the root (the reference throws), 4 a network value was NaN/Inf or a legal prior negative/NaN/Inf (the
 * reference throws in CompletePending / Expand; here the leaf stays unexpanded and nothing is backed up). */
LZB_API int lzb_tree_advance_roots(const lzb_tree *tree, const lzb_tree *scratch, const int32_t *actions,
                                   const uint64_t *reset_states, const uint8_t *reset_mask, int32_t *work, void *stream);
/* complete_pending (:554-590): expand every status-0 leaf with dense priors f32[T*K,220] / values f32[T*K],
 * then back up (do_backup = 0 for roots, :575). */
LZB_API int lzb_tree_expand_backup(const lzb_tree *tree, int32_t K, const int32_t *leaf_node, const int32_t *leaf_status,
                                   const float *priors, const float *values, int32_t do_backup, double virtual_loss,
                                   const int32_t *leaf_path, void *stream);
/* complete_pending of wave w + select_leaves of wave w + 1 in ONE launch (trees are independent, so each warp expands,
 * backs up and descends again without a grid-wide barrier): same arguments as the two calls; leaf_node / leaf_status /
 * leaf_states / leaf_path are read (wave w) and then rewritten (wave w + 1); inputs_c64 (optional, may be NULL) receives
 * the new leaves' network input as in lzb_tree_select, with the same zero-padding precondition. */
LZB_API int lzb_tree_expand_select(const lzb_tree *tree, int32_t K, int32_t *leaf_node, int32_t *leaf_status,
                                   const float *priors, const float *values, double exploration_weight, double virtual_loss,
                                   uint64_t *leaf_states, int32_t *leaf_path, void *inputs_c64, void *stream);
/* root_outputs + root_priors (:592-624,:664-737); any output pointer may be NULL. */
LZB_API int lzb_tree_root_outputs(const lzb_tree *tree, int32_t *visit_counts, float *root_action_values,
                                  float *root_values, uint8_t *legal_masks, uint8_t *terminal, float *root_priors,
                                  void *stream);
/* set_root_priors (:626-662): renormalises priors f32[T,220] over each root's children. */
LZB_API int lzb_tree_set_root_priors(const lzb_tree *tree, const float *priors, void *stream);

/* Model-input planes from packed states (a6 on the native layout): layout 0 = f32 [n,11,6,6];
 * layout 1 = bf16 channels-last ([n,6,6,11] physical) ready for the bf16 network; layout 2 = the same padded to 64
 * channels ([n,6,6,64] physical, channels 11..63 zero): the K = 64 operand of our tcgen05 stem convolution. */
LZB_API int lzb_encode_inputs_packed(const uint64_t *states, int64_t n, int32_t layout, void *out, void *stream);
/* Fused a7 + value decode on packed states: fp32 heads [n,36] x3 + value logits [n,bins] ->
 * priors f32[n,220] (softmax over the scalar-engine legal set) and values f32[n]. */
LZB_API int lzb_heads_to_priors(const uint64_t *states, int64_t n, const float *log_p1, const float *log_p2,
                                const float *log_pmc, const float *value_logits, int32_t bins, float *priors,
                                float *values, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (a17 glue) Fused elementwise epilogues around the network's cuDNN convolutions, bf16 channels-last
 * (replaces PyTorch's separate eval-BatchNorm / ReLU / residual-add passes of
 * src/neural_network.py:83-96,250-254):
 *   v == NULL : out_act = relu(scale * u + shift)
 *   v != NULL : sum = u + v (stored to out_sum if non-NULL) ; out_act = relu(scale * sum + shift)
 * u, v, out_* bf16[rows, channels]; scale / shift f32[channels] (BatchNorm folded: scale = w / sqrt(var + eps),
 * shift = b - mean * scale).
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_bn_relu_bf16(const void *u, const void *v, const float *scale, const float *shift, int64_t rows,
                             int32_t channels, void *out_sum, void *out_act, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (a17) The network's convolutions as hand-written tcgen05 implicit GEMMs with the pre-activation-ResNet
 * epilogue fused in (replaces F.conv2d + eval BatchNorm + ReLU + residual add of PreActResBlock,
 * src/neural_network.py:83-96,250-254; csrc/lz_conv.cu).
 *   x bf16 [n,6,6,cin] channels-last, w bf16 [taps][128][cin] (tap = ky*3+kx; BatchNorm that follows the conv
 *   folded into w / bias), cin = 128 or 64, taps = 9 (3x3, pad 1) or 1 (1x1), n a multiple of 64.
 *   v    = conv(x, w) + bias (+ residual) ; optional ReLU (relu1)
 *   out1 = bf16(v)                                   (may be NULL)
 *   out2 = bf16(relu(scale * float(out1) + shift))   (may be NULL)
 * ---------------------------------------------------------------------------------------------- */
LZB_API int lzb_conv_bf16(const void *x, const void *w, int64_t n, int32_t cin, int32_t taps, const float *bias,
                          const void *residual, const float *scale, const float *shift, int32_t relu1, void *out1,
                          void *out2, void *stream);

/* The whole ChessNet trunk + the heads' 1x1 convolution as ONE persistent kernel (csrc/lz_trunk.cu): replaces the stem
 * conv, the 2 x blocks residual-block convs with their BatchNorm / ReLU / residual adds, and PolicyHead.conv1 +
 * ValueHead.conv1 with their BatchNorm + ReLU (src/neural_network.py:83-96,98-151,213-259).  Activations stay in shared
 * memory / tensor memory across all layers; the residual stream is kept in fp32.
 * planes bf16 [n,6,6,64] (lzb_encode_inputs_packed layout 2; channels 16..63 MUST be zero -- the stem only multiplies the
 * first 16 channels, the network has 11); w_stem bf16 [9][128][64]; w_trunk bf16 [2*blocks*9+1][128][128]
 * (conv1_0, conv2_0, ..., heads 1x1; tap-major, K-major rows, BatchNorm folded where it follows a conv); params f32 in
 * DEVICE memory, compact: stem bias | scale | shift (384), per block conv1 bias (128) + conv2 scale | shift (256), heads
 * conv bias (128) -- copied to constant memory in stream order at every launch; blocks <= 10; out bf16 [n,6,6,128]. */
LZB_API int lzb_trunk_bf16(const void *planes, int64_t n, const void *w_stem, const void *w_trunk, const float *params,
                           int32_t blocks, void *out, void *stream);

/* Fused network heads: everything of PolicyHead / ValueHead after their 1x1 convolutions
 * (src/neural_network.py:98-151: global pooling, gpool_linear, bn2 + relu, the three output convs,
 * log-softmax, value MLP) + bucket expectation (:201-210) + masked softmax over the legal actions of the
 * packed state (project_policy_logits_fast.cpp:16-164) in one kernel.
 * pv bf16[n,36,pc+vc] = relu(bn1(conv1x1)) of both heads (policy channels first); weights fp32, transposed:
 * wout[3][pc] plain; the three dense layers (gpool_linear [3pc -> pc], fc1 [3vc -> mlp], fc2 [mlp -> bins]) come
 * pre-packed in mma.sync m16n8k8 B-fragment order, TF32-rounded: w*_t = float2[ceil(N/8)][ceil(K/8)][32] with
 * element (nt, ks, lane) = (W[n][k], W[n][k + 4]), n = nt*8 + lane/4, k = ks*8 + lane%4, zero outside [N) x [K)
 * (liuzhou_b200.net.pack_mma_b builds it from the nn.Linear weight [N][K]). Any output may be NULL:
 * priors f32[n,220] (needs states), values f32[n], log_heads f32[n,3,36], value_logits f32[n,bins]. */
LZB_API int lzb_heads_tail(const void *pv, int64_t n, int32_t pc, int32_t vc, int32_t mlp, int32_t bins,
                           const float *wgl_t, const float *bn2_scale, const float *bn2_shift, const float *wout,
                           const float *wfc1_t, const float *bfc1, const float *wfc2_t, const float *bfc2,
                           const uint64_t *states, float *priors, float *values, float *log_heads,
                           float *value_logits, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Refilling self-play actor (csrc/lz_actor.cu, liuzhou_b200/actor.py): per-slot game arenas of fixed rows and a
 * linear output of finished games.  Row format = liuzhou_b200.compact.compact_rows_fixed (42 x i64 = 336 B): words
 * 0..3 boards of the side to move + phase << 36, 4..7 legal bits, 8..39 64 x f32 policy in ascending legal order,
 * 40 value | soft value (f32 pair), 41 flags (bit 0 = not representable).
 * Arena row of (slot g, ply p) = g * max_plies + p; signs i8 / actions i16 arenas are indexed the same way.
 * ctl u64[48]: [0] output row cursor, [1] output game cursor, [2] next game serial, [3] sticky overflow flags
 * (1 output capacity, 2 arena), [4] OR of the flags words emitted, [5] block ticket (0 between launches),
 * [6..8] black wins / white wins / draws, [9..46) games by piece delta (black - white) clamped to [-18, 18].
 *
 * lzb_actor_record: for every slot with active[g] != 0, the row of the state BEFORE its move: planes and the
 * encode_actions_fast legal bits of states u64[G,4], the policy row f32[G,220], value words NaN; signs = +1 black /
 * -1 white to move; actions = chosen i64[G] (-1 = no move); nrows i32[G] (rows of the game so far) += 1.
 * lzb_actor_emit: for every slot with finished[g] != 0, in ascending slot order: its nrows[g] rows with word 40 =
 * (sign * result[g], sign * soft[g]) (f32 products; result / soft from black's perspective) are appended at the row
 * cursor of out_rows i64[capacity,42] with 16-byte copies, their actions at the same rows of out_actions
 * i16[capacity], and one record i64[8] = {serial, slot, length, first output row, step, piece delta of states u64[G,4],
 * result | soft value (f32 pair), 0} at the game cursor of records i64[capacity,8].  A game that does not fit is not
 * written and sets ctl[3] bit 0.  nrows of the finished slots is reset to 0.  Offsets come from a scan, not from
 * atomics: the output is bit-reproducible. */
LZB_API int lzb_actor_record(const uint64_t *states, const uint8_t *active, const float *policy, const int64_t *chosen,
                             int64_t G, int32_t max_plies, int32_t *nrows, int64_t *arena, int8_t *signs,
                             int16_t *actions, uint64_t *ctl, void *stream);
LZB_API int lzb_actor_emit(const uint8_t *finished, const float *result, const float *soft, const uint64_t *states,
                           int64_t G, int32_t max_plies, int32_t *nrows, const int64_t *arena, const int8_t *signs,
                           const int16_t *actions, int64_t *out_rows, int16_t *out_actions, int64_t *records,
                           int64_t capacity, uint64_t *ctl, int64_t step, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* LIUZHOU_B200_H */
