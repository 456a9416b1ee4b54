/*
 * gaz_net.h -- C ABI of the policy/value network evaluator inside libgaz_b200.so.
 *
 * Replaces the reference's evaluator transport + runtime: Client_Server.Server.start
 * (Client_Server.py:162-217: batch -> onnxruntime sess.run -> scatter) and the ORT/TensorRT session
 * built by Self_Play.py:288-341, for the models of {Gomoku,Connect4,TicTacToe}/Build_Model.py.  The network is described as a
 * flat op list over numbered activation buffers (built by grok_alpha_zero_b200/net.py from netspec.py).
 *
 * Activation layout ("padded rows"): a board of H x W cells is stored as (H+1) x (W+1) rows of C
 * channels - one zero row above each board and one zero column right of each row - so a k=3 "same"
 * convolution tap (dy,dx) is the row shift dy*(W+1)+dx of one 2-D TMA tile and the zero padding comes
 * from the layout (and TMA out-of-bounds fill at both ends of the batch).
 */
#ifndef GAZ_NET_H
#define GAZ_NET_H
#include <stdint.h>
#include "gaz_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gaz_net gaz_net;

/* most networks one engine can hold (gaz_attach_nets) */
#define GAZ_MAX_NETS 8

enum { GAZ_OP_STEM = 0, GAZ_OP_CONV_TC = 1, GAZ_OP_SE = 2, GAZ_OP_HEADCONV = 3, GAZ_OP_DENSE = 4, GAZ_OP_POLICY_OUT = 5 };
enum { GAZ_BUF_ROWS_BF16 = 0, GAZ_BUF_ROWS_F32 = 1, GAZ_BUF_FLAT_F32 = 2 };
enum { GAZ_ACT_NONE = 0, GAZ_ACT_RELU = 1, GAZ_ACT_GELU = 2, GAZ_ACT_TANH = 3 };
enum { GAZ_POLICY_SOFTMAX = 0, GAZ_POLICY_STABLEMAX = 1, GAZ_POLICY_LINEAR = 2 };

typedef struct gaz_net_buf {
    int32_t kind;   /* GAZ_BUF_* */
    int32_t width;  /* channels per padded row, or features per board for FLAT */
} gaz_net_buf;

/* Offsets index the float32 blob (wf) unless stated; -1 = absent. */
typedef struct gaz_net_op {
    int32_t type;
    int32_t in_buf, res_buf, out_raw, out_a, out_b; /* buffer ids, -1 = none */
    int32_t cin, cout, ksize, act;                  /* act: stem activation / dense post-activation */
    int32_t flags;                                  /* DENSE: bit0 pre-affine, bit1 pre-relu, bit2 writes value output */
    int32_t pad;
    int64_t w;      /* STEM/HEADCONV/DENSE: float blob; CONV_TC: offset into the bf16 blob, layout [cout][taps*cin] */
    int64_t bias;
    int64_t scale_a, shift_a, scale_b, shift_b;     /* fused BN affines of the activated outputs / dense pre-affine */
    int64_t w2, bias2, w3, bias3;                   /* SE: dense1 (w2,bias2) and dense2 (w3,bias3) */
} gaz_net_op;

typedef struct gaz_net_desc {
    int32_t game;        /* GAZ_GAME_* */
    int32_t max_batch;   /* leaves per forward pass */
    int32_t n_bufs, n_ops;
    int32_t policy_mode; /* GAZ_POLICY_* (Build_Model.py: "policy" activation) */
    int32_t device;
    const gaz_net_buf *bufs;
    const gaz_net_op *ops;
    const float *wf;      int64_t n_wf;
    const uint16_t *wh;   int64_t n_wh;   /* bf16 bit patterns */
} gaz_net_desc;

int gaz_net_create(const gaz_net_desc *desc, gaz_net **out);
/* gaz_net_create, but the new network uses the activation workspace of `share` (share == NULL: gaz_net_create): every
 * allocation that scales with max_batch (the activation buffers, the bf16 trunk copy of a tensor-core head, the dense
 * layers' bf16 inputs and the host-forward staging).  Weights, per-op tables, streams, events and the per-chunk counters
 * stay the network's own.  `share` must have the same game, device and max_batch, the same buffer list (kind, width) and
 * the same op structure (type, buffer ids, cin, cout, ksize, act, flags); otherwise the call fails naming the first
 * difference.  The workspace is reference-counted: it lives until the last network using it is destroyed, in any order.
 * Rule: networks that share a workspace must not run forward passes at the same time.  Networks attached to one engine
 * serve a round one after another on the engine's stream, and gaz_net_forward_host synchronises before it returns, so
 * both uses are safe from one host thread. */
int gaz_net_create_shared(const gaz_net_desc *desc, gaz_net *share, gaz_net **out);
void gaz_net_destroy(gaz_net *net);

/* session.run(["policy","value"], {"inputs": x}) for a host batch (MCTS.py:224-235,
 * Client_Server.py:206): states = n * H*W*C int8 (HWC); outputs float32: policy n*P, value n,
 * logits n*P (optional, pre-activation policy for the tolerance check). */
int gaz_net_forward_host(gaz_net *net, const int8_t *states, int n, float *policy, float *value, float *logits);

/* Attach to an engine: gaz_eval_net() then serves the outstanding leaf requests of gaz_select()
 * on the engine's stream with no host round trip. */
int gaz_attach_net(gaz_engine *e, gaz_net *net);
/* Self_Play.py:39-57 keeps one tree per player; in a match or a tournament each tree's leaves go to the network of its
 * side.  nets: n_nets (1..GAZ_MAX_NETS) non-null networks of the engine's game.  n_nets == 1 is gaz_attach_net(e, nets[0]).
 * Several networks must have the same policy size and cannot be combined with the evaluation cache (its key does not
 * include the network).  Every round, the leaf list is partitioned by network (stable), each network serves its packed
 * list in chunks of the whole leaf bound, and the outputs are scattered back to leaf order.  A refused call changes
 * nothing.  Attaching fewer networks than the tree table names resets the table to network 0. */
int gaz_attach_nets(gaz_engine *e, gaz_net *const *nets, int n_nets);
/* tree_net: n_trees bytes, network index of every tree (< n_nets).  Stream-ordered upload; a captured round graph stays
 * valid (it reads the table from device memory). */
int gaz_set_tree_nets(gaz_engine *e, const uint8_t *tree_net);

/* Symmetric network evaluation.  GAZ_SYM_NONE (the default) evaluates every request once, in the orientation it was
 * reached in, as the reference does.  GAZ_SYM_RANDOM evaluates each request under one board symmetry g drawn from a hash
 * of (seed, the tree's key of gaz_set_tree_keys or seed ^ tree, the input-state bytes), so the draw does not depend on
 * slots, batch layout, chunking or the number of GPUs (oracle/sym_hash.py is the hash's Python twin).  GAZ_SYM_ENSEMBLE
 * evaluates it under all n_sym symmetries and averages the mapped-back outputs: fp32 sums in the order g = 0..n_sym-1,
 * times 1/n_sym, for the policy row as the head returns it (probabilities, or logits for a linear head) and the value.
 * Tables: n_sym rows of S = H*W*C (perm_state) and P (perm_policy) int32 entries, each row a permutation:
 *   state_g[j] = state[perm_state[g][j]]        (the transformed input state)
 *   p[a]       = q_g[perm_policy[g][a]]         (q_g = the network's policy row for state_g, p = the mapped-back row)
 * grok_alpha_zero_b200.games.eval_symmetries builds them from the board geometry.  Applies to gaz_eval_net and
 * gaz_rounds_net*, root evaluations included; not to gaz_put_evals or gaz_eval_hash.  Any mode but NONE routes the leaves
 * like several networks do (also with one network) and cannot be combined with the evaluation cache.  Changing the mode,
 * n_sym or seed re-captures the round graph; new tables of the same shape do not.  With GAZ_SYM_NONE the tables are
 * ignored (may be NULL).  A refused call changes nothing. */
enum { GAZ_SYM_NONE = 0, GAZ_SYM_RANDOM = 1, GAZ_SYM_ENSEMBLE = 2 };
#define GAZ_MAX_SYM 8
int gaz_set_eval_symmetry(gaz_engine *e, int mode, int n_sym, const int32_t *perm_state, const int32_t *perm_policy,
                          uint64_t seed);
int gaz_eval_net(gaz_engine *e);
/* n_rounds x (select -> network -> expand), stream-ordered, no host sync inside; returns 0 */
int gaz_rounds_net(gaz_engine *e, int n_rounds);
/* same without the trailing stream synchronise */
int gaz_rounds_net_async(gaz_engine *e, int n_rounds);

/* timing / introspection for bench.py */
/* Bracket every tcgen05 conv launch with CUDA events on the launching stream (max_launches = event
 * pairs to keep; 0 disables) and read the totals back after a stream synchronise. */
int gaz_net_profile(gaz_net *net, int max_launches);
int gaz_net_profile_read(gaz_net *net, float *total_ms, int *n_launches, float *per_op_ms);
/* device bytes the network allocated itself (a shared activation workspace counts for its creator only) */
int64_t gaz_net_bytes(gaz_net *net);
int gaz_net_launches_per_forward(gaz_net *net);
/* residual blocks run by the launch of op `op`: consecutive fused blocks share one launch of up to 6 layers (gaz_block.cuh);
 * 0 = the op launches no block kernel (not a block, or absorbed into an earlier op's launch) */
int gaz_net_op_blocks(gaz_net *net, int op);
/* times `iters` forward passes of `n` resident leaves with CUDA events on the net's stream;
 * ms_out[0] = average milliseconds per pass */
int gaz_net_time_forward(gaz_net *net, int n, int iters, float *ms_out);

#ifdef __cplusplus
}
#endif
#endif
