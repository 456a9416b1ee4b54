// gaz_engine.cu -- engine object, kernels and the C ABI (include/gaz_b200.h).
//
// Build (product):  nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false ... -> libgaz_b200.so
// Build (tests)  :  g++ -x c++ -DGAZ_EMUL ...  -> tests/_emul/libgaz_emul.so  (host emulation of the
//                   warp code for the CPU test-suite; never loaded by the package).
#include "gaz_internal.h"

#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>

using namespace gaz;

static thread_local std::string g_err;
int gaz_fail(const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return -1;
}
#define fail gaz_fail

template <class T> static int ealloc(gaz_engine *e, T **p, size_t count) {
    void *q = nullptr;
    if (dev_alloc(&q, count * sizeof(T)) != 0) return -1;
    e->allocs.push_back(q);
    e->bytes += (int64_t)(count * sizeof(T));
    *p = (T *)q;
    return 0;
}

// --------------------------------------------------------------- kernels ----
static constexpr int WARPS = 4;
static constexpr int THREADS = WARPS * 32;

// hash evaluator: one warp per leaf (oracle/hash_eval.py, oracle/mcts_oracle.c:orc_hash_eval)
GAZ_HD uint64_t mix64(uint64_t z) {
    z ^= z >> 30; z *= 0xbf58476d1ce4e5b9ULL;
    z ^= z >> 27; z *= 0x94d049bb133111ebULL;
    z ^= z >> 31;
    return z;
}
#define GAZ_GOLD 0x9E3779B97F4A7C15ULL

template <class CG>
GAZ_HD void hash_eval_leaf(const CG &cg, const View &v, int leaf, uint64_t salt, int logits, const int8_t *states, float *policy,
                           float *value) {
    const int n = v.ncell * v.C;
    const int8_t *st = states + (size_t)leaf * n;
    uint64_t acc = 0;
    for (int i = cg.lane; i < n; i += cg.width())
        acc += (uint64_t)(int64_t)(st[i] + 2) * mix64((uint64_t)(i + 1) * GAZ_GOLD);
    acc = cg.sum64(acc);
    uint64_t h0 = mix64(acc + salt * 0xD1B54A32D192ED03ULL);
    float *pol = policy + (size_t)leaf * v.P;
    for (int i = cg.lane; i < v.P; i += cg.width()) {
        uint64_t r = mix64(h0 + (uint64_t)(i + 1) * GAZ_GOLD);
        uint32_t k = (uint32_t)(((r >> 52) << 8) | (uint64_t)i) + 1u;
        pol[i] = logits ? (float)k * 0x1p-17f - 4.0f : (float)k;
    }
    if (cg.lane == 0) {
        uint64_t rv = mix64(h0 + 0x5851F42D4C957F2DULL);
        value[leaf] = (float)(rv >> 40) * 0x1p-23f - 1.0f;
    }
}

// ---- evaluation cache ----------------------------------------------------------------------------------------
struct CacheView {
    long long entries;
    int scope, S, P;
    int8_t *state;
    unsigned long long *tag;
    float *pol, *val;
    int32_t *claim, *miss_idx, *miss_count;
    int8_t *packed_state;
    float *packed_pol, *packed_val;
    unsigned long long *stats;
    int epoch;
};
template <class CG> GAZ_HD unsigned long long cache_hash(const CG &cg, const View &v, const CacheView &c, int leaf) {
    const int8_t *st = v.leaf_state + (size_t)leaf * c.S;
    uint64_t acc = 0;
    for (int i = cg.lane; i < c.S; i += cg.width())
        acc += (uint64_t)(int64_t)(st[i] + 2) * mix64((uint64_t)(i + 1) * 0xC2B2AE3D27D4EB4FULL);
    acc = cg.sum64(acc);
    if (c.scope == 0) {   // per game: positions of different games never share an entry
        const int tree = v.leaves[leaf].tree;
        const uint64_t gkey = v.tree_keys ? v.tree_keys[tree] / (uint64_t)v.trees_per_game : (uint64_t)(tree / v.trees_per_game);
        acc += mix64(gkey + 0x9E3779B97F4A7C15ULL);
    }
    return mix64(acc) | 0x8000000000000000ULL;
}
// one leaf request: hit -> outputs copied to the leaf's slots; miss -> appended to the packed list the evaluator serves
template <class CG> GAZ_HD void cache_lookup_leaf(const CG &cg, const View &v, const CacheView &c, int leaf) {
    const unsigned long long h = cache_hash(cg, v, c, leaf);
    const long long slot = (long long)(h % (unsigned long long)c.entries);
    const int8_t *st = v.leaf_state + (size_t)leaf * c.S;
    bool same = c.tag[slot] == h;
    if (same) {   // the full state decides: a hash collision can never return another position's outputs
        const int8_t *cs = c.state + (size_t)slot * c.S;
        int diff = 0;
        for (int i = cg.lane; i < c.S; i += cg.width()) diff |= cs[i] != st[i];
        same = cg.sum(diff) == 0;
    }
    if (same) {
        const float *cp = c.pol + (size_t)slot * c.P;
        float *po = v.policy + (size_t)leaf * c.P;
        for (int i = cg.lane; i < c.P; i += cg.width()) po[i] = cp[i];
        if (cg.lane == 0) v.value[leaf] = c.val[slot];
    } else {
        int m = 0;
        if (cg.lane == 0) {
#if defined(__CUDA_ARCH__)
            m = atomicAdd(c.miss_count, 1);
#else
            m = (*c.miss_count)++;
#endif
            c.miss_idx[m] = leaf;
        }
        m = cg.bcast(m, 0);
        int8_t *ps = c.packed_state + (size_t)m * c.S;
        for (int i = cg.lane; i < c.S; i += cg.width()) ps[i] = st[i];
    }
    if (cg.lane == 0) {
#if defined(__CUDA_ARCH__)
        atomicAdd(c.stats, 1ULL);
        if (same) atomicAdd(c.stats + 1, 1ULL);
#else
        c.stats[0]++;
        if (same) c.stats[1]++;
#endif
    }
}
// packed miss m: results back to its leaf, and into the table (one writer per slot and pass: the first to claim it)
template <class CG> GAZ_HD void cache_fill_miss(const CG &cg, const View &v, const CacheView &c, int m) {
    const int leaf = c.miss_idx[m];
    const float *pp = c.packed_pol + (size_t)m * c.P;
    float *po = v.policy + (size_t)leaf * c.P;
    for (int i = cg.lane; i < c.P; i += cg.width()) po[i] = pp[i];
    if (cg.lane == 0) v.value[leaf] = c.packed_val[m];
    const unsigned long long h = cache_hash(cg, v, c, leaf);
    const long long slot = (long long)(h % (unsigned long long)c.entries);
    int mine = 0;
    if (cg.lane == 0) {
#if defined(__CUDA_ARCH__)
        mine = atomicExch(c.claim + slot, c.epoch) != c.epoch;
#else
        mine = c.claim[slot] != c.epoch;
        c.claim[slot] = c.epoch;
#endif
    }
    mine = cg.bcast(mine, 0);
    if (!mine) return;
    const int8_t *st = v.leaf_state + (size_t)leaf * c.S;
    int8_t *cs = c.state + (size_t)slot * c.S;
    float *cp = c.pol + (size_t)slot * c.P;
    for (int i = cg.lane; i < c.S; i += cg.width()) cs[i] = st[i];
    for (int i = cg.lane; i < c.P; i += cg.width()) cp[i] = pp[i];
    cg.sync();
    if (cg.lane == 0) { c.val[slot] = c.packed_val[m]; c.tag[slot] = h; }
}
static CacheView cache_view(const gaz_eval_cache *c) {
    CacheView cv;
    cv.entries = c->entries; cv.scope = c->scope; cv.S = c->S; cv.P = c->P; cv.state = c->state; cv.tag = c->tag; cv.pol = c->pol;
    cv.val = c->val; cv.claim = c->claim; cv.miss_idx = c->miss_idx; cv.miss_count = c->miss_count; cv.packed_state = c->packed_state;
    cv.packed_pol = c->packed_pol; cv.packed_val = c->packed_val; cv.stats = c->stats; cv.epoch = c->epoch;
    return cv;
}

// Start of run(): budget rules MCTS.py:542-546 / MCTS_Gumbel.py:570-599
template <class CG> GAZ_HD void run_begin_tree(const CG &cg, const View &v, int tree, int limit) {
    TreeState &ts = v.trees[tree];
    const GameState &g = v.games[tree / v.trees_per_game];
    int nids = n_action_ids(v);
    int n_legal = 0;
    for (int a = cg.lane; a < nids; a += cg.width()) n_legal += action_legal(v, g.board, a) ? 1 : 0;
    n_legal = cg.sum(n_legal);
    cg.sync();
    if (cg.lane != 0) return;
    ts.iter = 0;
    if (limit <= 0 || ts.root < 0) { ts.limit = 0; ts.g_state = GS_IDLE; return; }
    if (!v.gumbel) {
        if (n_legal == 1) limit = 1;
        else if (limit < n_legal) limit = n_legal * 3;
        ts.limit = limit;
    } else {
        if (ts.g_m > n_legal) ts.g_m = n_legal; // permanent (MCTS_Gumbel.py:581-582)
        ts.g_n = limit;
        ts.g_phase = 0;
        ts.g_curiter = 0;
        ts.g_ntop = nr_L(*node_ptr(v, tree, ts.root));
        ts.g_cur = 0;
        ts.g_done_in_child = -1;
        if (n_legal > 1) { ts.g_state = GS_HALVE; ts.limit = 1; ts.g_best_slot = -1; }
        else { ts.g_state = GS_DONE; ts.limit = 0; ts.g_best_slot = 0; }
    }
}

// game.do_action + check_win (Self_Play.py:142-144)
GAZ_HD void apply_action_game(const View &v, int gi, int action, int32_t *winners) {
    GameState &g = v.games[gi];
    if (action >= 0 && g.winner == -2) {
        int r = reply_result(v, g.board, action, g.next_player);
        board_play(v, g.board, action, g.next_player);
        if (r == TERM_WIN) g.winner = g.next_player;
        else if (r == TERM_DRAW) g.winner = 0;
        g.last3 = push_last3(g.last3, action);
        g.hist_len++;
        g.last_action = action;
        g.next_player = -g.next_player;
    }
    if (winners) winners[gi] = g.winner;
}


// Root statistics of every tree as dense per-action vectors (the rows of MCTS.run, MCTS.py:591-600,
// scattered by action id the way compute_policy_improvement does, Gomoku.py:257-262).
template <class CG>
GAZ_HD void root_dense_tree(const CG &cg, const View &v, int tree, uint32_t *visits, float *values, int32_t *info) {
    const TreeState &ts = v.trees[tree];
    uint32_t *vo = visits + (size_t)tree * v.P;
    float *qo = values ? values + (size_t)tree * v.P : nullptr;
    for (int i = cg.lane; i < v.P; i += cg.width()) { vo[i] = 0; if (qo) qo[i] = 0.0f; }
    cg.sync();
    int32_t *io = info + (size_t)tree * 4;
    if (ts.root < 0) {
        if (cg.lane == 0) { io[0] = 0; io[1] = -1; io[2] = ts.iter; io[3] = ts.evals; }
        return;
    }
    const NodeRec r = *node_ptr(v, tree, ts.root);
    const auto sa = slota_ptr(v, tree);
    const int L = nr_L(r);
    uint32_t bestv = 0;
    int besti = L;
    for (int i = cg.lane; i < L; i += cg.width()) {
        int c = child_at(v, tree, r, i);
        if (c < 0) continue;
        const NodeRec *cr = node_ptr(v, tree, c);
        int a = sa[r.slot_base + i];
        vo[a] = cr->visits;
        if (qo) qo[a] = cr->value;
        if (cr->visits > bestv) { bestv = cr->visits; besti = i; } // first max inside the lane's stride
    }
    // np.argmax(child_visits): first maximum over slot order (MCTS.py:603)
    uint32_t mx = cg.umax(bestv);
    int cand = (bestv == mx && besti < L) ? besti : L;
    cand = cg.imin(cand);
    if (cg.lane == 0) {
        io[0] = (int32_t)ts.root_visits;
        io[1] = v.gumbel ? (ts.g_best_slot >= 0 ? sa[r.slot_base + ts.g_best_slot] : -1)
                         : (L > 0 ? sa[r.slot_base + (cand < L ? cand : 0)] : -1);
        io[2] = ts.iter;
        io[3] = ts.evals;
    }
}

// Pages a tree owns beyond its allocation cursor go back to the engine's pool (after re-rooting compacted the tree or a
// fresh root reset it).  Runs as its own pass: inside it pages are only pushed, inside every other kernel only popped.
GAZ_HD void release_pages(const View &v, int tree) {
    TreeState &ts = v.trees[tree];
    const int keep = (ts.n_slots + PAGE_SLOTS - 1) >> PAGE_SHIFT;
    for (int pg = keep; pg < ts.n_pages; pg++) {
#if defined(__CUDA_ARCH__)
        const int pos = atomicAdd(v.free_top, 1);
#else
        const int pos = (*v.free_top)++;
#endif
        v.free_pages[pos] = v.page_table[(size_t)tree * v.max_pages + pg];
    }
    if (ts.n_pages > keep) ts.n_pages = keep;
}

// Batched upload of live games: cells int8 [n_games][ncell], meta int32 [n_games][4] =
// next_player, hist_len, last3 (packed), last_action
GAZ_HD void set_game_from_cells(const View &v, int gi, const int8_t *cells, const int32_t *meta) {
    GameState g;
    for (int w = 0; w < MAXNW; w++) g.board[w] = 0;
    const int8_t *c = cells + (size_t)gi * v.ncell;
    for (int i = 0; i < v.ncell; i++) {
        if (c[i] == 0) continue;
        int p = c[i] > 0 ? 1 : 0;
        if (v.game == GAME_GOMOKU) {
            int y = i / 15, x = i - y * 15;
            g.board[p * 8 + (y >> 1)] |= 1u << (x + (y & 1) * 16);
        } else if (v.game == GAME_C4) {
            int y = i / 7, x = i - y * 7;
            int bit = x * 7 + (5 - y);
            g.board[p * 2 + (bit >> 5)] |= 1u << (bit & 31);
        } else {
            g.board[p] |= 1u << i;
        }
    }
    g.next_player = meta[gi * 4 + 0];
    g.hist_len = meta[gi * 4 + 1];
    g.last3 = (uint32_t)meta[gi * 4 + 2];
    g.winner = -2;
    g.last_action = meta[gi * 4 + 3];
    g.pad[0] = g.pad[1] = g.pad[2] = 0;
    v.games[gi] = g;
}

#ifndef GAZ_EMUL
#define WARP_PROLOGUE(count)                                          \
    const int widx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;    \
    if (widx >= (count)) return;                                      \
    __shared__ Scratch s_sc[WARPS];                                   \
    Scratch &sc = s_sc[threadIdx.x >> 5];                             \
    Coop cg;

__global__ void __launch_bounds__(THREADS) k_select(View v) {
    WARP_PROLOGUE(v.n_trees)
    if (v.gumbel) gumbel_step(cg, v, widx, sc);
    else puct_select_step(cg, v, widx, sc);
}
__global__ void __launch_bounds__(THREADS) k_expand(View v) {
    WARP_PROLOGUE(*v.leaf_count)
    expand_finish(cg, v, widx, sc);
}
__global__ void __launch_bounds__(THREADS) k_hash_eval(View v, uint64_t salt, int logits, const int32_t *count, const int8_t *states,
                                                       float *policy, float *value) {
    const int widx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (widx >= *count) return;
    Coop cg;
    hash_eval_leaf(cg, v, widx, salt, logits, states, policy, value);
}
__global__ void __launch_bounds__(THREADS) k_cache_lookup(View v, CacheView c) {
    const int widx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (widx >= *v.leaf_count) return;
    Coop cg;
    cache_lookup_leaf(cg, v, c, widx);
}
__global__ void __launch_bounds__(THREADS) k_cache_fill(View v, CacheView c) {
    const int widx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (widx >= *c.miss_count) return;
    Coop cg;
    cache_fill_miss(cg, v, c, widx);
}
__global__ void __launch_bounds__(THREADS) k_new_roots(View v, const uint8_t *mask) {
    WARP_PROLOGUE(v.n_trees)
    if (mask && !mask[widx]) return;
    root_begin(cg, v, widx, sc);
}
__global__ void __launch_bounds__(THREADS) k_run_begin(View v, const int32_t *limits) {
    const int widx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (widx >= v.n_trees) return;
    Coop cg;
    run_begin_tree(cg, v, widx, limits[widx]);
}
__global__ void __launch_bounds__(THREADS) k_prune(View v, const int16_t *actions, int create_new_root) {
    WARP_PROLOGUE(v.n_trees)
    if (actions[widx] < 0) return;
    prune_step(cg, v, widx, actions[widx], create_new_root, sc);
}
__global__ void k_apply(View v, const int16_t *actions, int32_t *winners) {
    int gi = blockIdx.x * blockDim.x + threadIdx.x;
    if (gi >= v.n_games) return;
    apply_action_game(v, gi, actions[gi], winners);
}
__global__ void k_remaining(View v, int32_t *counter) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    bool run = false;
    if (t < v.n_trees) {
        const TreeState &ts = v.trees[t];
        run = v.gumbel ? (ts.limit > 0 && ts.g_state != GS_DONE && ts.g_state != GS_IDLE)
                       : (ts.limit > 0 && ts.iter < ts.limit);
        run = run || ts.pending;
    }
    unsigned m = __ballot_sync(0xffffffffu, run);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(counter, __popc(m));
}
__global__ void k_reset_counter(int32_t *c) { *c = 0; }
__global__ void k_release(View v) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < v.n_trees) release_pages(v, t);
}
__global__ void __launch_bounds__(32) k_gumbel_pi(View v, int tree, float *out) {
    __shared__ Scratch sc;
    Coop cg;
    gumbel_final_pi(cg, v, tree, sc, out);
}
__global__ void __launch_bounds__(THREADS) k_root_dense(View v, uint32_t *visits, float *values, int32_t *info) {
    const int widx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (widx >= v.n_trees) return;
    Coop cg;
    root_dense_tree(cg, v, widx, visits, values, info);
}
// get_input_state of every live game (Self_Play.py:77: board_states.append(game.get_input_state()))
__global__ void __launch_bounds__(THREADS) k_game_states(View v, int8_t *states, int32_t *info) {
    const int widx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (widx >= v.n_games) return;
    Coop cg;
    const GameState &g = v.games[widx];
    encode_state(cg, v, g.board, -g.next_player, g.hist_len, g.last3, states + (size_t)widx * v.ncell * v.C);
    if (cg.lane == 0) {
        info[widx * 4 + 0] = g.next_player; info[widx * 4 + 1] = g.hist_len;
        info[widx * 4 + 2] = g.winner; info[widx * 4 + 3] = g.last_action;
    }
}
__global__ void k_set_games(View v, const int8_t *cells, const int32_t *meta) {
    int gi = blockIdx.x * blockDim.x + threadIdx.x;
    if (gi >= v.n_games) return;
    set_game_from_cells(v, gi, cells, meta);
}
__global__ void __launch_bounds__(THREADS) k_gumbel_pi_dense(View v, float *out) {
    WARP_PROLOGUE(v.n_trees)
    gumbel_final_pi_dense(cg, v, widx, sc, out);
}
// table-driven augmentation gather: out[a][t][j] = in[t][perm[a][j]] for states (int8) and policies (float)
__global__ void k_augment(const int8_t *states, const float *policies, long long n_pos, int S, int P, const int32_t *perm_s,
                          const int32_t *perm_p, int n_aug, int8_t *states_out, float *policies_out) {
    const long long per_aug_s = n_pos * S, per_aug_p = n_pos * P;
    const long long total_s = per_aug_s * n_aug, total = total_s + per_aug_p * n_aug;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        if (i < total_s) {
            const int a = (int)(i / per_aug_s);
            const long long r = i - (long long)a * per_aug_s;
            const long long t = r / S;
            const int j = (int)(r - t * S);
            states_out[i] = states[t * S + perm_s[a * S + j]];
        } else {
            const long long k = i - total_s;
            const int a = (int)(k / per_aug_p);
            const long long r = k - (long long)a * per_aug_p;
            const long long t = r / P;
            const int j = (int)(r - t * P);
            policies_out[k] = policies[t * P + perm_p[a * P + j]];
        }
    }
}
static inline int grid_warps(int n) { return (n + WARPS - 1) / WARPS; }
#endif

// ------------------------------------------------------------- launchers ----
static int launch_select(gaz_engine *e) {
#ifdef GAZ_EMUL
    *e->v.leaf_count = 0;
    for (int t = 0; t < e->v.n_trees; t++) {
        Coop cg; Scratch sc;
        if (e->v.gumbel) gumbel_step(cg, e->v, t, sc);
        else puct_select_step(cg, e->v, t, sc);
    }
#else
    k_reset_counter<<<1, 1, 0, e->stream>>>(e->v.leaf_count);
    k_select<<<grid_warps(e->v.n_trees), THREADS, 0, e->stream>>>(e->v);
    CK(cudaGetLastError());
#endif
    return 0;
}
static int launch_expand(gaz_engine *e) {
#ifdef GAZ_EMUL
    for (int l = 0; l < *e->v.leaf_count; l++) { Coop cg; Scratch sc; expand_finish(cg, e->v, l, sc); }
    *e->v.leaf_count = 0;
#else
    k_expand<<<grid_warps(e->v.n_trees), THREADS, 0, e->stream>>>(e->v);
    CK(cudaGetLastError());
#endif
    return 0;
}
int gaz_internal_cache_lookup(gaz_engine *e) {
    gaz_eval_cache *c = e->cache;
    if (dev_zero(c->miss_count, sizeof(int32_t), e->stream) != 0) return -1;
    const CacheView cv = cache_view(c);
#ifdef GAZ_EMUL
    for (int l = 0; l < *e->v.leaf_count; l++) { Coop cg; cache_lookup_leaf(cg, e->v, cv, l); }
#else
    k_cache_lookup<<<grid_warps(e->v.n_trees), THREADS, 0, e->stream>>>(e->v, cv);
    CK(cudaGetLastError());
#endif
    return 0;
}
int gaz_internal_cache_fill(gaz_engine *e) {
    gaz_eval_cache *c = e->cache;
    c->epoch++;
    const CacheView cv = cache_view(c);
#ifdef GAZ_EMUL
    for (int m = 0; m < *c->miss_count; m++) { Coop cg; cache_fill_miss(cg, e->v, cv, m); }
#else
    k_cache_fill<<<grid_warps(e->v.n_trees), THREADS, 0, e->stream>>>(e->v, cv);
    CK(cudaGetLastError());
#endif
    return 0;
}
static int launch_hash(gaz_engine *e, uint64_t salt, int logits) {
    const View &v = e->v;
    gaz_eval_cache *c = e->cache;
    if (c && gaz_internal_cache_lookup(e) != 0) return -1;
    const int32_t *count = c ? c->miss_count : v.leaf_count;
    const int8_t *states = c ? c->packed_state : v.leaf_state;
    float *pol = c ? c->packed_pol : v.policy, *val = c ? c->packed_val : v.value;
#ifdef GAZ_EMUL
    for (int l = 0; l < *count; l++) { Coop cg; hash_eval_leaf(cg, v, l, salt, logits, states, pol, val); }
#else
    k_hash_eval<<<grid_warps(v.n_trees), THREADS, 0, e->stream>>>(v, salt, logits, count, states, pol, val);
    CK(cudaGetLastError());
#endif
    if (c && gaz_internal_cache_fill(e) != 0) return -1;
    return 0;
}
int gaz_internal_launch_select(gaz_engine *e) { return launch_select(e); }
int gaz_internal_alloc(gaz_engine *e, void **p, size_t bytes) { return ealloc(e, (uint8_t **)p, bytes); }
void gaz_internal_free(gaz_engine *e, void *p, size_t bytes) {
    for (size_t i = 0; i < e->allocs.size(); i++)
        if (e->allocs[i] == p) {
            e->allocs.erase(e->allocs.begin() + (long)i);
            e->bytes -= (int64_t)bytes;
            dev_free(p);
            return;
        }
}
int gaz_internal_launch_expand(gaz_engine *e) { return launch_expand(e); }
static int read_leaf_count(gaz_engine *e) {
    int32_t n = 0;
    if (d2h(&n, e->v.leaf_count, sizeof n, e->stream) != 0) return -1;
    return n;
}

// ------------------------------------------------------------------ ABI -----
extern "C" {

const char *gaz_last_error(void) { return g_err.c_str(); }
int gaz_abi_version(void) { return 4; }

int gaz_create(const gaz_config *cfg, gaz_engine **out) {
    if (!cfg || !out) return fail("null argument");
    if (cfg->game < 0 || cfg->game > 2) return fail("bad game %d", cfg->game);
    if (cfg->n_games <= 0 || cfg->trees_per_game <= 0 || cfg->trees_per_game > 2) return fail("bad n_games/trees_per_game");
    if (cfg->node_cap < 8 || cfg->slot_cap < 256) return fail("node_cap/slot_cap too small");
#ifndef GAZ_EMUL
    {
        int ndev = 0;
        cudaError_t ce = cudaGetDeviceCount(&ndev);
        if (ce != cudaSuccess || ndev <= 0)
            return fail("no CUDA device (%s): libgaz_b200 has no CPU path", cudaGetErrorString(ce));
        CK(cudaSetDevice(cfg->device));
    }
#endif
    gaz_engine *e = new gaz_engine();
    e->cfg = *cfg;
    e->bytes = 0;
    for (int k = 0; k < GAZ_MAX_NETS; k++) e->nets[k] = nullptr;
    e->n_nets = 0;
    e->tree_net_max = 0;
    e->d_tree_net = nullptr;
    e->route = nullptr;
    e->sym = nullptr;
    e->cache = nullptr;
    e->leaf_bound = 0;
    e->round_graph = nullptr; e->round_graph_chunks = 0; e->round_graph_warm = 0;
    e->attach_epoch = 0; e->round_graph_attach = 0;
    e->view_epoch = 0; e->round_graph_epoch = 0;
    View &v = e->v;
    memset(&v, 0, sizeof v);
    v.game = cfg->game;
    if (cfg->game == GAME_TTT) { v.H = 3; v.W = 3; v.C = 2; v.P = 9; v.NW = 2; }
    else if (cfg->game == GAME_C4) { v.H = 6; v.W = 7; v.C = 4; v.P = 7; v.NW = 4; }
    else { v.H = 15; v.W = 15; v.C = 2; v.P = 225; v.NW = 16; }
    v.ncell = v.H * v.W;
    v.n_games = cfg->n_games;
    v.trees_per_game = cfg->trees_per_game;
    v.n_trees = cfg->n_games * cfg->trees_per_game;
    v.node_cap = cfg->node_cap;
    v.slot_cap = cfg->slot_cap;
    v.gumbel = cfg->mode == GAZ_MODE_GUMBEL;
    v.c_init = cfg->c_puct_init;
    v.c_base = cfg->c_puct_base;
    v.c_visit = (float)cfg->c_visit;
    v.c_scale = (float)cfg->c_scale;
    v.c_visit_d = cfg->c_visit;
    v.c_scale_d = cfg->c_scale;
    v.use_softmax = cfg->use_softmax;
    v.gm_cap = MAXL;
    v.lut_n = cfg->lut_n > 0 ? cfg->lut_n : (1 << 20);
#ifndef GAZ_EMUL
    CK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
#else
    e->stream = 0;
#endif
    const size_t NT = (size_t)v.n_trees;
    int rc = 0;
    rc |= ealloc(e, &v.nodes, NT * v.node_cap);
    rc |= ealloc(e, &v.boards, NT * v.node_cap * v.NW);
    // child slots: one pool of pages for the whole engine (gaz_core.cuh); slot_cap is the per-tree VIRTUAL limit.  The default
    // pool gives every tree its full limit (no sharing risk); cfg->slot_pool sizes it from the expected mean occupancy
    v.max_pages = (v.slot_cap + PAGE_SLOTS - 1) / PAGE_SLOTS;
    {
        int64_t pool = cfg->slot_pool > 0 ? (cfg->slot_pool + PAGE_SLOTS - 1) / PAGE_SLOTS : (int64_t)NT * v.max_pages;
        if (pool < (int64_t)NT) pool = (int64_t)NT;          // at least one page per tree
        if (pool > (int64_t)NT * v.max_pages) pool = (int64_t)NT * v.max_pages;
        if (pool > 0x7fffffff) { delete e; return fail("slot pool of %lld pages is too large", (long long)pool); }
        v.pool_pages = (int)pool;
    }
    const size_t pool_slots = (size_t)v.pool_pages << PAGE_SHIFT;
    rc |= ealloc(e, &v.slot_val, pool_slots);
    rc |= ealloc(e, &v.slot_act, pool_slots);
    if (v.gumbel) rc |= ealloc(e, &v.slot_child, pool_slots);
    rc |= ealloc(e, &v.page_table, NT * v.max_pages);
    rc |= ealloc(e, &v.free_pages, (size_t)v.pool_pages);
    rc |= ealloc(e, &v.free_top, 4);
    rc |= ealloc(e, &v.trees, NT);
    rc |= ealloc(e, &v.games, (size_t)v.n_games);
    rc |= ealloc(e, &v.remap, NT * v.node_cap);
    rc |= ealloc(e, &v.leaf_count, 4);
    rc |= ealloc(e, &v.leaves, NT);
    rc |= ealloc(e, &v.leaf_state, NT * v.ncell * v.C);
    rc |= ealloc(e, &v.policy, NT * v.P);
    rc |= ealloc(e, &v.value, NT);
    rc |= ealloc(e, &v.status, 4);
    if (v.gumbel) {
        rc |= ealloc(e, &v.gm_ids, NT * v.gm_cap);
        rc |= ealloc(e, &v.gm_g, NT * v.gm_cap);
    }
    rc |= ealloc(e, &e->d_limits, NT);
    rc |= ealloc(e, &e->d_actions, NT);
    rc |= ealloc(e, &e->d_mask, NT);
    rc |= ealloc(e, &e->d_counter, 4);
    rc |= ealloc(e, &e->d_winners, (size_t)v.n_games);
    rc |= ealloc(e, &e->d_lut, (size_t)v.lut_n);
    rc |= ealloc(e, &e->d_pi, MAXL);
    e->d_noise = nullptr;
    e->d_states = nullptr; e->d_ginfo = nullptr; e->d_keys = nullptr;
    e->d_cells = nullptr; e->d_meta = nullptr; e->d_dense_vis = nullptr; e->d_dense_val = nullptr; e->d_dense_info = nullptr;
#ifndef GAZ_EMUL
    e->ev0 = nullptr; e->ev1 = nullptr;
#endif
    if (rc != 0) { gaz_destroy(e); return g_err.empty() ? fail("allocation failed") : -1; }
    v.c_lut = e->d_lut;
    *out = e;
    if (gaz_set_puct_params(e, cfg->c_puct_init, cfg->c_puct_base) < 0) { gaz_destroy(e); *out = nullptr; return -1; }
    if (gaz_set_gumbel_params(e, cfg->gumbel_m, cfg->c_visit, cfg->c_scale, cfg->use_softmax) < 0) { gaz_destroy(e); *out = nullptr; return -1; }
    if (gaz_reset_games(e) < 0) { gaz_destroy(e); *out = nullptr; return -1; }
    return 0;
}

void gaz_destroy(gaz_engine *e) {
    if (!e) return;
#ifndef GAZ_EMUL
    cudaStreamSynchronize(e->stream);
    if (e->round_graph) cudaGraphExecDestroy((cudaGraphExec_t)e->round_graph);
#endif
    for (void *p : e->allocs) dev_free(p);
    delete e->cache;
    delete e->route;
    delete e->sym;
#ifndef GAZ_EMUL
    if (e->ev0) { cudaEventDestroy(e->ev0); cudaEventDestroy(e->ev1); }
    cudaStreamDestroy(e->stream);
#endif
    delete e;
}

int gaz_set_puct_params(gaz_engine *e, float c_init, float c_base) {
    if (!e) return fail("null engine");
    e->v.c_init = c_init;
    e->v.c_base = c_base;
    e->view_epoch++;
    // C(N) = c_init + ln((N + c_base + 1) / c_base) with the host libm (glibc) so it equals the
    // oracle's / numba's values (SURVEY V1, V7)
    std::vector<double> lut((size_t)e->v.lut_n);
    for (int N = 0; N < e->v.lut_n; N++)
        lut[(size_t)N] = (double)c_init + log(((double)N + (double)c_base + 1.0) / (double)c_base);
    if (h2d(e->d_lut, lut.data(), lut.size() * sizeof(double), e->stream) != 0) return -1;
    return stream_sync(e->stream);
}

int gaz_set_gumbel_params(gaz_engine *e, int m, double c_visit, double c_scale, int use_softmax) {
    if (!e) return fail("null engine");
    View &v = e->v;
    v.c_visit = (float)c_visit; v.c_scale = (float)c_scale;
    v.c_visit_d = c_visit; v.c_scale_d = c_scale;
    v.use_softmax = use_softmax;
    e->cfg.gumbel_m = m;
    e->view_epoch++;
    std::vector<TreeState> ts((size_t)v.n_trees);
    if (d2h(ts.data(), v.trees, ts.size() * sizeof(TreeState), e->stream) != 0) return -1;
    for (auto &t : ts) t.g_m = m;
    if (h2d(v.trees, ts.data(), ts.size() * sizeof(TreeState), e->stream) != 0) return -1;
    return stream_sync(e->stream);
}

static void cells_to_board(const View &v, const int8_t *cells, uint32_t *b) {
    for (int w = 0; w < MAXNW; w++) b[w] = 0;
    for (int c = 0; c < v.ncell; c++) {
        if (cells[c] == 0) continue;
        int p = cells[c] > 0 ? 1 : 0;
        if (v.game == GAME_GOMOKU) {
            int y = c / 15, x = c % 15;
            b[p * 8 + (y >> 1)] |= 1u << (x + (y & 1) * 16);
        } else if (v.game == GAME_C4) {
            int y = c / 7, x = c % 7;
            int bit = x * 7 + (5 - y);
            b[p * 2 + (bit >> 5)] |= 1u << (bit & 31);
        } else {
            b[p] |= 1u << c;
        }
    }
}

int gaz_set_game(gaz_engine *e, int game, const int8_t *board, int next_player, const int16_t *hist_tail, int hist_len) {
    if (!e || !board) return fail("null argument");
    if (game < 0 || game >= e->v.n_games) return fail("game index %d out of range", game);
    GameState g;
    memset(&g, 0, sizeof g);
    cells_to_board(e->v, board, g.board);
    g.next_player = next_player;
    g.hist_len = hist_len;
    g.last3 = 0;
    int cnt = hist_len < 3 ? hist_len : 3;
    for (int i = cnt - 1; i >= 0; i--) g.last3 = push_last3(g.last3, hist_tail[i]);
    g.winner = -2;
    g.last_action = cnt > 0 ? hist_tail[0] : -1;
    if (h2d(e->v.games + game, &g, sizeof g, e->stream) != 0) return -1;
    return stream_sync(e->stream);
}

int gaz_reset_games(gaz_engine *e) {
    if (!e) return fail("null engine");
    std::vector<GameState> gs((size_t)e->v.n_games);
    memset(gs.data(), 0, gs.size() * sizeof(GameState));
    for (auto &g : gs) { g.next_player = -1; g.winner = -2; g.last_action = -1; }
    if (h2d(e->v.games, gs.data(), gs.size() * sizeof(GameState), e->stream) != 0) return -1;
    std::vector<TreeState> ts((size_t)e->v.n_trees);
    memset(ts.data(), 0, ts.size() * sizeof(TreeState));
    for (auto &t : ts) { t.root = -1; t.g_m = e->cfg.gumbel_m; }
    if (h2d(e->v.trees, ts.data(), ts.size() * sizeof(TreeState), e->stream) != 0) return -1;
    if (dev_zero(e->v.leaf_count, sizeof(int32_t), e->stream) != 0) return -1;
    {   // no tree owns a slot page: the whole pool is free
        std::vector<int32_t> fp((size_t)e->v.pool_pages);
        for (int i = 0; i < e->v.pool_pages; i++) fp[(size_t)i] = e->v.pool_pages - 1 - i;   // page 0 is popped first
        const int32_t top = e->v.pool_pages;
        if (h2d(e->v.free_pages, fp.data(), fp.size() * sizeof(int32_t), e->stream) != 0) return -1;
        if (h2d(e->v.free_top, &top, sizeof top, e->stream) != 0) return -1;
    }
    return stream_sync(e->stream);
}

int gaz_apply_actions(gaz_engine *e, const int16_t *actions, int32_t *winners_out) {
    if (!e || !actions) return fail("null argument");
    const View &v = e->v;
    if (h2d(e->d_actions, actions, (size_t)v.n_games * sizeof(int16_t), e->stream) != 0) return -1;
#ifdef GAZ_EMUL
    for (int g = 0; g < v.n_games; g++) apply_action_game(v, g, e->d_actions[g], e->d_winners);
#else
    k_apply<<<(v.n_games + 127) / 128, 128, 0, e->stream>>>(v, e->d_actions, e->d_winners);
    CK(cudaGetLastError());
#endif
    if (winners_out) return d2h(winners_out, e->d_winners, (size_t)v.n_games * sizeof(int32_t), e->stream);
    return stream_sync(e->stream);
}

int gaz_get_game(gaz_engine *e, int game, int8_t *board_out, int32_t *info_out) {
    if (!e) return fail("null engine");
    if (game < 0 || game >= e->v.n_games) return fail("game index %d out of range", game);
    GameState g;
    if (d2h(&g, e->v.games + game, sizeof g, e->stream) != 0) return -1;
    if (board_out)
        for (int c = 0; c < e->v.ncell; c++) board_out[c] = (int8_t)cell_value(e->v, g.board, c);
    if (info_out) { info_out[0] = g.next_player; info_out[1] = g.hist_len; info_out[2] = g.winner; }
    return 0;
}

int gaz_new_roots(gaz_engine *e, const uint8_t *tree_mask) {
    if (!e) return fail("null engine");
    const View &v = e->v;
    const uint8_t *dm = nullptr;
    if (tree_mask) {
        if (h2d(e->d_mask, tree_mask, (size_t)v.n_trees, e->stream) != 0) return -1;
        dm = e->d_mask;
    }
#ifdef GAZ_EMUL
    *v.leaf_count = 0;
    for (int t = 0; t < v.n_trees; t++) {
        if (dm && !dm[t]) continue;
        Coop cg; Scratch sc;
        root_begin(cg, v, t, sc);
    }
    for (int t = 0; t < v.n_trees; t++) release_pages(v, t);
#else
    k_reset_counter<<<1, 1, 0, e->stream>>>(v.leaf_count);
    k_new_roots<<<grid_warps(v.n_trees), THREADS, 0, e->stream>>>(v, dm);
    k_release<<<(v.n_trees + 127) / 128, 128, 0, e->stream>>>(v);
    CK(cudaGetLastError());
#endif
    int nl = read_leaf_count(e);
    e->leaf_bound = nl > 0 ? nl : 1;
    return nl;
}

int gaz_run_begin(gaz_engine *e, const int32_t *limits) {
    if (!e || !limits) return fail("null argument");
    const View &v = e->v;
    if (h2d(e->d_limits, limits, (size_t)v.n_trees * sizeof(int32_t), e->stream) != 0) return -1;
    int running = 0;
    for (int t = 0; t < v.n_trees; t++) running += limits[t] > 0 ? 1 : 0;
    e->leaf_bound = running > 0 ? running : 1;
#ifdef GAZ_EMUL
    for (int t = 0; t < v.n_trees; t++) { Coop cg; run_begin_tree(cg, v, t, e->d_limits[t]); }
#else
    k_run_begin<<<grid_warps(v.n_trees), THREADS, 0, e->stream>>>(v, e->d_limits);
    CK(cudaGetLastError());
#endif
    return stream_sync(e->stream);
}

int gaz_select(gaz_engine *e) {
    if (!e) return fail("null engine");
    if (launch_select(e) != 0) return -1;
    return read_leaf_count(e);
}

int gaz_get_leaves(gaz_engine *e, int8_t *states_out, int32_t *trees_out) {
    if (!e) return fail("null engine");
    const View &v = e->v;
    int n = read_leaf_count(e);
    if (n <= 0) return n;
    if (states_out && d2h(states_out, v.leaf_state, (size_t)n * v.ncell * v.C, e->stream) != 0) return -1;
    if (trees_out) {
        std::vector<LeafRec> lr((size_t)n);
        if (d2h(lr.data(), v.leaves, lr.size() * sizeof(LeafRec), e->stream) != 0) return -1;
        for (int i = 0; i < n; i++) trees_out[i] = lr[(size_t)i].tree;
    }
    return n;
}

int gaz_get_leaf_depths(gaz_engine *e, int32_t *depths_out) {
    if (!e || !depths_out) return fail("null argument");
    const View &v = e->v;
    int n = read_leaf_count(e);
    if (n <= 0) return n;
    std::vector<LeafRec> lr((size_t)n);
    if (d2h(lr.data(), v.leaves, lr.size() * sizeof(LeafRec), e->stream) != 0) return -1;
    // MCTS.py:346 (root: len(game.action_history)) and :468-472 (child: len(node.action_history) of the PARENT node)
    for (int i = 0; i < n; i++) depths_out[i] = lr[(size_t)i].kind == LEAF_ROOT ? lr[(size_t)i].hist_len : lr[(size_t)i].hist_len - 1;
    return n;
}

int gaz_put_evals(gaz_engine *e, const float *policy, const float *value, int n) {
    if (!e || !policy || !value) return fail("null argument");
    const View &v = e->v;
    if (n < 0 || n > v.n_trees) return fail("bad eval count %d", n);
    if (n == 0) return 0;
    if (h2d(v.policy, policy, (size_t)n * v.P * sizeof(float), e->stream) != 0) return -1;
    if (h2d(v.value, value, (size_t)n * sizeof(float), e->stream) != 0) return -1;
    return stream_sync(e->stream);
}

int gaz_eval_hash(gaz_engine *e, uint64_t salt, int logits) {
    if (!e) return fail("null engine");
    return launch_hash(e, salt, logits);
}

int gaz_expand(gaz_engine *e) {
    if (!e) return fail("null engine");
    if (launch_expand(e) != 0) return -1;
    return stream_sync(e->stream);
}

int gaz_remaining(gaz_engine *e) {
    if (!e) return fail("null engine");
    const View &v = e->v;
#ifdef GAZ_EMUL
    int c = 0;
    for (int t = 0; t < v.n_trees; t++) {
        const TreeState &ts = v.trees[t];
        bool run = v.gumbel ? (ts.limit > 0 && ts.g_state != GS_DONE && ts.g_state != GS_IDLE)
                            : (ts.limit > 0 && ts.iter < ts.limit);
        c += (run || ts.pending) ? 1 : 0;
    }
    return c;
#else
    k_reset_counter<<<1, 1, 0, e->stream>>>(e->d_counter);
    k_remaining<<<(v.n_trees + 127) / 128, 128, 0, e->stream>>>(v, e->d_counter);
    CK(cudaGetLastError());
    int32_t c = 0;
    if (d2h(&c, e->d_counter, sizeof c, e->stream) != 0) return -1;
    return c;
#endif
}

int gaz_rounds_hash(gaz_engine *e, int n_rounds, uint64_t salt, int logits) {
    if (!e) return fail("null engine");
    for (int r = 0; r < n_rounds; r++) {
        if (launch_select(e) != 0) return -1;
        if (launch_hash(e, salt, logits) != 0) return -1;
        if (launch_expand(e) != 0) return -1;
    }
    return stream_sync(e->stream);
}

int gaz_prune(gaz_engine *e, const int16_t *actions, int create_new_root) {
    if (!e || !actions) return fail("null argument");
    const View &v = e->v;
    if (h2d(e->d_actions, actions, (size_t)v.n_trees * sizeof(int16_t), e->stream) != 0) return -1;
#ifdef GAZ_EMUL
    *v.leaf_count = 0;
    for (int t = 0; t < v.n_trees; t++) {
        if (e->d_actions[t] < 0) continue;
        Coop cg; Scratch sc;
        prune_step(cg, v, t, e->d_actions[t], create_new_root, sc);
    }
    for (int t = 0; t < v.n_trees; t++) release_pages(v, t);
#else
    k_reset_counter<<<1, 1, 0, e->stream>>>(v.leaf_count);
    k_prune<<<grid_warps(v.n_trees), THREADS, 0, e->stream>>>(v, e->d_actions, create_new_root);
    k_release<<<(v.n_trees + 127) / 128, 128, 0, e->stream>>>(v);
    CK(cudaGetLastError());
#endif
    int nl = read_leaf_count(e);
    e->leaf_bound = nl > 0 ? nl : 1;
    return nl;
}

int gaz_root_stats(gaz_engine *e, int tree, int16_t *actions, uint32_t *visits, float *values, float *priors,
                   float *raws, int8_t *term, int8_t *expanded, int64_t *info_out) {
    if (!e) return fail("null engine");
    const View &v = e->v;
    if (tree < 0 || tree >= v.n_trees) return fail("tree index %d out of range", tree);
    TreeState ts;
    if (d2h(&ts, v.trees + tree, sizeof ts, e->stream) != 0) return -1;
    if (ts.root < 0) return fail("tree %d has no root", tree);
    NodeRec r;
    if (d2h(&r, v.nodes + (size_t)tree * v.node_cap + ts.root, sizeof r, e->stream) != 0) return -1;
    const int L = nr_L(r);
    std::vector<uint32_t> sv((size_t)(L ? L : 1)), sch((size_t)(L ? L : 1));
    std::vector<uint8_t> sa((size_t)(L ? L : 1));
    if (L > 0) {   // a node's slot block is contiguous inside one page of the pool
        int32_t page = 0;
        if (d2h(&page, v.page_table + (size_t)tree * v.max_pages + (r.slot_base >> PAGE_SHIFT), sizeof page, e->stream) != 0) return -1;
        const size_t off = ((size_t)page << PAGE_SHIFT) + (r.slot_base & (PAGE_SLOTS - 1));
        if (d2h(sv.data(), v.slot_val + off, (size_t)L * 4, e->stream) != 0) return -1;
        if (d2h(sa.data(), v.slot_act + off, (size_t)L, e->stream) != 0) return -1;
        if (v.gumbel && d2h(sch.data(), v.slot_child + off, (size_t)L * 4, e->stream) != 0) return -1;
    }
    int nexp = 0;
    for (int i = 0; i < L; i++) {
        int child;
        if (v.gumbel) child = sch[(size_t)i] == 0xffffffffu ? -1 : (int)sch[(size_t)i];
        else child = (nr_tparent(r) || i < nr_nexp(r)) ? (int)sv[(size_t)i] : -1;
        if (actions) actions[i] = sa[(size_t)i];
        if (child >= 0) {
            NodeRec c;
            if (d2h(&c, v.nodes + (size_t)tree * v.node_cap + child, sizeof c, e->stream) != 0) return -1;
            if (visits) visits[i] = c.visits;
            if (values) values[i] = c.value;
            if (priors) priors[i] = c.prior;
            if (raws) raws[i] = c.raw;
            if (term) term[i] = (int8_t)nr_term(c);
            if (expanded) expanded[i] = 1;
            nexp++;
        } else {
            if (visits) visits[i] = 0;
            if (values) values[i] = 0.0f;
            if (priors) priors[i] = u2f(sv[(size_t)i]);
            if (raws) raws[i] = 0.0f;
            if (term) term[i] = TERM_NONE;
            if (expanded) expanded[i] = 0;
        }
    }
    if (info_out) {
        info_out[0] = L; info_out[1] = nexp; info_out[2] = ts.root_visits; info_out[3] = ts.g_best_slot;
        info_out[4] = ts.n_nodes; info_out[5] = ts.n_slots; info_out[6] = ts.iter; info_out[7] = ts.evals;
    }
    return L;
}

int gaz_gumbel_pi(gaz_engine *e, int tree, float *pi_out) {
    if (!e || !pi_out) return fail("null argument");
    const View &v = e->v;
    if (!v.gumbel) return fail("engine is not in Gumbel mode");
    if (tree < 0 || tree >= v.n_trees) return fail("tree index %d out of range", tree);
#ifdef GAZ_EMUL
    { Coop cg; Scratch sc; gumbel_final_pi(cg, v, tree, sc, e->d_pi); }
#else
    k_gumbel_pi<<<1, 32, 0, e->stream>>>(v, tree, e->d_pi);
    CK(cudaGetLastError());
#endif
    return d2h(pi_out, e->d_pi, MAXL * sizeof(float), e->stream);
}

int gaz_set_gumbel_noise(gaz_engine *e, const double *noise) {
    if (!e) return fail("null engine");
    e->view_epoch++;
    if (!noise) { e->v.gumbel_noise = nullptr; return 0; }
    if (!e->d_noise && ealloc(e, &e->d_noise, (size_t)e->v.n_trees * MAXL) != 0) return -1;
    if (h2d(e->d_noise, noise, (size_t)e->v.n_trees * MAXL * sizeof(double), e->stream) != 0) return -1;
    e->v.gumbel_noise = e->d_noise;
    return stream_sync(e->stream);
}

int gaz_set_games(gaz_engine *e, const int8_t *boards, const int32_t *meta) {
    if (!e || !boards || !meta) return fail("null argument");
    const View &v = e->v;
    if (!e->d_cells) {
        if (ealloc(e, &e->d_cells, (size_t)v.n_games * v.ncell) != 0) return -1;
        if (ealloc(e, &e->d_meta, (size_t)v.n_games * 4) != 0) return -1;
    }
    if (h2d(e->d_cells, boards, (size_t)v.n_games * v.ncell, e->stream) != 0) return -1;
    if (h2d(e->d_meta, meta, (size_t)v.n_games * 4 * sizeof(int32_t), e->stream) != 0) return -1;
#ifdef GAZ_EMUL
    for (int g = 0; g < v.n_games; g++) set_game_from_cells(v, g, e->d_cells, e->d_meta);
#else
    k_set_games<<<(v.n_games + 127) / 128, 128, 0, e->stream>>>(v, e->d_cells, e->d_meta);
    CK(cudaGetLastError());
#endif
    return 0; // stream-ordered; the next call on this engine observes the new games
}

int gaz_root_dense(gaz_engine *e, uint32_t *visits_out, float *values_out, int32_t *info_out) {
    if (!e || !visits_out || !info_out) return fail("null argument");
    const View &v = e->v;
    const size_t NT = (size_t)v.n_trees;
    if (!e->d_dense_vis && ealloc(e, &e->d_dense_vis, NT * v.P) != 0) return -1;
    if (!e->d_dense_val && ealloc(e, &e->d_dense_val, NT * v.P) != 0) return -1;
    if (!e->d_dense_info && ealloc(e, &e->d_dense_info, NT * 4) != 0) return -1;
#ifdef GAZ_EMUL
    for (int t = 0; t < v.n_trees; t++) { Coop cg; root_dense_tree(cg, v, t, e->d_dense_vis, e->d_dense_val, e->d_dense_info); }
    memcpy(visits_out, e->d_dense_vis, NT * v.P * 4);
    if (values_out) memcpy(values_out, e->d_dense_val, NT * v.P * 4);
    memcpy(info_out, e->d_dense_info, NT * 4 * sizeof(int32_t));
    return 0;
#else
    k_root_dense<<<grid_warps(v.n_trees), THREADS, 0, e->stream>>>(v, e->d_dense_vis, e->d_dense_val, e->d_dense_info);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(visits_out, e->d_dense_vis, NT * v.P * 4, cudaMemcpyDeviceToHost, e->stream));
    if (values_out) CK(cudaMemcpyAsync(values_out, e->d_dense_val, NT * v.P * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(info_out, e->d_dense_info, NT * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    return stream_sync(e->stream);
#endif
}

int gaz_get_states(gaz_engine *e, int8_t *states_out, int32_t *info_out) {
    if (!e || !states_out || !info_out) return fail("null argument");
    const View &v = e->v;
    const size_t ss = (size_t)v.ncell * v.C;
    if (!e->d_states) {
        if (ealloc(e, &e->d_states, (size_t)v.n_games * ss) != 0) return -1;
        if (ealloc(e, &e->d_ginfo, (size_t)v.n_games * 4) != 0) return -1;
    }
#ifdef GAZ_EMUL
    for (int g = 0; g < v.n_games; g++) {
        Coop cg;
        const GameState &gs = v.games[g];
        encode_state(cg, v, gs.board, -gs.next_player, gs.hist_len, gs.last3, e->d_states + (size_t)g * ss);
        e->d_ginfo[g * 4 + 0] = gs.next_player; e->d_ginfo[g * 4 + 1] = gs.hist_len;
        e->d_ginfo[g * 4 + 2] = gs.winner; e->d_ginfo[g * 4 + 3] = gs.last_action;
    }
    memcpy(states_out, e->d_states, (size_t)v.n_games * ss);
    memcpy(info_out, e->d_ginfo, (size_t)v.n_games * 4 * sizeof(int32_t));
    return 0;
#else
    k_game_states<<<grid_warps(v.n_games), THREADS, 0, e->stream>>>(v, e->d_states, e->d_ginfo);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(states_out, e->d_states, (size_t)v.n_games * ss, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(info_out, e->d_ginfo, (size_t)v.n_games * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    return stream_sync(e->stream);
#endif
}

int gaz_gumbel_pi_dense(gaz_engine *e, float *pi_out) {
    if (!e || !pi_out) return fail("null argument");
    const View &v = e->v;
    if (!v.gumbel) return fail("engine is not in Gumbel mode");
    const size_t NT = (size_t)v.n_trees;
    if (!e->d_dense_val && ealloc(e, &e->d_dense_val, NT * v.P) != 0) return -1;
#ifdef GAZ_EMUL
    for (int t = 0; t < v.n_trees; t++) { Coop cg; Scratch sc; gumbel_final_pi_dense(cg, v, t, sc, e->d_dense_val); }
    memcpy(pi_out, e->d_dense_val, NT * v.P * 4);
    return 0;
#else
    k_gumbel_pi_dense<<<grid_warps(v.n_trees), THREADS, 0, e->stream>>>(v, e->d_dense_val);
    CK(cudaGetLastError());
    return d2h(pi_out, e->d_dense_val, NT * v.P * 4, e->stream);
#endif
}

int gaz_set_tree_keys(gaz_engine *e, const uint64_t *keys) {
    if (!e) return fail("null engine");
    if ((keys != nullptr) != (e->v.tree_keys != nullptr)) e->view_epoch++;   // the pointer in the View changes
    if (!keys) { e->v.tree_keys = nullptr; return 0; }
    if (!e->d_keys && ealloc(e, &e->d_keys, (size_t)e->v.n_trees) != 0) return -1;
    if (h2d(e->d_keys, keys, (size_t)e->v.n_trees * sizeof(uint64_t), e->stream) != 0) return -1;
    e->v.tree_keys = e->d_keys;
    return stream_sync(e->stream);
}

int gaz_set_noise(gaz_engine *e, float dirichlet_alpha, float dirichlet_epsilon, uint64_t seed) {
    if (!e) return fail("null engine");
    if (dirichlet_epsilon < 0.0f || dirichlet_epsilon >= 1.0f) return fail("dirichlet_epsilon must be in [0, 1)");
    if (dirichlet_epsilon > 0.0f && !(dirichlet_alpha > 0.0f)) return fail("dirichlet_alpha must be positive");
    e->v.dir_alpha = dirichlet_alpha;
    e->v.dir_eps = dirichlet_epsilon;
    e->v.noise_seed = seed;
    e->view_epoch++;
    return 0;
}

int gaz_timer_begin(gaz_engine *e) {
    if (!e) return fail("null engine");
#ifndef GAZ_EMUL
    if (!e->ev0) { CK(cudaEventCreate(&e->ev0)); CK(cudaEventCreate(&e->ev1)); }
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaEventRecord(e->ev0, e->stream));
#endif
    return 0;
}

int gaz_timer_end(gaz_engine *e, float *ms_out) {
    if (!e || !ms_out) return fail("null argument");
    *ms_out = 0.0f;
#ifndef GAZ_EMUL
    if (!e->ev0) return fail("gaz_timer_begin was not called");
    CK(cudaEventRecord(e->ev1, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaEventElapsedTime(ms_out, e->ev0, e->ev1));
#endif
    return 0;
}

int gaz_sync(gaz_engine *e) {
    if (!e) return fail("null engine");
    return stream_sync(e->stream);
}

int gaz_status(gaz_engine *e) {
    if (!e) return fail("null engine");
    int32_t s = 0;
    if (d2h(&s, e->v.status, sizeof s, e->stream) != 0) return -1;
    return s;
}

int gaz_tree_sizes(gaz_engine *e, int32_t *out) {
    if (!e || !out) return fail("null argument");
    const View &v = e->v;
    std::vector<TreeState> ts((size_t)v.n_trees);
    if (d2h(ts.data(), v.trees, ts.size() * sizeof(TreeState), e->stream) != 0) return -1;
    for (int t = 0; t < v.n_trees; t++) { out[2 * t] = ts[t].n_nodes; out[2 * t + 1] = ts[t].n_slots; }
    return 0;
}

int gaz_augment(int device, const int8_t *states, const float *policies, int64_t n_pos, int S, int P, const int32_t *perm_state,
                const int32_t *perm_policy, int n_aug, int8_t *states_out, float *policies_out) {
    if (!states || !policies || !perm_state || !perm_policy || !states_out || !policies_out) return fail("null argument");
    if (n_pos < 0 || S <= 0 || P <= 0 || n_aug <= 0) return fail("bad augmentation shape");
    for (int i = 0; i < n_aug * S; i++) if (perm_state[i] < 0 || perm_state[i] >= S) return fail("state permutation entry %d out of range", i);
    for (int i = 0; i < n_aug * P; i++) if (perm_policy[i] < 0 || perm_policy[i] >= P) return fail("policy permutation entry %d out of range", i);
    if (n_pos == 0) return 0;
#ifdef GAZ_EMUL
    (void)device;
    for (int a = 0; a < n_aug; a++)
        for (int64_t t = 0; t < n_pos; t++) {
            for (int j = 0; j < S; j++) states_out[((int64_t)a * n_pos + t) * S + j] = states[t * S + perm_state[a * S + j]];
            for (int j = 0; j < P; j++) policies_out[((int64_t)a * n_pos + t) * P + j] = policies[t * P + perm_policy[a * P + j]];
        }
    return 0;
#else
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev <= 0) return fail("no CUDA device (%s): libgaz_b200 has no CPU path", cudaGetErrorString(ce));
    CK(cudaSetDevice(device));
    int8_t *d_s = nullptr, *d_so = nullptr;
    float *d_p = nullptr, *d_po = nullptr;
    int32_t *d_ps = nullptr, *d_pp = nullptr;
    const size_t bs = (size_t)n_pos * S, bp = (size_t)n_pos * P * 4;
    int rc = 0;
    auto done = [&](int r) { cudaFree(d_s); cudaFree(d_so); cudaFree(d_p); cudaFree(d_po); cudaFree(d_ps); cudaFree(d_pp); return r; };
    if (cudaMalloc(&d_s, bs) != cudaSuccess || cudaMalloc(&d_so, bs * n_aug) != cudaSuccess || cudaMalloc(&d_p, bp) != cudaSuccess ||
        cudaMalloc(&d_po, bp * n_aug) != cudaSuccess || cudaMalloc(&d_ps, (size_t)n_aug * S * 4) != cudaSuccess ||
        cudaMalloc(&d_pp, (size_t)n_aug * P * 4) != cudaSuccess) {
        cudaGetLastError();
        return done(fail("gaz_augment: device allocation of %zu bytes failed (call it on smaller batches)", (bs + bp) * (n_aug + 1)));
    }
    cudaStream_t st = nullptr; // the legacy default stream: copies and kernel are ordered, the call is synchronous
    rc |= cudaMemcpyAsync(d_s, states, bs, cudaMemcpyHostToDevice, st) != cudaSuccess;
    rc |= cudaMemcpyAsync(d_p, policies, bp, cudaMemcpyHostToDevice, st) != cudaSuccess;
    rc |= cudaMemcpyAsync(d_ps, perm_state, (size_t)n_aug * S * 4, cudaMemcpyHostToDevice, st) != cudaSuccess;
    rc |= cudaMemcpyAsync(d_pp, perm_policy, (size_t)n_aug * P * 4, cudaMemcpyHostToDevice, st) != cudaSuccess;
    k_augment<<<148 * 8, 256, 0, st>>>(d_s, d_p, (long long)n_pos, S, P, d_ps, d_pp, n_aug, d_so, d_po);
    rc |= cudaGetLastError() != cudaSuccess;
    rc |= cudaMemcpyAsync(states_out, d_so, bs * n_aug, cudaMemcpyDeviceToHost, st) != cudaSuccess;
    rc |= cudaMemcpyAsync(policies_out, d_po, bp * n_aug, cudaMemcpyDeviceToHost, st) != cudaSuccess;
    rc |= cudaStreamSynchronize(st) != cudaSuccess;
    if (rc) return done(fail("gaz_augment: %s", cudaGetErrorString(cudaGetLastError())));
    return done(0);
#endif
}

int gaz_eval_cache_enable(gaz_engine *e, int64_t entries, int shared_scope) {
    if (!e) return fail("null engine");
    if (e->cache) return fail("the evaluation cache is already enabled");
    // the cache key does not include the network: a hit could hand one network's output to the other's trees
    if (e->n_nets > 1) return fail("the evaluation cache cannot be used with more than one attached network");
    // a cache hit would return the symmetry drawn for the position's first evaluation
    if (e->sym && e->sym->mode != GAZ_SYM_NONE) return fail("the evaluation cache cannot be used with symmetric evaluation");
    if (entries < 1024) return fail("evaluation cache: at least 1024 entries");
    const View &v = e->v;
    gaz_eval_cache *c = new gaz_eval_cache();
    memset(c, 0, sizeof *c);
    c->entries = entries; c->scope = shared_scope ? 1 : 0; c->S = v.ncell * v.C; c->P = v.P; c->epoch = 0;
    const size_t NT = (size_t)v.n_trees, E = (size_t)entries;
    int rc = 0;
    rc |= ealloc(e, &c->state, E * c->S);
    rc |= ealloc(e, &c->tag, E);
    rc |= ealloc(e, &c->pol, E * c->P);
    rc |= ealloc(e, &c->val, E);
    rc |= ealloc(e, &c->claim, E);
    rc |= ealloc(e, &c->miss_idx, NT);
    rc |= ealloc(e, &c->miss_count, 4);
    rc |= ealloc(e, &c->packed_state, NT * c->S);
    rc |= ealloc(e, &c->packed_pol, NT * c->P);
    rc |= ealloc(e, &c->packed_val, NT);
    rc |= ealloc(e, &c->stats, 2);
    if (rc != 0) { delete c; return g_err.empty() ? fail("evaluation cache: allocation failed") : -1; }
    e->cache = c;
    e->view_epoch++;   // the captured round graph does not contain the cache passes
    return 0;
}

int gaz_eval_cache_stats(gaz_engine *e, int64_t *out) {
    if (!e || !out) return fail("null argument");
    out[0] = out[1] = out[2] = 0;
    if (!e->cache) return 0;
    unsigned long long st[2] = {0, 0};
    if (d2h(st, e->cache->stats, sizeof st, e->stream) != 0) return -1;
    out[0] = (int64_t)st[0]; out[1] = (int64_t)st[1]; out[2] = e->cache->entries;
    return 0;
}

int gaz_pool_info(gaz_engine *e, int64_t *out) {
    if (!e || !out) return fail("null argument");
    int32_t top = 0;
    if (d2h(&top, e->v.free_top, sizeof top, e->stream) != 0) return -1;
    out[0] = e->v.pool_pages; out[1] = top; out[2] = PAGE_SLOTS; out[3] = e->v.max_pages;
    return 0;
}

int64_t gaz_bytes_allocated(gaz_engine *e) { return e ? e->bytes : 0; }

} // extern "C"
