// gaz_internal.h -- engine internals shared by gaz_engine.cu and gaz_net.cu (not part of the ABI).
#pragma once
#include "../../include/gaz_b200.h"
#include "../../include/gaz_net.h"
#include "gaz_core.cuh"

#include <string>
#include <vector>

#ifndef GAZ_EMUL
#include <cuda_runtime.h>
#endif

int gaz_fail(const char *fmt, ...);

// ---------------------------------------------------------------- memory ----
#ifdef GAZ_EMUL
typedef int gaz_stream_t;
inline int dev_alloc(void **p, size_t n) { *p = calloc(1, n ? n : 1); return *p ? 0 : -1; }
inline void dev_free(void *p) { free(p); }
inline int h2d(void *d, const void *h, size_t n, gaz_stream_t) { memcpy(d, h, n); return 0; }
inline int d2h(void *h, const void *d, size_t n, gaz_stream_t) { memcpy(h, d, n); return 0; }
inline int dev_zero(void *d, size_t n, gaz_stream_t) { memset(d, 0, n); return 0; }
inline int stream_sync(gaz_stream_t) { return 0; }
#else
typedef cudaStream_t gaz_stream_t;
#define CK(x)                                                                                         \
    do {                                                                                              \
        cudaError_t _e = (x);                                                                         \
        if (_e != cudaSuccess) return gaz_fail("%s: %s (%s:%d)", #x, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)
inline int dev_alloc(void **p, size_t n) {
    CK(cudaMalloc(p, n ? n : 1));
    CK(cudaMemset(*p, 0, n ? n : 1));
    return 0;
}
inline void dev_free(void *p) { if (p) cudaFree(p); }
inline int h2d(void *d, const void *h, size_t n, gaz_stream_t s) {
    CK(cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, s));
    return 0;
}
inline int d2h(void *h, const void *d, size_t n, gaz_stream_t s) {
    CK(cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 0;
}
inline int dev_zero(void *d, size_t n, gaz_stream_t s) { CK(cudaMemsetAsync(d, 0, n, s)); return 0; }
inline int stream_sync(gaz_stream_t s) { CK(cudaStreamSynchronize(s)); return 0; }
#endif

struct gaz_engine {
    gaz_config cfg;
    gaz::View v;
    gaz_stream_t stream;
    int64_t bytes;
    std::vector<void *> allocs;
    // attached evaluators (gaz_net.cu): n_nets == 0 none, 1 every leaf goes to nets[0], >= 2 the leaves of tree t go to
    // nets[tree_net[t]] (gaz_attach_nets / gaz_set_tree_nets)
    struct gaz_net *nets[GAZ_MAX_NETS];
    int n_nets;
    uint8_t *d_tree_net;   // [n_trees], allocated with the route buffers
    int tree_net_max;      // largest index in the uploaded table (host copy)
    struct gaz_route *route; // packed per-network leaf lists, or null until two networks or a symmetry mode were set
    struct gaz_sym *sym;     // symmetric evaluation (gaz_set_eval_symmetry), or null until it was first set
    struct gaz_eval_cache *cache; // evaluation cache or null
    int leaf_bound;      // host-side upper bound of outstanding leaf requests (0 = n_trees)
    // CUDA graph of one search round (select -> network -> expand), built by gaz_net.cu on first use
    void *round_graph;   // cudaGraphExec_t
    unsigned attach_epoch, round_graph_attach; // bumped by every attach: the graph bakes in the attached network set
    uint64_t round_graph_chunks; // forward chunks of every attached network, 8 bits per network
    int round_graph_warm;
    // Kernels take the View BY VALUE, so a captured graph bakes in the hyper-parameters and pointers of its capture time.
    // Every setter that changes e->v bumps view_epoch; run_rounds re-captures when the graph's epoch is stale.
    unsigned view_epoch, round_graph_epoch;
    int32_t *d_limits;   // [n_trees]
    int16_t *d_actions;  // [n_trees]
    uint8_t *d_mask;     // [n_trees]
    int32_t *d_counter;  // scratch counter
    int32_t *d_winners;  // [n_games]
    double *d_noise;
    double *d_lut;
    float *d_pi;         // [MAXL]
    int8_t *d_states;    // [n_games][H*W*C] staging of gaz_get_states
    int32_t *d_ginfo;    // [n_games][4]
    uint64_t *d_keys;    // [n_trees] noise stream keys
    int8_t *d_cells;     // [n_games][ncell] staging of gaz_set_games
    int32_t *d_meta;     // [n_games][4]
    uint32_t *d_dense_vis; // [n_trees][P] staging of gaz_root_dense
    float *d_dense_val;
    int32_t *d_dense_info; // [n_trees][4]
#ifndef GAZ_EMUL
    cudaEvent_t ev0, ev1; // gaz_timer_begin / gaz_timer_end
#endif
};


// Evaluation cache (Session_Cache.Cache_Wrapper on the device, gaz_eval_cache_enable): direct-mapped table of evaluated
// positions.  A round's leaf requests are looked up first; the hits get their outputs at once, the misses are packed into a
// dense list that the evaluator serves, and a fill pass scatters the results back and stores them.
struct gaz_eval_cache {
    int64_t entries;
    int scope;                 // 0 = per game (the key includes the game's stream key / tree's game), 1 = shared by all games
    int S, P;
    int8_t *state;             // [entries][S]
    unsigned long long *tag;   // [entries]: 0 = empty, else hash | 1<<63
    float *pol;                // [entries][P]
    float *val;                // [entries]
    int32_t *claim;            // [entries]: fill epoch of the last writer (one writer per slot and pass)
    int32_t *miss_idx;         // [n_trees]: leaf index of packed miss m
    int32_t *miss_count;       // device counter
    int8_t *packed_state;      // [n_trees][S]
    float *packed_pol;         // [n_trees][P]
    float *packed_val;         // [n_trees]
    unsigned long long *stats; // [2]: look-ups, hits
    int epoch;
};
// look-up pass over the current leaf list / fill pass after the evaluator served the packed misses (stream-ordered)
int gaz_internal_cache_lookup(gaz_engine *e);
int gaz_internal_cache_fill(gaz_engine *e);

// Several attached networks (a match, a tournament): every round the leaf list is partitioned by the network of each
// leaf's tree, each network serves its own packed list and the outputs are scattered back to the leaf order (gaz_net.cu).
// Lists 0..n_alloc-1 are allocated; attaching more networks later allocates the missing ones.  A packed list holds `cap`
// rows: n_trees, or n_sym x n_trees while GAZ_SYM_ENSEMBLE evaluates every leaf under n_sym symmetries.
struct gaz_route {
    int n_alloc;
    size_t cap;
    int32_t *idx[GAZ_MAX_NETS];   // [n_trees]: leaf index of packed leaf m of network k
    int32_t *count;               // [GAZ_MAX_NETS] device counts (leaves)
    int32_t *rows;                // [GAZ_MAX_NETS] device counts of packed rows (symmetric evaluation)
    uint8_t *sym[GAZ_MAX_NETS];   // [n_trees]: GAZ_SYM_RANDOM's symmetry of packed leaf m of network k
    int8_t *state[GAZ_MAX_NETS];  // [cap][S]
    float *pol[GAZ_MAX_NETS];     // [cap][P]
    float *val[GAZ_MAX_NETS];     // [cap]
};
// Symmetric network evaluation (gaz_set_eval_symmetry): the tables live on the device as int16 (S, P <= 32767).
struct gaz_sym {
    int mode, n;                  // GAZ_SYM_*, rows of the tables
    uint64_t seed;
    int16_t *perm_state;          // [GAZ_MAX_SYM][S]
    int16_t *perm_policy;         // [GAZ_MAX_SYM][P]
};
// engine-owned device allocation (counted in gaz_bytes_allocated, freed with the engine, or earlier by gaz_internal_free)
int gaz_internal_alloc(gaz_engine *e, void **p, size_t bytes);
void gaz_internal_free(gaz_engine *e, void *p, size_t bytes);

int gaz_internal_launch_select(gaz_engine *e);
int gaz_internal_launch_expand(gaz_engine *e);
