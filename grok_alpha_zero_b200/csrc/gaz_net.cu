// gaz_net.cu -- policy/value network evaluator (include/gaz_net.h).
//
// Trunk convolutions (C_in in {64,128,256}, C_out in {32,64,128}) run as implicit GEMMs on the 5th-gen tensor cores
// (tcgen05.mma cta_group::2, bf16 x bf16 -> fp32 in TMEM, operands staged by TMA): gaz_conv.cuh (one convolution per
// launch, any board geometry; dx-merged head convolutions; tensor-core dense layers), gaz_block.cuh (whole residual blocks,
// up to six per launch, when a 256-row tile is a whole number of boards), gaz_stem.cuh (stems as implicit GEMMs, the Gomoku
// one fused with the first block's shortcut projection), gaz_small.cuh (small layers on mma.sync).  This file holds the
// remaining CUDA-core kernels - SE fallback, generic head convolution, fp32 dense layer, policy activation - and the executor
// that walks the op list of include/gaz_net.h: it decides the fusions (gaz_net_create), runs the two heads as two stream
// branches where they are separable and is captured into the search round's CUDA graph by gaz_engine.cu.
// Reference network definitions: */Build_Model.py, Net/ResNet/ResNet_Block.py:27-41,
// Net/SE/SE_Block.py:15-23, Net/Stablemax.py:7-11.
#include "../../include/gaz_net.h"
#include "gaz_internal.h"
#include "gaz_tc.cuh"
#include "gaz_conv.cuh"
#include "gaz_block.cuh"
#include "gaz_stem.cuh"
#include "gaz_small.cuh"

#include <cuda_bf16.h>
#include <math.h>
#include <stdio.h>

using namespace gaz_tc;
using gaz_conv::f32_blk_index;

#define CKN(x)                                                                                             \
    do {                                                                                                   \
        cudaError_t _e = (x);                                                                              \
        if (_e != cudaSuccess) return gaz_fail("%s: %s (%s:%d)", #x, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

// ====================================================================== CUDA-core kernels ==
struct SeArgs {
    const int32_t *count;
    int max_count, H, W, C, R, P_pad, Wp;
    const float *c2;  // conv2 output (+bias), fp32 padded rows
    const float *res; // residual stream
    const float *w1, *b1, *w2, *b2; // dense1 [C][R], dense2 [R][C]
    float *out_raw;
    __nv_bfloat16 *out_a, *out_b;
    const float *scale_a, *shift_a, *scale_b, *shift_b;
};

// Net/SE/SE_Block.py:15-23 + the block's skip add; one CTA per board, thread = channel.  Fallback for geometries
// where a board is not one 256-row tile (the fused epilogue of conv_board_kernel handles Gomoku).
__global__ void __launch_bounds__(128) se_kernel(SeArgs p) {
    __shared__ float s_mean[128], s_hid[64], s_gate[128];
    int cnt = *p.count;
    if (cnt > p.max_count) cnt = p.max_count;
    const int c = threadIdx.x;
    for (int b = blockIdx.x; b < cnt; b += gridDim.x) {
        const long long row0 = (long long)b * p.P_pad;
        float s = 0.0f;
        for (int y = 0; y < p.H; y++)
            for (int x = 0; x < p.W; x++) s += p.c2[f32_blk_index(row0 + (y + 1) * p.Wp + x, c, p.C)];
        s_mean[c] = s / (float)(p.H * p.W);
        __syncthreads();
        if (c < p.R) {
            float h = p.b1[c];
            for (int i = 0; i < p.C; i++) h = fmaf(s_mean[i], p.w1[i * p.R + c], h);
            s_hid[c] = fmaxf(h, 0.0f);
        }
        __syncthreads();
        {
            float g = p.b2[c];
            for (int i = 0; i < p.R; i++) g = fmaf(s_hid[i], p.w2[i * p.C + c], g);
            s_gate[c] = 1.0f / (1.0f + expf(-g));
        }
        const float gate = s_gate[c];
        for (int pos = 0; pos < p.P_pad; pos++) {
            const int yy = pos / p.Wp, xx = pos - yy * p.Wp;
            const bool live = yy != 0 && yy <= p.H && xx != p.Wp - 1;
            const size_t ob = f32_blk_index(row0 + pos, c, p.C);
            const size_t o = (size_t)(row0 + pos) * p.C + c;
            float v = live ? fmaf(p.c2[ob], gate, p.res[ob]) : 0.0f;
            if (p.out_raw) p.out_raw[ob] = v;
            if (p.out_a) p.out_a[o] = __float2bfloat16_rn(live ? fmaxf(fmaf(p.scale_a[c], v, p.shift_a[c]), 0.0f) : 0.0f);
            if (p.out_b) p.out_b[o] = __float2bfloat16_rn(live ? fmaxf(fmaf(p.scale_b[c], v, p.shift_b[c]), 0.0f) : 0.0f);
        }
        __syncthreads();
    }
}

struct HeadConvArgs {
    const int32_t *count;
    int max_count, H, W, Cin, Cout, K, P_pad, Wp, in_f32;
    long long in_rows;  // allocated rows of the input buffer
    const void *in;     // padded rows, bf16 or fp32
    const float *w;     // [K*K][Cin][Cout]
    const float *bias;
    float *out;         // flat [leaf][H*W*Cout] (H,W,C order)
    __nv_bfloat16 *out_act; // optional: relu(act_scale[f] * out + act_shift[f]) as bf16, same flat order (operand of a
    const float *act_scale, *act_shift; // tensor-core dense layer)
    int act_ld;         // row pitch of out_act in elements (features padded to a multiple of 8 for the TMA pitch rule)
};

// small convolutions of the heads (C_out <= 16): thread per (leaf, cell), weights in shared memory
__global__ void __launch_bounds__(128) headconv_kernel(HeadConvArgs p) {
    extern __shared__ float s_w[];
    const int nW = p.K * p.K * p.Cin * p.Cout;
    for (int i = threadIdx.x; i < nW; i += blockDim.x) s_w[i] = p.w[i];
    __syncthreads();
    int cnt = *p.count;
    if (cnt > p.max_count) cnt = p.max_count;
    const int ncell = p.H * p.W;
    const long long total = (long long)cnt * ncell;
    const int kh = p.K >> 1;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(idx / ncell), cell = (int)(idx - (long long)b * ncell);
        const int y = cell / p.W, x = cell - y * p.W;
        const long long r0 = (long long)b * p.P_pad + (y + 1) * p.Wp + x;
        float acc[16];
#pragma unroll
        for (int j = 0; j < 16; j++) acc[j] = j < p.Cout ? p.bias[j] : 0.0f;
        for (int ky = 0; ky < p.K; ky++)
            for (int kx = 0; kx < p.K; kx++) {
                const long long r = r0 + (ky - kh) * p.Wp + (kx - kh);
                if (r < 0 || r >= p.in_rows) continue;
                const float *wp = s_w + (size_t)((ky * p.K + kx) * p.Cin) * p.Cout;
                if (p.in_f32) {
                    for (int ci = 0; ci < p.Cin; ci++) {
                        const float a = ((const float *)p.in)[f32_blk_index(r, ci, p.Cin)];
#pragma unroll
                        for (int j = 0; j < 16; j++) if (j < p.Cout) acc[j] = fmaf(a, wp[ci * p.Cout + j], acc[j]);
                    }
                } else {
                    const __nv_bfloat16 *ip = (const __nv_bfloat16 *)p.in + r * p.Cin;
                    for (int ci = 0; ci < p.Cin; ci++) {
                        const float a = __bfloat162float(ip[ci]);
#pragma unroll
                        for (int j = 0; j < 16; j++) if (j < p.Cout) acc[j] = fmaf(a, wp[ci * p.Cout + j], acc[j]);
                    }
                }
            }
        float *op = p.out + (size_t)b * ncell * p.Cout + (size_t)cell * p.Cout;
#pragma unroll
        for (int j = 0; j < 16; j++) if (j < p.Cout) op[j] = acc[j];
    }
}

// Head convolutions on a 32-channel bf16 row tensor (Gomoku policy_conv1 3x3 32->8, value_conv1 1x1 32->4) on the
// warp-level tensor-core path (mma.sync m16n8k16 - far too small for a tcgen05 pipeline: 0.5 MFLOP per board).  One CTA
// stages a whole board (+ halo rows) in shared memory (64-byte rows, 16-byte chunks XOR-swizzled so ldmatrix is
// conflict-free); an M tile is 16 consecutive padded rows, a filter tap is a row shift of the ldmatrix addresses, N = 8
// output channels (zero padded), K = 32 input channels = 2 k-steps.  Weights stay fp32-accurate: every B fragment is
// split into bf16 hi + lo parts and issued as two MMAs (inputs are bf16 already, accumulation is fp32).
template <int K>
__global__ void __launch_bounds__(128) headconv_mma_kernel(HeadConvArgs p) {
    constexpr int TAPS = K * K, kh = K >> 1;
    extern __shared__ __align__(16) uint8_t s_board[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int halo = kh * (p.Wp + 1);
    const int n_mt = (p.P_pad + 15) >> 4;
    const int srows = n_mt * 16 + 2 * halo;
    // B fragments (k x n, "col" layout): this lane holds k = (lane & 3) * 2 + {0, 1} (+ 8 for the second register), n = lane >> 2.
    // They live in shared memory as [tap][k-step][lane] uint4 = {hi0, hi1, lo0, lo1} (one conflict-free LDS.128 per use):
    // in registers (72) they cap the kernel at 3 CTAs per SM.
    uint4 *s_frag = reinterpret_cast<uint4 *>(s_board + (size_t)srows * 64);
    if (warp == 0) {
        const int nn = lane >> 2, k0 = (lane & 3) * 2;
        for (int t = 0; t < TAPS; t++)
            for (int ks = 0; ks < 2; ks++) {
                uint32_t hi[2], lo[2];
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    float w2[2];
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int ci = ks * 16 + h * 8 + k0 + e;
                        w2[e] = nn < p.Cout ? p.w[(size_t)(t * 32 + ci) * p.Cout + nn] : 0.0f;
                    }
                    const __nv_bfloat16 h0 = __float2bfloat16_rn(w2[0]), h1 = __float2bfloat16_rn(w2[1]);
                    const __nv_bfloat16 l0 = __float2bfloat16_rn(w2[0] - __bfloat162float(h0)), l1 = __float2bfloat16_rn(w2[1] - __bfloat162float(h1));
                    hi[h] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
                    lo[h] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
                }
                s_frag[(t * 2 + ks) * 32 + lane] = make_uint4(hi[0], hi[1], lo[0], lo[1]);
            }
    }
    int cnt = *p.count;
    if (cnt > p.max_count) cnt = p.max_count;
    const int ncell = p.H * p.W;
    const uint4 *gin = reinterpret_cast<const uint4 *>(p.in); // 4 uint4 per 64-byte row
    uint4 *sin = reinterpret_cast<uint4 *>(s_board);
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(s_board);
    // ldmatrix.x4: lane -> (matrix mi = lane >> 3, row lane & 7); matrices = (rows 0-7 | 8-15) x (k 0-7 | 8-15)
    const int a_row = ((lane >> 3) & 1) * 8 + (lane & 7), a_chunk = lane >> 4;
    const float bias0 = (lane & 3) * 2 < p.Cout ? p.bias[(lane & 3) * 2] : 0.0f;
    const float bias1 = (lane & 3) * 2 + 1 < p.Cout ? p.bias[(lane & 3) * 2 + 1] : 0.0f;
    for (int b = blockIdx.x; b < cnt; b += gridDim.x) {
        __syncthreads();
        const long long g0 = ((long long)b * p.P_pad - halo) * 4;
        for (int i = threadIdx.x; i < srows * 4; i += blockDim.x) {
            const long long gi = g0 + i;
            const int row = i >> 2, ch = i & 3;
            sin[row * 4 + (ch ^ ((row >> 1) & 3))] = (gi >= 0 && gi < p.in_rows * 4) ? gin[gi] : make_uint4(0u, 0u, 0u, 0u);
        }
        __syncthreads();
        for (int mt = warp; mt < n_mt; mt += 4) {
            float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
            for (int t = 0; t < TAPS; t++) {
                const int sr = halo + mt * 16 + a_row + (t / K - kh) * p.Wp + (t % K - kh);
#pragma unroll
                for (int ks = 0; ks < 2; ks++) {
                    const uint32_t addr = sbase + (uint32_t)(sr * 64 + (((ks * 2 + a_chunk) ^ ((sr >> 1) & 3)) << 4));
                    uint32_t a0, a1, a2, a3;
                    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                                 : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3) : "r"(addr));
                    const uint4 bf = s_frag[(t * 2 + ks) * 32 + lane];
                    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                                 : "+f"(acc[0]), "+f"(acc[1]), "+f"(acc[2]), "+f"(acc[3])
                                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(bf.x), "r"(bf.y));
                    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                                 : "+f"(acc[0]), "+f"(acc[1]), "+f"(acc[2]), "+f"(acc[3])
                                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(bf.z), "r"(bf.w));
                }
            }
            // C fragment: acc[0..1] = row lane >> 2, columns (lane & 3) * 2 + {0, 1}; acc[2..3] = row + 8
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int pos = mt * 16 + (lane >> 2) + h * 8;
                const int yy = pos / p.Wp - 1, xx = pos % p.Wp;
                if (pos >= p.P_pad || yy < 0 || yy >= p.H || xx >= p.W) continue;
                const int cell = yy * p.W + xx;
                const int co = (lane & 3) * 2;           // Cout is even: the channel pair is in or out together
                if (co >= p.Cout) continue;
                const size_t f = (size_t)cell * p.Cout + co;
                const float v0 = acc[2 * h] + bias0, v1 = acc[2 * h + 1] + bias1;
                if (p.out_act) {
                    *reinterpret_cast<__nv_bfloat162 *>(p.out_act + (size_t)b * p.act_ld + f) =
                        __floats2bfloat162_rn(fmaxf(fmaf(p.act_scale[f], v0, p.act_shift[f]), 0.0f),
                                              fmaxf(fmaf(p.act_scale[f + 1], v1, p.act_shift[f + 1]), 0.0f));
                } else {
                    *reinterpret_cast<float2 *>(p.out + (size_t)b * ncell * p.Cout + f) = make_float2(v0, v1);
                }
            }
        }
    }
}

struct DenseArgs {
    const int32_t *count;
    int max_count, In, Out, act, pre_affine, pre_relu;
    const float *in;  // [leaf][In]
    const float *w;   // [In][Out]
    const float *bias;
    const float *pre_scale, *pre_shift;
    float *out;       // [leaf][Out]
};

// fp32 GEMM, 64x64 tile, 16-deep K slices, 4x4 outputs per thread.  The global loads of slice i+1 are issued before
// the FMAs of slice i (register prefetch): the small head GEMMs run one CTA per SM and were bound by load latency.
__global__ void __launch_bounds__(256) dense_kernel(DenseArgs p) {
    __shared__ float sA[16][64 + 1], sB[16][64 + 1];
    int cnt = *p.count;
    if (cnt > p.max_count) cnt = p.max_count;
    const int m0 = blockIdx.x * 64, n0 = blockIdx.y * 64;
    if (m0 >= cnt) return;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = 0.0f;
    float ra[4], rb[4];
    auto fetch = [&](int k0) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = threadIdx.x + u * 256;
            const int kk = i & 15, mm = i >> 4;
            const int k = k0 + kk, m = m0 + mm;
            float a = 0.0f;
            if (k < p.In && m < cnt) {
                a = p.in[(size_t)m * p.In + k];
                if (p.pre_affine) a = fmaf(p.pre_scale[k], a, p.pre_shift[k]);
                if (p.pre_relu) a = fmaxf(a, 0.0f);
            }
            ra[u] = a;
            const int nn = i & 63, kb = i >> 6;
            const int k2 = k0 + kb, n = n0 + nn;
            rb[u] = (k2 < p.In && n < p.Out) ? p.w[(size_t)k2 * p.Out + n] : 0.0f;
        }
    };
    fetch(0);
    for (int k0 = 0; k0 < p.In; k0 += 16) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = threadIdx.x + u * 256;
            sA[i & 15][i >> 4] = ra[u];
            sB[i >> 6][i & 63] = rb[u];
        }
        __syncthreads();
        if (k0 + 16 < p.In) fetch(k0 + 16);
#pragma unroll
        for (int kk = 0; kk < 16; kk++) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; i++) a[i] = sA[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; j++) b[j] = sB[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int m = m0 + ty * 4 + i;
        if (m >= cnt) continue;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int n = n0 + tx * 4 + j;
            if (n >= p.Out) continue;
            float v = acc[i][j] + p.bias[n];
            if (p.act == GAZ_ACT_RELU) v = fmaxf(v, 0.0f);
            else if (p.act == GAZ_ACT_TANH) v = tanhf(v);
            p.out[(size_t)m * p.Out + n] = v;
        }
    }
}

// "policy" output activation (Build_Model.py: softmax in float64 / Net/Stablemax.py / linear); warp per leaf
__global__ void __launch_bounds__(128) policy_out_kernel(const int32_t *count, int max_count, int P, int mode,
                                                         const float *logits, float *policy) {
    int cnt = *count;
    if (cnt > max_count) cnt = max_count;
    const int leaf = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (leaf >= cnt) return;
    const float *lg = logits + (size_t)leaf * P;
    float *po = policy + (size_t)leaf * P;
    if (mode == GAZ_POLICY_LINEAR) {
        for (int i = lane; i < P; i += 32) po[i] = lg[i];
        return;
    }
    if (mode == GAZ_POLICY_SOFTMAX) {
        double mx = -1e300;
        for (int i = lane; i < P; i += 32) mx = fmax(mx, (double)lg[i]);
        for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        double s = 0.0;
        for (int i = lane; i < P; i += 32) s += exp((double)lg[i] - mx);
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        for (int i = lane; i < P; i += 32) po[i] = (float)(exp((double)lg[i] - mx) / s);
        return;
    }
    float s = 0.0f;
    for (int i = lane; i < P; i += 32) {
        float x = lg[i];
        s += x >= 0.0f ? x + 1.0f : 1.0f / (1.0f - x);
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    for (int i = lane; i < P; i += 32) {
        float x = lg[i];
        po[i] = (x >= 0.0f ? x + 1.0f : 1.0f / (1.0f - x)) / s;
    }
}

__global__ void set_count_kernel(int32_t *c, int v) { *c = v; }
static constexpr int MAX_CHUNKS = 255;   // forward chunks per network and evaluation: 8 bits each in the round graph's key
// leaves [offset, offset + max) of the request list form one forward chunk
__global__ void chunk_count_kernel(const int32_t *total, int offset, int max, int32_t *out) {
    int c = *total - offset;
    *out = c < 0 ? 0 : (c > max ? max : c);
}

// ---- several attached networks (gaz_attach_nets): route the leaf list by network, serve each packed list, scatter back
// Stable K-way partition of the round's leaf list by tree_net[tree of the leaf]: network k gets the ascending leaf indices of
// its leaves in r.idx[k] and their number in r.count[k].  One CTA (a round has at most n_trees <= 32768 leaves) walks tiles
// of 1024 leaves, one per thread.  In a tile, a leaf's rank among the same-network leaves of its warp comes from
// __match_any_sync; the per-warp per-network counts are scanned (warp k scans network k's 32 warp counts) and added to the
// network's carry from the earlier tiles.
__global__ void __launch_bounds__(1024) route_leaves_kernel(const gaz::LeafRec *leaves, const int32_t *leaf_count,
                                                            const uint8_t *tree_net, int K, const gaz_route r) {
    __shared__ int off[GAZ_MAX_NETS][32];   // leaves of network k in warp w of the tile, then their first packed index
    __shared__ int carry[GAZ_MAX_NETS];     // leaves of network k in the earlier tiles
    __shared__ int tile[GAZ_MAX_NETS];
    const int n = *leaf_count, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x < GAZ_MAX_NETS) carry[threadIdx.x] = 0;
    for (int base = 0; base < n; base += 1024) {
        if (threadIdx.x < GAZ_MAX_NETS * 32) off[threadIdx.x >> 5][threadIdx.x & 31] = 0;
        __syncthreads();
        const int i = base + (int)threadIdx.x;
        const int k = i < n ? (int)tree_net[leaves[i].tree] : GAZ_MAX_NETS;   // lanes past the end form a group of their own
        const unsigned peers = __match_any_sync(0xffffffffu, k);
        const int rank = __popc(peers & ((1u << lane) - 1u));
        if (k < K && rank == 0) off[k][wid] = __popc(peers);
        __syncthreads();
        if (wid < K) {
            const int c = off[wid][lane];
            int x = c;
            for (int d = 1; d < 32; d <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, x, d);
                if (lane >= d) x += y;
            }
            off[wid][lane] = carry[wid] + x - c;
            if (lane == 31) tile[wid] = x;
        }
        __syncthreads();
        if (k < K) r.idx[k][off[k][wid] + rank] = i;
        if (threadIdx.x < K) carry[threadIdx.x] += tile[threadIdx.x];
        __syncthreads();
    }
    __syncthreads();
    if (threadIdx.x < K) r.count[threadIdx.x] = carry[threadIdx.x];
}

// packed row `row` of the concatenated lists (network 0's, then network 1's, ...) -> its network k and index m in k's list
__device__ __forceinline__ bool route_row(const int32_t *count, int K, int row, int &k, int &m) {
    int base = 0;
    for (k = 0; k < K; k++) {
        const int c = count[k];
        if (row < base + c) { m = row - base; return true; }
        base += c;
    }
    return false;
}

// warp per packed leaf: the input state of leaf idx_k[m] becomes packed row m of network k
__global__ void __launch_bounds__(128) route_states_kernel(const int8_t *leaf_state, int S, int K, const gaz_route r) {
    const int row = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    int k, m;
    if (!route_row(r.count, K, row, k, m)) return;
    const int8_t *src = leaf_state + (size_t)r.idx[k][m] * S;
    int8_t *dst = r.state[k] + (size_t)m * S;
    for (int j = lane; j < S; j += 32) dst[j] = src[j];
}

// warp per packed leaf: network k's policy row / value of packed leaf m go back to leaf idx_k[m] of the request list
__global__ void __launch_bounds__(128) scatter_evals_kernel(int P, int K, const gaz_route r, float *policy, float *value) {
    const int row = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    int k, m;
    if (!route_row(r.count, K, row, k, m)) return;
    const int leaf = r.idx[k][m];
    const float *src = r.pol[k] + (size_t)m * P;
    float *dst = policy + (size_t)leaf * P;
    for (int j = lane; j < P; j += 32) dst[j] = src[j];
    if (lane == 0) value[leaf] = r.val[k][m];
}

// ---- symmetric evaluation (gaz_set_eval_symmetry): route -> pack (leaf, g) rows through perm_state[g] -> each network's
// chunks -> map back through perm_policy[g] (and average the n_sym rows of a leaf in ENSEMBLE mode).
__device__ __forceinline__ uint64_t sym_mix(uint64_t z) {   // splitmix64 finaliser
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
    z ^= z >> 27; z *= 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// GAZ_SYM_RANDOM's choice for one request, computed by a whole warp; oracle/sym_hash.py is the bit-identical twin.
// acc = sum over the 8-byte little-endian words w_i of the state (zero-padded) of mix(w_i + (i + 1) * GOLD) mod 2^64;
// h = mix(mix(mix(seed + GOLD) ^ key) ^ acc); g = (h >> 32) % n.
__device__ __forceinline__ int sym_draw(const int8_t *st, int S, uint64_t seed, uint64_t key, int n, int lane) {
    const uint64_t GOLD = 0x9E3779B97F4A7C15ull;
    uint64_t acc = 0;
    for (int w = lane; w * 8 < S; w += 32) {
        uint64_t word = 0;
        for (int b = 0; b < 8 && w * 8 + b < S; b++) word |= (uint64_t)(uint8_t)st[w * 8 + b] << (8 * b);
        acc += sym_mix(word + (uint64_t)(w + 1) * GOLD);
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    const uint64_t h = sym_mix(sym_mix(sym_mix(seed + GOLD) ^ key) ^ acc);
    return (int)((h >> 32) % (uint64_t)n);
}

struct SymArgs {
    const int16_t *perm;          // [n][S] (pack) or [n][P] (scatter)
    int n, ensemble;              // table rows; 1 = every leaf gets n rows, 0 = one row of a drawn symmetry
    uint64_t seed;
    const uint64_t *tree_keys;    // per-tree keys or null (seed ^ tree)
    float inv_n;                  // 1 / n (ENSEMBLE average)
};

// warp per packed row.  Packed leaf m of network k (route_leaves_kernel) becomes rows m*n .. m*n+n-1 of k's list (ENSEMBLE,
// row m*n+g under symmetry g) or row m (RANDOM, under the drawn symmetry, kept in r.sym[k][m]); r.rows[k] = rows of k.
__global__ void __launch_bounds__(256) sym_states_kernel(const gaz::LeafRec *leaves, const int8_t *leaf_state, int S, int K,
                                                         const gaz_route r, const SymArgs a) {
    extern __shared__ int16_t s_perm[];   // [n][S]
    __shared__ int s_count[GAZ_MAX_NETS];
    for (int i = threadIdx.x; i < a.n * S; i += blockDim.x) s_perm[i] = a.perm[i];
    if (threadIdx.x < K) {
        s_count[threadIdx.x] = r.count[threadIdx.x];
        if (blockIdx.x == 0) r.rows[threadIdx.x] = r.count[threadIdx.x] * (a.ensemble ? a.n : 1);
    }
    __syncthreads();
    int total = 0;
    for (int k = 0; k < K; k++) total += s_count[k];
    const int per = a.ensemble ? a.n : 1, lane = threadIdx.x & 31;
    const int warps = (int)(gridDim.x * blockDim.x >> 5);
    for (int row = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < total * per; row += warps) {
        int k, m;
        route_row(s_count, K, row / per, k, m);
        const int leaf = r.idx[k][m];
        const int8_t *src = leaf_state + (size_t)leaf * S;
        int g = row % per;
        if (!a.ensemble) {
            const int tree = leaves[leaf].tree;
            const uint64_t key = a.tree_keys ? a.tree_keys[tree] : a.seed ^ (uint64_t)(uint32_t)tree;
            g = sym_draw(src, S, a.seed, key, a.n, lane);
            if (lane == 0) r.sym[k][m] = (uint8_t)g;
        }
        int8_t *dst = r.state[k] + ((size_t)m * per + (a.ensemble ? g : 0)) * S;
        const int16_t *pm = s_perm + g * S;
        for (int j = lane; j < S; j += 32) dst[j] = src[pm[j]];
    }
}

// warp per packed leaf: its row(s) go back to the leaf through perm_policy[g]; ENSEMBLE sums the n rows in g order in fp32
// and multiplies by 1/n (policy entries and value alike)
__global__ void __launch_bounds__(256) sym_scatter_kernel(int P, int K, const gaz_route r, const SymArgs a, float *policy,
                                                          float *value) {
    extern __shared__ int16_t s_perm[];   // [n][P]
    __shared__ int s_count[GAZ_MAX_NETS];
    for (int i = threadIdx.x; i < a.n * P; i += blockDim.x) s_perm[i] = a.perm[i];
    if (threadIdx.x < K) s_count[threadIdx.x] = r.count[threadIdx.x];
    __syncthreads();
    int total = 0;
    for (int k = 0; k < K; k++) total += s_count[k];
    const int lane = threadIdx.x & 31, warps = (int)(gridDim.x * blockDim.x >> 5);
    for (int row = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < total; row += warps) {
        int k, m;
        route_row(s_count, K, row, k, m);
        const int leaf = r.idx[k][m];
        float *dst = policy + (size_t)leaf * P;
        if (!a.ensemble) {
            const int g = r.sym[k][m];
            const float *src = r.pol[k] + (size_t)m * P;
            const int16_t *pm = s_perm + g * P;
            for (int j = lane; j < P; j += 32) dst[j] = src[pm[j]];
            if (lane == 0) value[leaf] = r.val[k][m];
            continue;
        }
        const float *src = r.pol[k] + (size_t)m * a.n * P;
        for (int j = lane; j < P; j += 32) {
            float s = 0.0f;
            for (int g = 0; g < a.n; g++) s += src[(size_t)g * P + s_perm[g * P + j]];
            dst[j] = s * a.inv_n;
        }
        if (lane == 0) {
            float s = 0.0f;
            for (int g = 0; g < a.n; g++) s += r.val[k][(size_t)m * a.n + g];
            value[leaf] = s * a.inv_n;
        }
    }
}

// ====================================================================== executor ==
typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct NetBuf { int kind, width; void *ptr; size_t bytes; };
struct NetOp {
    gaz_net_op d;
    CUtensorMap tmA2;     // activations: 152-row half-slab box
    CUtensorMap tmB2;     // weights: half of the output channels per CTA of a pair
    CUtensorMap tmOa, tmOb; // epilogue: bf16 outputs as 32-row x 32-channel SWIZZLE_64B store boxes
    int fused_se;         // this conv carries the following SE op in its epilogue
    gaz_net_op se;        // ... whose parameters are here
    int skip;             // SE op folded into the previous conv
    int block_fused;      // this conv1 runs the whole residual block (gaz_block.cuh) together with the next conv (+SE)
    int in_block;         // this conv2 is executed by the previous op's fused block kernel
    int trunk_len;        // block_fused conv1 that starts a launch: number of consecutive residual blocks the launch runs (1..MAX_LAYERS)
    int in_trunk;         // block_fused conv1 whose block runs inside an earlier op's trunk launch
    int dxm;              // 3x3 C -> 32 convolution run dx-merged (conv_board_kernel<96>): d_wt = filters repacked [dx*32+c][dy*Cin+k]
    int dual_partner;     // HEADCONV: index of a later head convolution on the same fp32 input that this op's launch computes
    int dual_skip;        // as well (gaz_small::headconv_wide_kernel, N = 16); dual_skip marks that later op
    int head_wide;        // HEADCONV on the fp32 stream through headconv_wide_kernel: d_frag / d_hbias are set
    int head_tc;          // HEADCONV (3x3, <= 8 + 8 outputs) on tcgen05 (conv_board_kernel<48>, dx-merged) reading the bf16 copy of the
                          // trunk output that the last residual block writes: tmA2 / tmB2 / d_wt / par[0..15] (biases) are set
    __nv_bfloat16 *d_xbf; // conv2 op of the last block: plain bf16 copy of its fp32 output (tmOa stores into it, no ReLU)
    uint4 *d_frag;        // mma.sync B fragments (stem_mma_kernel / headconv_wide_kernel)
    float *d_hbias;       // [16] biases of the (up to) two heads of a wide head convolution
    int head_G;           // boards per CTA iteration of the wide head convolution / the mma stem
    int chain_len;        // DENSE: this op starts a chain of chain_len dense layers run by ONE mlp_chain_kernel launch
    int chain_skip;       // DENSE executed by an earlier op's chain launch
    uint4 *d_frag0;       // DENSE chain start: layer 0's weights as mma.sync B fragments (hi | lo), or null (CUDA-core layer 0)
    int chain_partner;    // DENSE chain start: index of a later chain whose input is already complete; it runs in this launch (grid.y = 2)
    int chain_joined;     // DENSE chain start executed by an earlier chain's launch
    float par[5 * 128];   // host copy of bias | scale_a | shift_a | scale_b | shift_b for the kernel-argument bank
    float *d_se_b1;       // fused SE: dense1 bias with the conv bias folded in (b1 + W1^T bias)
    // dense layer on the tensor cores (DENSE op fed by a HEADCONV op): bf16 activated input + bf16 [Out][In] weights
    int dense_tc;
    __nv_bfloat16 *d_act; // [rows_dense][In]: written by the producing head convolution
    __nv_bfloat16 *d_wt;  // [Out][In]
    int stem_tc;          // stem on the tensor cores (gaz_stem.cuh): d_stem_w / d_stem_par / tmOa (out_a) / tmOb (out_q) are set
    int stem_tile;        // stem with 128 filters on tiles of whole boards (gaz_stem::stem_tile_kernel): d_stem_w / d_stem_par / tmOa set
    int stem_proj;        // ... and it also runs the next op, the 1x1 projection of the first block's shortcut (stem_proj_kernel)
    uint16_t *d_stem_w;   // [256][64] bf16 hi | lo split filters
    float *d_stem_par;    // stem_tc: [4][256] BN scale | shift + scale * bias | scale_a | shift_a; mma stem: [5][Cout] conv bias |
                          // BN scale | BN shift | scale_a | shift_a
    CUtensorMap tmDA, tmDW2;
    long long rows_dense;
};

// Activation workspace: every allocation of a network that scales with max_batch, in creation order.  Networks of one
// structure make the same allocations in the same order, so gaz_net_create_shared hands the i-th of them to the sharer.
// Reference-counted; freed with the last network that uses it.
struct NetWorkspace {
    int refs;
    std::vector<void *> ptrs;
    std::vector<size_t> bytes;
};

struct gaz_net {
    int game, H, W, Cin, P, Wp, P_pad, max_batch, policy_mode, device;
    NetWorkspace *ws;
    long long rows_alloc;
    std::vector<NetBuf> bufs;
    std::vector<NetOp> ops;
    float *wf;
    uint16_t *wh;
    int64_t bytes;
    int n_sm;
    cudaStream_t stream;
    cudaStream_t stream2;          // side stream of the second head (fork / join inside net_forward)
    cudaEvent_t ev_fork, ev_join;
    gaz_block::TrunkArgs *trunk_args;   // host staging of a trunk launch's arguments
    int head1_begin, head2_begin;  // op indices: first op of the first / second head; head2_begin = 0: the heads are not separable
    // I/O buffers for the host path (workspace)
    int8_t *d_states;
    int32_t *d_count;
    int32_t *d_chunk_count; // [chunk_cap] per-chunk leaf counts of an engine-driven forward
    int chunk_cap;          // 16, or MAX_CHUNKS once an ENSEMBLE evaluation needed more (reserve_chunk_counts)
    int32_t *d_chunk_count16; // the first 16-entry buffer after a growth (a round graph captured before may still read it)
    float *d_policy, *d_value;
    int logits_buf; // id of the flat buffer holding the policy logits
    // profiling of the tcgen05 conv launches
    int profile;
    int dbg;               // timing-experiment bits of the convolution kernels; always 0 unless built with -DGAZ_BLOCK_CLK
    std::vector<cudaEvent_t> ev;
    size_t ev_used;
    std::vector<int> ev_op;
};

static int make_map_ex(PFN_encodeTiled enc, CUtensorMap *m, void *ptr, uint64_t inner, uint64_t rows, uint32_t box_inner,
                       uint32_t box_rows, CUtensorMapSwizzle sw) {
    cuuint64_t dims[2] = {inner, rows};
    cuuint64_t strides[1] = {inner * 2};
    cuuint32_t box[2] = {box_inner, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return gaz_fail("cuTensorMapEncodeTiled failed (%d) inner=%llu rows=%llu box=%ux%u", (int)r,
                                           (unsigned long long)inner, (unsigned long long)rows, box_inner, box_rows);
    return 0;
}
static int make_map(PFN_encodeTiled enc, CUtensorMap *m, void *ptr, uint64_t inner, uint64_t rows, uint32_t box_rows) {
    return make_map_ex(enc, m, ptr, inner, rows, 64, box_rows, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <int BN> static int launch_conv_board(gaz_net *n, NetOp &op, const gaz_conv::BoardConvArgs &a, cudaStream_t s) {
    static bool attr_set = false;
    if (!attr_set) {
        CKN(cudaFuncSetAttribute(gaz_conv::conv_board_kernel<BN, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 gaz_conv::BoardCfg<BN, true>::SMEM));
        attr_set = true;
    }
    // CTA pairs: clusters of 2 (one TPC), the leader issues cta_group::2 MMAs for both
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3((unsigned)(n->n_sm & ~1), 1, 1);
    cfg.blockDim = dim3(384, 1, 1);
    cfg.dynamicSmemBytes = gaz_conv::BoardCfg<BN, true>::SMEM;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    CKN(cudaLaunchKernelEx(&cfg, gaz_conv::conv_board_kernel<BN, true>, op.tmA2, op.tmB2, op.tmOa, op.tmOb, a));
    return 0;
}

// one launch = trunk_len consecutive residual blocks starting at op `first` (gaz_block.cuh)
static int launch_res_trunk(gaz_net *n, size_t first, const int32_t *count, cudaStream_t s) {
    static bool attr_set = false;
    if (!attr_set) {
        CKN(cudaFuncSetAttribute(gaz_block::res_trunk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, gaz_block::Cfg::SMEM));
        attr_set = true;
    }
    auto buf = [&](int id) -> void * { return id < 0 ? nullptr : n->bufs[(size_t)id].ptr; };
    gaz_block::TrunkArgs &a = *n->trunk_args;   // 29 KB: kept off the stack (one per network); the launch copies it
    memset(&a, 0, sizeof a);
    a.count = count; a.max_count = n->max_batch; a.Wp = n->Wp; a.H = n->H; a.P_pad = n->P_pad; a.n_cells = n->H * n->W; a.dbg = n->dbg;
    a.n_layers = n->ops[first].trunk_len;
    size_t oi = first;
    for (int l = 0; l < a.n_layers; l++) {
        NetOp &c1 = n->ops[oi], &c2 = n->ops[oi + 1];
        gaz_block::TrunkLayer &L = a.L[l];
        L.tmA = c1.tmA2; L.tmW1 = c1.tmB2; L.tmW2 = c2.tmB2; L.tmOa = c2.tmOa; L.tmOb = c2.tmOb;
        L.nkc1 = c1.d.cin / 64;
        L.dep = l > 0;
        memcpy(L.par1, c1.par, sizeof L.par1);   // conv1 bias | BN2 scale | BN2 shift
        memcpy(L.par2, c2.par, sizeof L.par2);
        const gaz_net_op &o = c2.fused_se ? c2.se : c2.d;
        L.res = (const float *)buf(o.res_buf); L.out_raw = (float *)buf(o.out_raw);
        L.out_a = (__nv_bfloat16 *)buf(o.out_a); L.out_b = (__nv_bfloat16 *)buf(o.out_b);
        if (c2.d_xbf) { L.out_a = c2.d_xbf; L.plain_a = 1; }   // bf16(x) for a tensor-core head convolution (scale 1, shift 0, no ReLU)
        if (c2.fused_se) {
            L.se = 1; L.se_r = c2.se.cin;
            L.se_w1 = n->wf + c2.se.w2; L.se_b1 = c2.d_se_b1; L.se_w2 = n->wf + c2.se.w3; L.se_b2 = n->wf + c2.se.bias3;
        }
        oi += c2.fused_se ? 3 : 2;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3((unsigned)(n->n_sm & ~1), 1, 1);
    cfg.blockDim = dim3(512, 1, 1);
    cfg.dynamicSmemBytes = gaz_block::Cfg::SMEM;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    CKN(cudaLaunchKernelEx(&cfg, gaz_block::res_trunk_kernel, a));
    return 0;
}

static const float *wfp(gaz_net *n, int64_t off) { return off < 0 ? nullptr : n->wf + off; }

static int net_forward(gaz_net *n, const int8_t *states, const int32_t *count, float *policy, float *value, cudaStream_t s_main) {
    n->ev_used = n->profile ? n->ev_used : 0;
    // Two heads that share nothing but the trunk output run as two branches: the second head's ops go to the network's side
    // stream between a fork (event recorded where the first head starts) and a join at the end.  Inside a stream capture the
    // side stream joins the capture through the event wait, so the round graph gets two parallel branches.
    const bool two = n->head2_begin > 0;
    for (size_t oi = 0; oi < n->ops.size(); oi++) {
        if (two && (int)oi == n->head1_begin) {
            CKN(cudaEventRecord(n->ev_fork, s_main));
            CKN(cudaStreamWaitEvent(n->stream2, n->ev_fork, 0));
        }
        cudaStream_t s = (two && (int)oi >= n->head2_begin) ? n->stream2 : s_main;
        NetOp &op = n->ops[oi];
        const gaz_net_op &d = op.d;
        auto buf = [&](int id) -> void * { return id < 0 ? nullptr : n->bufs[(size_t)id].ptr; };
        switch (d.type) {
        case GAZ_OP_STEM: {
            if (op.stem_proj) {
                static bool attr_set = false;
                if (!attr_set) {
                    CKN(cudaFuncSetAttribute(gaz_stem::stem_proj_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, gaz_stem::ProjCfg::SMEM));
                    attr_set = true;
                }
                const gaz_net_op &pj = n->ops[oi + 1].d;
                gaz_stem::StemProjArgs t;
                t.count = count; t.max_count = n->max_batch; t.states = states; t.H = n->H; t.W = n->W; t.Wp = n->Wp;
                t.relu = d.act == GAZ_ACT_RELU; t.wpack = op.d_stem_w; t.par = op.d_stem_par;
                t.wproj = n->wh + pj.w; t.pbias = n->wf + pj.bias; t.out_res = (float *)buf(pj.out_raw);
                gaz_stem::stem_proj_kernel<<<n->n_sm, 512, gaz_stem::ProjCfg::SMEM, s>>>(op.tmOa, t);
                break;
            }
            if (op.stem_tc) {
                static bool attr_set = false;
                if (!attr_set) {
                    CKN(cudaFuncSetAttribute(gaz_stem::stem_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, gaz_stem::Cfg::SMEM));
                    attr_set = true;
                }
                gaz_stem::StemTcArgs t;
                t.count = count; t.max_count = n->max_batch; t.states = states; t.H = n->H; t.W = n->W; t.Wp = n->Wp;
                t.relu = d.act == GAZ_ACT_RELU; t.wpack = op.d_stem_w; t.par = op.d_stem_par;
                t.has_q = d.out_b >= 0; t.has_a = d.out_a >= 0;
                gaz_stem::stem_tc_kernel<<<2 * n->n_sm, 256, gaz_stem::Cfg::SMEM, s>>>(op.tmOb, op.tmOa, t);
                break;
            }
            if (op.stem_tile) {
                gaz_stem::StemTileArgs t;
                t.count = count; t.max_count = n->max_batch; t.states = states; t.H = n->H; t.W = n->W; t.Wp = n->Wp; t.P_pad = n->P_pad;
                t.act = d.act; t.wpack = op.d_stem_w; t.par = op.d_stem_par; t.out_raw = (float *)buf(d.out_raw); t.has_a = d.out_a >= 0;
                const int tiles = (int)(n->rows_alloc / 256);
                const int grid = tiles < 2 * n->n_sm ? tiles : 2 * n->n_sm;
#define STEM_TILE(K_, C_)                                                                                                       \
    do {                                                                                                                        \
        const int sm = gaz_stem::TileCfg<K_, C_>::smem(n->H, n->W, n->P_pad);                                                    \
        static bool attr_set = false;                                                                                           \
        if (!attr_set) {                                                                                                        \
            CKN(cudaFuncSetAttribute(gaz_stem::stem_tile_kernel<K_, C_>, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));      \
            attr_set = true;                                                                                                    \
        }                                                                                                                       \
        gaz_stem::stem_tile_kernel<K_, C_><<<grid, 256, sm, s>>>(op.tmOa, t);                                                    \
    } while (0)
                if (d.ksize == 3 && d.cin == 4) STEM_TILE(3, 4);
                else if (d.ksize == 3 && d.cin == 2) STEM_TILE(3, 2);
                else STEM_TILE(5, 2);
#undef STEM_TILE
                break;
            }
            {   // every other stem shape: implicit GEMM on mma.sync (gaz_small.cuh)
                gaz_small::StemMmaArgs a;
                a.count = count; a.max_count = n->max_batch; a.states = states; a.H = n->H; a.W = n->W; a.Cout = d.cout;
                a.P_pad = n->P_pad; a.Wp = n->Wp; a.act = d.act; a.G = op.head_G; a.frags = op.d_frag; a.par = op.d_stem_par;
                a.out_q = (__nv_bfloat16 *)buf(d.out_b); a.out_raw = (float *)buf(d.out_raw); a.out_a = (__nv_bfloat16 *)buf(d.out_a);
                const int groups = (int)((n->rows_alloc / n->P_pad + a.G) / a.G);
                const int grid = groups < 2 * n->n_sm ? groups : 2 * n->n_sm;
                size_t sm;
#define STEM_MMA(K_, C_)                                                                                                        \
    do {                                                                                                                        \
        sm = gaz_small::StemMmaCfg<K_, C_>::smem(n->H, n->W, d.cout, a.G);                                                       \
        static bool attr_set = false;                                                                                           \
        if (!attr_set) {                                                                                                        \
            CKN(cudaFuncSetAttribute(gaz_small::stem_mma_kernel<K_, C_>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024)); \
            attr_set = true;                                                                                                    \
        }                                                                                                                       \
        if (sm > 96 * 1024) return gaz_fail("stem: %zu bytes of shared memory", sm);                                             \
        gaz_small::stem_mma_kernel<K_, C_><<<grid, 256, sm, s>>>(a);                                                             \
    } while (0)
                if (d.ksize == 3 && d.cin == 2) STEM_MMA(3, 2);        // Gomoku-shaped boards with a stem the tcgen05 kernel does not cover
                else if (d.ksize == 3 && d.cin == 4) STEM_MMA(3, 4);   // Connect4
                else if (d.ksize == 5 && d.cin == 2) STEM_MMA(5, 2);   // TicTacToe
                else return gaz_fail("stem k=%d cin=%d unsupported", d.ksize, d.cin);
#undef STEM_MMA
            }
            break;
        }
        case GAZ_OP_CONV_TC: {
            if (op.in_block || op.in_trunk) break; // executed by an earlier op's block / trunk kernel
            if (n->profile && n->ev_used + 2 <= n->ev.size()) {
                n->ev_op.push_back((int)oi);
                CKN(cudaEventRecord(n->ev[n->ev_used++], s));
            }
            int rc;
            if (op.block_fused) {
                rc = launch_res_trunk(n, oi, count, s);
            } else {
                gaz_conv::BoardConvArgs a;
                memset(&a, 0, sizeof a);
                a.count = count; a.max_count = n->max_batch; a.P_pad = n->P_pad; a.Wp = n->Wp; a.H = n->H;
                a.taps = d.ksize * d.ksize; a.kpt = d.cin / 64; a.base_offset_mode = n->dbg;
                if (op.dxm) { a.taps = 3; a.dxm = 1; }
                const gaz_net_op &o = op.fused_se ? op.se : d; // outputs / residual of the fused SE op
                memcpy(a.par, op.par, sizeof a.par);
                a.res = (const float *)buf(o.res_buf); a.out_raw = (float *)buf(o.out_raw);
                a.out_a = (__nv_bfloat16 *)buf(o.out_a); a.out_b = (__nv_bfloat16 *)buf(o.out_b);
                if (op.fused_se) {
                    a.se = 1; a.se_r = op.se.cin; a.n_cells = n->H * n->W;
                    a.se_w1 = wfp(n, op.se.w2); a.se_b1 = wfp(n, op.se.bias2); a.se_w2 = wfp(n, op.se.w3); a.se_b2 = wfp(n, op.se.bias3);
                    a.se_b1 = op.d_se_b1; // conv bias folded into the dense1 bias (b1 + W1^T bias)
                }
                rc = op.dxm ? launch_conv_board<96>(n, op, a, s)
                     : d.cout == 128 ? launch_conv_board<128>(n, op, a, s) : d.cout == 64 ? launch_conv_board<64>(n, op, a, s)
                     : d.cout == 32 ? launch_conv_board<32>(n, op, a, s) : gaz_fail("conv_tc cout %d unsupported", d.cout);
            }
            if (rc != 0) return rc;
            if (n->profile && (n->ev_used & 1)) CKN(cudaEventRecord(n->ev[n->ev_used++], s));
            break;
        }
        case GAZ_OP_SE: {
            if (op.skip) break;
            SeArgs a;
            a.count = count; a.max_count = n->max_batch; a.H = n->H; a.W = n->W; a.C = d.cout; a.R = d.cin;
            a.P_pad = n->P_pad; a.Wp = n->Wp;
            a.c2 = (const float *)buf(d.in_buf); a.res = (const float *)buf(d.res_buf);
            a.w1 = wfp(n, d.w2); a.b1 = wfp(n, d.bias2); a.w2 = wfp(n, d.w3); a.b2 = wfp(n, d.bias3);
            a.out_raw = (float *)buf(d.out_raw); a.out_a = (__nv_bfloat16 *)buf(d.out_a); a.out_b = (__nv_bfloat16 *)buf(d.out_b);
            a.scale_a = wfp(n, d.scale_a); a.shift_a = wfp(n, d.shift_a); a.scale_b = wfp(n, d.scale_b); a.shift_b = wfp(n, d.shift_b);
            if (d.cout != 128 || d.cin > 64) return gaz_fail("SE supports C=128, R<=64");
            se_kernel<<<n->n_sm * 16, 128, 0, s>>>(a);
            break;
        }
        case GAZ_OP_HEADCONV: {
            if (op.dual_skip) break;
            if (op.head_tc) {     // bf16 copy of the trunk output -> both heads' 3x3 convolutions as one dx-merged tcgen05 pass
                gaz_conv::BoardConvArgs a;
                memset(&a, 0, sizeof a);
                a.count = count; a.max_count = n->max_batch; a.P_pad = n->P_pad; a.Wp = n->Wp; a.H = n->H; a.W = n->W;
                a.taps = 3; a.kpt = d.cin / 64; a.dxm = 1; a.base_offset_mode = 0;
                memcpy(a.par, op.par, sizeof a.par);
                a.head_out[0] = (float *)buf(d.out_raw); a.head_c[0] = d.cout;
                if (op.dual_partner >= 0) {
                    const NetOp &o2 = n->ops[(size_t)op.dual_partner];
                    a.head_out[1] = (float *)buf(o2.d.out_raw); a.head_c[1] = o2.d.cout;
                }
                if (launch_conv_board<48>(n, op, a, s) != 0) return -1;
                break;
            }
            if (op.head_wide) {   // fp32 trunk output -> both heads' small convolutions in one mma.sync pass (gaz_small.cuh)
                gaz_small::HeadWideArgs a;
                a.count = count; a.max_count = n->max_batch; a.H = n->H; a.W = n->W; a.Cin = d.cin; a.K = d.ksize;
                a.P_pad = n->P_pad; a.Wp = n->Wp; a.G = op.head_G; a.in_rows = n->rows_alloc; a.in = (const float *)buf(d.in_buf);
                a.frags = op.d_frag; a.bias = op.d_hbias; a.cout1 = d.cout; a.out1 = (float *)buf(d.out_raw);
                a.cout2 = 0; a.out2 = nullptr;
                if (op.dual_partner >= 0) {
                    const NetOp &o2 = n->ops[(size_t)op.dual_partner];
                    a.cout2 = o2.d.cout; a.out2 = (float *)buf(o2.d.out_raw);
                }
                const size_t sm = gaz_small::head_wide_smem(d.cin, d.ksize, n->P_pad, n->Wp, a.G);
                static size_t attr_sm = 0;
                if (sm > attr_sm) {
                    CKN(cudaFuncSetAttribute(gaz_small::headconv_wide_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
                    CKN(cudaFuncSetAttribute(gaz_small::headconv_wide_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
                    attr_sm = sm;
                }
                const int groups = (n->max_batch + a.G - 1) / a.G;
                if (d.ksize == 3) gaz_small::headconv_wide_kernel<3><<<groups < n->n_sm ? groups : n->n_sm, 512, sm, s>>>(a);
                else gaz_small::headconv_wide_kernel<1><<<groups < n->n_sm ? groups : n->n_sm, 512, sm, s>>>(a);
                break;
            }
            HeadConvArgs a;
            a.count = count; a.max_count = n->max_batch; a.H = n->H; a.W = n->W; a.Cin = d.cin; a.Cout = d.cout; a.K = d.ksize;
            a.P_pad = n->P_pad; a.Wp = n->Wp; a.in_f32 = n->bufs[(size_t)d.in_buf].kind == GAZ_BUF_ROWS_F32;
            a.in_rows = n->rows_alloc; a.in = buf(d.in_buf); a.w = wfp(n, d.w); a.bias = wfp(n, d.bias); a.out = (float *)buf(d.out_raw);
            a.out_act = nullptr; a.act_scale = a.act_shift = nullptr; a.act_ld = 0;
            if (oi + 1 < n->ops.size() && n->ops[oi + 1].dense_tc) {
                const NetOp &nx = n->ops[oi + 1];
                a.out_act = nx.d_act; a.act_scale = wfp(n, nx.d.scale_a); a.act_shift = wfp(n, nx.d.shift_a);
                a.act_ld = (nx.d.cin + 7) & ~7;
            }
            const size_t sm = (size_t)d.ksize * d.ksize * d.cin * d.cout * 4;
            if (d.cin == 32 && !a.in_f32 && ((d.cout == 8 && d.ksize == 3) || (d.cout == 4 && d.ksize == 1))) {
                const int halo = (d.ksize / 2) * (n->Wp + 1);
                const size_t smm = (size_t)(((n->P_pad + 15) / 16) * 16 + 2 * halo) * 64 + (size_t)d.ksize * d.ksize * 2 * 32 * 16;
                if (smm <= 48 * 1024 && (((d.cout * n->H * n->W + 7) & ~7) & 1) == 0) {
                    if (d.ksize == 3) headconv_mma_kernel<3><<<n->n_sm * 8, 128, smm, s>>>(a);
                    else headconv_mma_kernel<1><<<n->n_sm * 8, 128, smm, s>>>(a);
                    break;
                }
            }
            if (a.out_act) return gaz_fail("headconv feeding a tensor-core dense layer needs the mma.sync kernel (cin 32)");
            if (d.cout > 16 || sm > 48 * 1024) return gaz_fail("headconv shape unsupported (cout %d, %zu B weights)", d.cout, sm);
            headconv_kernel<<<n->n_sm * 16, 128, sm, s>>>(a);   // generic shapes: thread per cell, fp32 CUDA cores
            break;
        }
        case GAZ_OP_DENSE: {
            if (op.chain_skip || op.chain_joined) break;
            if (op.chain_len > 0) {   // the dense stack behind a head as one launch (gaz_small::mlp_chain_kernel)
                gaz_small::MlpArgs a[2];
                memset(a, 0, sizeof a);
                size_t sm = 0;
                const int nch = op.chain_partner >= 0 ? 2 : 1;
                for (int c = 0; c < nch; c++) {
                    const size_t o0 = c == 0 ? oi : (size_t)op.chain_partner;
                    const NetOp &co = n->ops[o0];
                    a[c].count = count; a[c].max_count = n->max_batch; a[c].n_layers = co.chain_len; a[c].in = (const float *)buf(co.d.in_buf);
                    a[c].frag0 = co.d_frag0;
                    for (int li = 0; li < co.chain_len; li++) {
                        const gaz_net_op &dl = n->ops[o0 + (size_t)li].d;
                        gaz_small::MlpLayer &L = a[c].L[li];
                        L.In = dl.cin; L.Out = dl.cout; L.pre_affine = dl.flags & 1; L.pre_relu = (dl.flags >> 1) & 1; L.act = dl.act;
                        L.w = wfp(n, dl.w); L.bias = wfp(n, dl.bias); L.pre_scale = wfp(n, dl.scale_a); L.pre_shift = wfp(n, dl.shift_a);
                        if (li + 1 == co.chain_len) a[c].out = (dl.flags & 4) ? value : (float *)buf(dl.out_raw);
                    }
                    const size_t smc = gaz_small::mlp_smem(a[c], 32);
                    sm = smc > sm ? smc : sm;
                }
                // 32 leaves per CTA once that still leaves about three CTAs per SM, else 16
                const bool wide = (long long)((n->max_batch + 31) / 32) * nch >= 3LL * n->n_sm / 2;
                static size_t attr_sm = 48 * 1024;
                if (sm > attr_sm) {
                    CKN(cudaFuncSetAttribute(gaz_small::mlp_chain_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
                    CKN(cudaFuncSetAttribute(gaz_small::mlp_chain_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
                    attr_sm = sm;
                }
                const int tl = wide ? 32 : 16;
                dim3 grid((unsigned)((n->max_batch + tl - 1) / tl), (unsigned)nch);
                if (wide) gaz_small::mlp_chain_kernel<32><<<grid, 256, sm, s>>>(a[0], a[1]);
                else gaz_small::mlp_chain_kernel<16><<<grid, 256, sm, s>>>(a[0], a[1]);
                break;
            }
            if (op.dense_tc) { // [leaf][In] bf16 x [Out][In] bf16 on the board kernel: rows = leaves, 128 outputs per launch
                float *outp = (d.flags & 4) ? value : (float *)buf(d.out_raw);
                {   // one launch: work items are (row tile, 128-wide output slice) pairs (cout <= 512: the biases of up to four
                    // slices travel in par[0..511])
                    gaz_conv::BoardConvArgs a;
                    memset(&a, 0, sizeof a);
                    a.count = count; a.max_count = n->max_batch; a.P_pad = 1; a.Wp = 1;
                    a.taps = 1; a.kpt = (d.cin + 63) / 64; a.base_offset_mode = 0;
                    for (int c = 0; c < 512; c++) a.par[c] = c < d.cout ? op.par[c] : 0.0f;
                    a.dense = 1; a.n_off = 0; a.n_slices = (d.cout + 127) / 128; a.flat_out = outp; a.flat_ld = d.cout; a.flat_n = d.cout;
                    NetOp tmp = op; // maps: activations of this dense op, weights
                    tmp.tmA2 = op.tmDA; tmp.tmB2 = op.tmDW2;
                    if (launch_conv_board<128>(n, tmp, a, s) != 0) return -1;
                }
                break;
            }
            DenseArgs a;
            a.count = count; a.max_count = n->max_batch; a.In = d.cin; a.Out = d.cout; a.act = d.act;
            a.pre_affine = d.flags & 1; a.pre_relu = (d.flags >> 1) & 1;
            a.in = (const float *)buf(d.in_buf); a.w = wfp(n, d.w); a.bias = wfp(n, d.bias);
            a.pre_scale = wfp(n, d.scale_a); a.pre_shift = wfp(n, d.shift_a);
            a.out = (d.flags & 4) ? value : (float *)buf(d.out_raw);
            dim3 grid((unsigned)((n->max_batch + 63) / 64), (unsigned)((d.cout + 63) / 64));
            dense_kernel<<<grid, 256, 0, s>>>(a);
            break;
        }
        case GAZ_OP_POLICY_OUT: {
            policy_out_kernel<<<(n->max_batch + 3) / 4, 128, 0, s>>>(count, n->max_batch, n->P, n->policy_mode,
                                                                     (const float *)buf(d.in_buf), policy);
            break;
        }
        default:
            return gaz_fail("unknown op type %d", d.type);
        }
    }
    if (two) {
        CKN(cudaEventRecord(n->ev_join, n->stream2));
        CKN(cudaStreamWaitEvent(s_main, n->ev_join, 0));
    }
    CKN(cudaGetLastError());
    return 0;
}

extern "C" {

// first structural difference between `desc` and network `s`, or 0 if a network of `desc` may share s's workspace
static int structure_mismatch(const gaz_net_desc *desc, const gaz_net *s) {
    if (desc->game != s->game) return gaz_fail("shared workspace: game %d != %d", desc->game, s->game);
    if (desc->device != s->device) return gaz_fail("shared workspace: device %d != %d", desc->device, s->device);
    if (desc->max_batch != s->max_batch) return gaz_fail("shared workspace: max_batch %d != %d", desc->max_batch, s->max_batch);
    if (desc->n_bufs != (int)s->bufs.size()) return gaz_fail("shared workspace: %d buffers != %d", desc->n_bufs, (int)s->bufs.size());
    for (int i = 0; i < desc->n_bufs; i++)
        if (desc->bufs[i].kind != s->bufs[(size_t)i].kind || desc->bufs[i].width != s->bufs[(size_t)i].width)
            return gaz_fail("shared workspace: buffer %d is (kind %d, width %d), the shared network's is (kind %d, width %d)", i,
                            desc->bufs[i].kind, desc->bufs[i].width, s->bufs[(size_t)i].kind, s->bufs[(size_t)i].width);
    if (desc->n_ops != (int)s->ops.size()) return gaz_fail("shared workspace: %d ops != %d", desc->n_ops, (int)s->ops.size());
    for (int i = 0; i < desc->n_ops; i++) {
        const gaz_net_op &a = desc->ops[i], &b = s->ops[(size_t)i].d;
        const char *field = a.type != b.type ? "type" : a.in_buf != b.in_buf ? "in_buf" : a.res_buf != b.res_buf ? "res_buf"
                          : a.out_raw != b.out_raw ? "out_raw" : a.out_a != b.out_a ? "out_a" : a.out_b != b.out_b ? "out_b"
                          : a.cin != b.cin ? "cin" : a.cout != b.cout ? "cout" : a.ksize != b.ksize ? "ksize"
                          : a.act != b.act ? "act" : a.flags != b.flags ? "flags" : nullptr;
        if (field) return gaz_fail("shared workspace: op %d differs in %s from the shared network's", i, field);
    }
    return 0;
}

int gaz_net_create(const gaz_net_desc *desc, gaz_net **out) { return gaz_net_create_shared(desc, nullptr, out); }

int gaz_net_create_shared(const gaz_net_desc *desc, gaz_net *share, gaz_net **out) {
    if (!desc || !out) return gaz_fail("null argument");
    if (share && structure_mismatch(desc, share) != 0) return -1;
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev <= 0) return gaz_fail("no CUDA device (%s): the network has no CPU path", cudaGetErrorString(ce));
    CKN(cudaSetDevice(desc->device));
    PFN_encodeTiled enc = nullptr;
    {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        CKN(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess) return gaz_fail("cuTensorMapEncodeTiled not available");
        enc = (PFN_encodeTiled)fn;
    }
    gaz_net *n = new gaz_net();
    if (share) { n->ws = share->ws; n->ws->refs++; }
    else { n->ws = new NetWorkspace(); n->ws->refs = 1; }
    n->game = desc->game;
    if (desc->game == GAZ_GAME_TICTACTOE) { n->H = 3; n->W = 3; n->Cin = 2; n->P = 9; }
    else if (desc->game == GAZ_GAME_CONNECT4) { n->H = 6; n->W = 7; n->Cin = 4; n->P = 7; }
    else { n->H = 15; n->W = 15; n->Cin = 2; n->P = 225; }
    n->Wp = n->W + 1;
    // rows per board: (H+1) x (W+1) padded positions, rounded up to a divisor of the 256-row tile where possible (Connect4:
    // 56 -> 64, so a tile is four whole boards and the fused residual-block kernel applies; Gomoku 256, TicTacToe 16); the
    // extra rows are dead like the padding row and column
    n->P_pad = (n->H + 1) * n->Wp;
    if (n->P_pad <= 256) { int r = 16; while (r < n->P_pad) r <<= 1; n->P_pad = r; }
    n->max_batch = desc->max_batch;
    n->policy_mode = desc->policy_mode;
    n->device = desc->device;
    n->rows_alloc = (((long long)n->max_batch * n->P_pad + 255) / 256) * 256;
    n->bytes = 0;
    n->dbg = 0;
#ifdef GAZ_BLOCK_CLK   // instrumented A/B builds only (tools/build_variant.sh): timing-experiment bits of the convolution kernels
    { const char *e = getenv("GAZ_CONV_DBG"); n->dbg = e ? atoi(e) : 0; }
#endif
    n->profile = 0;
    n->ev_used = 0;
    n->logits_buf = -1;
    cudaDeviceProp prop;
    CKN(cudaGetDeviceProperties(&prop, desc->device));
    n->n_sm = prop.multiProcessorCount;
    CKN(cudaStreamCreateWithFlags(&n->stream, cudaStreamNonBlocking));
    CKN(cudaStreamCreateWithFlags(&n->stream2, cudaStreamNonBlocking));
    CKN(cudaEventCreateWithFlags(&n->ev_fork, cudaEventDisableTiming));
    CKN(cudaEventCreateWithFlags(&n->ev_join, cudaEventDisableTiming));
    n->head1_begin = 0; n->head2_begin = 0;
    n->trunk_args = new gaz_block::TrunkArgs();
    auto alloc = [&](void **p, size_t bytes) -> int {
        CKN(cudaMalloc(p, bytes ? bytes : 16));
        CKN(cudaMemset(*p, 0, bytes ? bytes : 16));
        n->bytes += (int64_t)bytes;
        return 0;
    };
    size_t ws_next = 0;   // allocations of the workspace taken so far
    auto walloc = [&](void **p, size_t bytes) -> int {
        if (share) {
            if (ws_next >= n->ws->ptrs.size() || n->ws->bytes[ws_next] != bytes)
                return gaz_fail("shared workspace: activation allocation %d (%zu bytes) has no match", (int)ws_next, bytes);
            *p = n->ws->ptrs[ws_next++];
            return 0;
        }
        if (alloc(p, bytes) != 0) return -1;
        n->ws->ptrs.push_back(*p);
        n->ws->bytes.push_back(bytes);
        return 0;
    };
    int rc = 0;
    rc |= alloc((void **)&n->wf, (size_t)desc->n_wf * 4);
    rc |= alloc((void **)&n->wh, (size_t)desc->n_wh * 2);
    if (rc == 0 && desc->n_wf) CKN(cudaMemcpy(n->wf, desc->wf, (size_t)desc->n_wf * 4, cudaMemcpyHostToDevice));
    if (rc == 0 && desc->n_wh) CKN(cudaMemcpy(n->wh, desc->wh, (size_t)desc->n_wh * 2, cudaMemcpyHostToDevice));
    for (int i = 0; i < desc->n_bufs && rc == 0; i++) {
        NetBuf b;
        b.kind = desc->bufs[i].kind;
        b.width = desc->bufs[i].width;
        if (b.kind == GAZ_BUF_ROWS_BF16) b.bytes = (size_t)n->rows_alloc * b.width * 2;
        else if (b.kind == GAZ_BUF_ROWS_F32) b.bytes = (size_t)n->rows_alloc * b.width * 4;
        else b.bytes = (size_t)n->max_batch * b.width * 4;
        b.ptr = nullptr;
        rc |= walloc(&b.ptr, b.bytes);
        n->bufs.push_back(b);
    }
    rc |= walloc((void **)&n->d_states, (size_t)n->max_batch * n->H * n->W * n->Cin);
    rc |= alloc((void **)&n->d_count, 16);
    rc |= alloc((void **)&n->d_chunk_count, 16 * 4);
    n->chunk_cap = 16;
    n->d_chunk_count16 = nullptr;
    rc |= walloc((void **)&n->d_policy, (size_t)n->max_batch * n->P * 4);
    rc |= walloc((void **)&n->d_value, (size_t)n->max_batch * 4);
    if (rc != 0) { gaz_net_destroy(n); return -1; }
    for (int i = 0; i < desc->n_ops; i++) {
        NetOp op;
        op.d = desc->ops[i];
        memset(&op.tmA2, 0, sizeof op.tmA2);
        memset(&op.tmB2, 0, sizeof op.tmB2);
        op.fused_se = 0;
        op.skip = 0;
        op.block_fused = 0;
        op.in_block = 0;
        op.trunk_len = 0; op.in_trunk = 0;
        op.dxm = 0;
        op.dual_partner = -1;
        op.dual_skip = 0;
        op.head_tc = 0; op.d_xbf = nullptr;
        op.head_wide = 0; op.d_frag = nullptr; op.d_hbias = nullptr; op.head_G = 1; op.chain_len = 0; op.chain_skip = 0; op.chain_partner = -1; op.chain_joined = 0; op.d_frag0 = nullptr;
        op.stem_tc = 0;
        op.stem_tile = 0;
        op.stem_proj = 0;
        op.d_stem_w = nullptr;
        op.d_stem_par = nullptr;
        op.d_se_b1 = nullptr;
        op.dense_tc = 0; op.d_act = nullptr; op.d_wt = nullptr; op.rows_dense = 0;
        memset(&op.se, 0, sizeof op.se);
        const gaz_net_op &d = op.d;
        if (d.type == GAZ_OP_CONV_TC) {
            if (d.cin % 64 != 0 || (d.cout != 32 && d.cout != 64 && d.cout != 128) || (d.ksize != 1 && d.ksize != 3)) {
                gaz_net_destroy(n);
                return gaz_fail("conv_tc op %d: unsupported shape cin=%d cout=%d k=%d", i, d.cin, d.cout, d.ksize);
            }
            const NetBuf &ib = n->bufs[(size_t)d.in_buf];
            if (ib.kind != GAZ_BUF_ROWS_BF16 || ib.width != d.cin) {
                gaz_net_destroy(n);
                return gaz_fail("conv_tc op %d: input buffer must be bf16 rows of width cin", i);
            }
            if (make_map(enc, &op.tmA2, ib.ptr, (uint64_t)d.cin, (uint64_t)n->rows_alloc, gaz_conv::SLAB_BOX_ROWS) != 0 ||
                make_map(enc, &op.tmB2, n->wh + d.w, (uint64_t)d.ksize * d.ksize * d.cin, (uint64_t)d.cout, (uint32_t)d.cout / 2) != 0) {
                gaz_net_destroy(n);
                return -1;
            }
            // 3x3 convolutions with 32 outputs and one bf16 output (the C128 -> C32 head convolutions): dx-merged form, the
            // three taps of a filter row side by side as N = 96 (gaz_conv.cuh).  Needs whole boards per tile and a row pitch
            // that divides the 32 rows of an epilogue warp.
#ifndef GAZ_NO_DXM         // A/B builds only
            if (d.cout == 32 && d.ksize == 3 && gaz_conv::TILE_ROWS % n->P_pad == 0 && 32 % n->Wp == 0 && d.out_a >= 0 && d.out_b < 0 &&
                d.out_raw < 0 && d.res_buf < 0 && (n->n_sm & ~1) >= 2) {
                const size_t ld = (size_t)3 * d.cin;
                std::vector<uint16_t> wt((size_t)96 * ld);
                for (int dy = 0; dy < 3; dy++)
                    for (int dx = 0; dx < 3; dx++)
                        for (int c = 0; c < 32; c++)
                            memcpy(&wt[(size_t)(dx * 32 + c) * ld + (size_t)dy * d.cin], desc->wh + d.w + (size_t)c * 9 * d.cin + (size_t)(dy * 3 + dx) * d.cin,
                                   (size_t)d.cin * 2);
                if (alloc((void **)&op.d_wt, wt.size() * 2) != 0) { gaz_net_destroy(n); return -1; }
                CKN(cudaMemcpy(op.d_wt, wt.data(), wt.size() * 2, cudaMemcpyHostToDevice));
                if (make_map(enc, &op.tmB2, op.d_wt, (uint64_t)ld, 96, 48) != 0) { gaz_net_destroy(n); return -1; }
                op.dxm = 1;
            }
#endif
        }
        if (d.type == GAZ_OP_POLICY_OUT) n->logits_buf = d.in_buf;
        // fold an SE op into the epilogue of the convolution that feeds it (tile == board geometries only)
        if (d.type == GAZ_OP_SE && n->P_pad == gaz_conv::TILE_ROWS && !n->ops.empty()) {
            NetOp &prev = n->ops.back();
            if (prev.d.type == GAZ_OP_CONV_TC && prev.d.out_raw == d.in_buf && prev.d.out_a < 0 && prev.d.out_b < 0 &&
                prev.d.res_buf < 0 && prev.d.cout == d.cout && d.cout == 128 && d.cin <= 64 && (d.cin & 1) == 0) {   // fused SE: R <= 64, even
                prev.fused_se = 1;
                prev.se = d;
                op.skip = 1;
            }
        }
        n->ops.push_back(op);
    }
    // dense layers fed by a head convolution and followed by nothing exotic go to the tensor cores:
    // DENSE with pre-affine + pre-relu, Out % 128 == 0, In * 2 bytes % 16 == 0 (TMA pitch), producer = HEADCONV on bf16 rows
    for (size_t oi = 1; oi < n->ops.size(); oi++) {
        NetOp &op = n->ops[oi];
        const gaz_net_op &d = op.d;
        if (d.type != GAZ_OP_DENSE || (d.flags & 3) != 3 || (d.flags & 4) || d.act != GAZ_ACT_NONE) continue;
        const NetOp &pr = n->ops[oi - 1];
        if (pr.d.type != GAZ_OP_HEADCONV || pr.d.out_raw != d.in_buf || pr.d.cin != 32) continue;
        if (n->bufs[(size_t)pr.d.in_buf].kind != GAZ_BUF_ROWS_BF16) continue;
        if (d.cout % 128 != 0 || d.cout > 512 || d.cin > 4096) continue;
        const int in_pad = (d.cin + 7) & ~7; // TMA row pitch must be a multiple of 16 bytes
        if (!((pr.d.cout == 8 && pr.d.ksize == 3) || (pr.d.cout == 4 && pr.d.ksize == 1))) continue; // headconv_board_kernel shapes
        op.rows_dense = (((long long)n->max_batch + 255) / 256) * 256;
        if (walloc((void **)&op.d_act, (size_t)op.rows_dense * in_pad * 2) != 0) { gaz_net_destroy(n); return -1; }
        std::vector<uint16_t> wt((size_t)d.cout * in_pad, (uint16_t)0);
        for (int i = 0; i < d.cin; i++)
            for (int o = 0; o < d.cout; o++) {
                float f = desc->wf[d.w + (int64_t)i * d.cout + o];
                uint32_t u; memcpy(&u, &f, 4);
                u = (u + 0x7FFFu + ((u >> 16) & 1u)) >> 16;      // round to nearest even bf16
                wt[(size_t)o * in_pad + i] = (uint16_t)u;
            }
        if (alloc((void **)&op.d_wt, wt.size() * 2) != 0) { gaz_net_destroy(n); return -1; }
        CKN(cudaMemcpy(op.d_wt, wt.data(), wt.size() * 2, cudaMemcpyHostToDevice));
        if (make_map(enc, &op.tmDA, op.d_act, (uint64_t)in_pad, (uint64_t)op.rows_dense, gaz_conv::SLAB_BOX_ROWS) != 0 ||
            make_map(enc, &op.tmDW2, op.d_wt, (uint64_t)in_pad, (uint64_t)d.cout, 64) != 0) { gaz_net_destroy(n); return -1; }
        for (int c = 0; c < 640; c++) op.par[c] = 0.0f;
        for (int o = 0; o < d.cout && o < 640; o++) op.par[o] = desc->wf[d.bias + o]; // bias of up to 640 outputs
        op.dense_tc = 1;
    }
    for (auto &op : n->ops) { // per-channel epilogue parameters of the tensor-core convolutions (host copies)
        if (op.d.type != GAZ_OP_CONV_TC) continue;
        const gaz_net_op &o = op.fused_se ? op.se : op.d;
        memset(&op.tmOa, 0, sizeof op.tmOa);
        memset(&op.tmOb, 0, sizeof op.tmOb);
        for (int k = 0; k < 2; k++) {
            const int id = k == 0 ? o.out_a : o.out_b;
            if (id < 0) continue;
            const NetBuf &ob = n->bufs[(size_t)id];
            if (ob.kind != GAZ_BUF_ROWS_BF16 || ob.width != op.d.cout) { gaz_net_destroy(n); return gaz_fail("conv_tc output buffer must be bf16 rows of width cout"); }
            if (make_map_ex(enc, k == 0 ? &op.tmOa : &op.tmOb, ob.ptr, (uint64_t)ob.width, (uint64_t)n->rows_alloc, 32, 32,
                            CU_TENSOR_MAP_SWIZZLE_64B) != 0) { gaz_net_destroy(n); return -1; }
        }
        const int64_t offs[5] = {op.d.bias, o.scale_a, o.shift_a, o.scale_b, o.shift_b};
        const float dflt[5] = {0.0f, 1.0f, 0.0f, 1.0f, 0.0f};
        for (int k = 0; k < 5; k++)
            for (int c = 0; c < 128; c++)
                op.par[k * 128 + c] = (offs[k] >= 0 && c < op.d.cout) ? desc->wf[offs[k] + c] : dflt[k];
        if (op.fused_se) {
            const int R = op.se.cin, Cc = op.d.cout;
            std::vector<float> b1((size_t)R);
            for (int j = 0; j < R; j++) {
                double acc = desc->wf[op.se.bias2 + j];
                for (int i = 0; i < Cc; i++) acc += (double)op.par[i] * (double)desc->wf[op.se.w2 + (int64_t)i * R + j];
                b1[(size_t)j] = (float)acc;
            }
            if (alloc((void **)&op.d_se_b1, (size_t)R * 4) != 0) { gaz_net_destroy(n); return -1; }
            CKN(cudaMemcpy(op.d_se_b1, b1.data(), (size_t)R * 4, cudaMemcpyHostToDevice));
        }
    }
    // whole-block fusion: conv1 (3x3 C128|C256 -> C128, bf16 out only) directly followed by conv2 (3x3 C128->C128 reading it)
    if (gaz_conv::TILE_ROWS % n->P_pad == 0 && (n->n_sm & ~1) >= 2) {   // a tile is a whole number of boards
        for (size_t oi = 0; oi + 1 < n->ops.size(); oi++) {
            NetOp &c1 = n->ops[oi], &c2 = n->ops[oi + 1];
            if (c1.d.type != GAZ_OP_CONV_TC || c2.d.type != GAZ_OP_CONV_TC || c1.block_fused || c1.in_block) continue;
            if ((c1.d.cin != 128 && c1.d.cin != 256) || c1.d.cout != 128 || c1.d.ksize != 3 || c2.d.cin != 128 || c2.d.cout != 128 || c2.d.ksize != 3) continue;
            if (c1.d.out_a < 0 || c1.d.out_b >= 0 || c1.d.out_raw >= 0 || c1.d.res_buf >= 0 || c1.fused_se) continue;
            if (c2.d.in_buf != c1.d.out_a) continue;
            c1.block_fused = 1;
            c2.in_block = 1;
        }
        // consecutive fused blocks, each reading the previous one's bf16 operand and fp32 stream, share a launch
        for (size_t oi = 0; oi < n->ops.size(); oi++) {
            if (!n->ops[oi].block_fused || n->ops[oi].in_trunk) continue;
            n->ops[oi].trunk_len = 1;
#ifndef GAZ_NO_TRUNK      // A/B builds only
            size_t cur = oi;
            while (n->ops[oi].trunk_len < gaz_block::MAX_LAYERS) {
                const NetOp &c2 = n->ops[cur + 1];
                const gaz_net_op &o = c2.fused_se ? c2.se : c2.d;
                const size_t nx = cur + (c2.fused_se ? 3 : 2);
                if (nx + 1 >= n->ops.size() || !n->ops[nx].block_fused) break;
                const NetOp &n2 = n->ops[nx + 1];
                const gaz_net_op &o2 = n2.fused_se ? n2.se : n2.d;
                if (n->ops[nx].d.in_buf != o.out_a || o.out_a < 0 || o2.res_buf != o.out_raw || o.out_raw < 0) break;
                n->ops[nx].in_trunk = 1;
                n->ops[oi].trunk_len++;
                cur = nx;
            }
#endif
        }
    }
    // Head convolutions that read the fp32 trunk output (Connect4, TicTacToe) run on headconv_wide_kernel; a second head
    // convolution with the same input, taps and input channels joins the launch as columns 8..15 (N = 16).
    {
        auto boards_per_iter = [&](int want_rows) {   // G boards per CTA iteration: G * P_pad a multiple of 16, about want_rows rows
            int g0 = 1;
            while ((g0 * n->P_pad) % 16 != 0) g0++;
            int G = g0;
            while ((G + g0) * n->P_pad <= want_rows) G += g0;
            return G;
        };
        for (size_t i = 0; i < n->ops.size(); i++) {
            NetOp &o1 = n->ops[i];
            const gaz_net_op &d1 = o1.d;
            if (d1.type != GAZ_OP_HEADCONV || o1.dual_skip || o1.head_wide) continue;
            if (d1.cout > 8 || (d1.ksize != 1 && d1.ksize != 3) || d1.cin % 16 != 0 || d1.cin > 256) continue;
            if (n->bufs[(size_t)d1.in_buf].kind != GAZ_BUF_ROWS_F32) continue;
            if (i + 1 < n->ops.size() && n->ops[i + 1].dense_tc) continue;
            const int G = boards_per_iter(d1.ksize == 3 ? 224 : 256);
            if (gaz_small::head_wide_smem(d1.cin, d1.ksize, n->P_pad, n->Wp, G) > 220 * 1024) continue;
            const gaz_net_op *d2p = nullptr;
            for (size_t j = i + 1; j < n->ops.size(); j++) {
                NetOp &o2 = n->ops[j];
                const gaz_net_op &d2 = o2.d;
                if (d2.type != GAZ_OP_HEADCONV || d2.in_buf != d1.in_buf || d2.cin != d1.cin || d2.cout > 8 || d2.ksize != d1.ksize ||
                    o2.dual_skip || o2.head_wide) continue;
                if (j + 1 < n->ops.size() && n->ops[j + 1].dense_tc) continue;
                o1.dual_partner = (int)j;
                o2.dual_skip = 1;
                d2p = &o2.d;
                break;
            }
            const int taps = d1.ksize * d1.ksize, KS = d1.cin / 16;
            std::vector<gaz_small::Frag> fr((size_t)taps * KS * 2 * 32);
            for (int tp = 0; tp < taps; tp++)
                for (int ks = 0; ks < KS; ks++)
                    for (int nt = 0; nt < 2; nt++) {
                        const gaz_net_op *dd = nt == 0 ? &d1 : d2p;
                        for (int lane = 0; lane < 32; lane++) {
                            auto wfun = [&](int k, int nn) -> float {   // [tap][Cin][Cout] filters of head nt, zero beyond its channels
                                if (!dd || nn >= dd->cout) return 0.0f;
                                return desc->wf[dd->w + ((int64_t)tp * dd->cin + k) * dd->cout + nn];
                            };
                            fr[(((size_t)tp * KS + ks) * 2 + nt) * 32 + lane] = gaz_small::host_frag(lane, wfun, ks * 16, 0);
                        }
                    }
            float hb[16];
            for (int c = 0; c < 16; c++) {
                const gaz_net_op *dd = c < 8 ? &d1 : d2p;
                hb[c] = (dd && (c & 7) < dd->cout) ? desc->wf[dd->bias + (c & 7)] : 0.0f;
            }
            if (alloc((void **)&o1.d_frag, fr.size() * sizeof(gaz_small::Frag)) != 0 || alloc((void **)&o1.d_hbias, sizeof hb) != 0) { gaz_net_destroy(n); return -1; }
            CKN(cudaMemcpy(o1.d_frag, fr.data(), fr.size() * sizeof(gaz_small::Frag), cudaMemcpyHostToDevice));
            CKN(cudaMemcpy(o1.d_hbias, hb, sizeof hb, cudaMemcpyHostToDevice));
            o1.head_wide = 1;
            o1.head_G = G;
        }
        // stems the tcgen05 kernel does not cover: fragments + parameters of stem_mma_kernel (set below once stem_tc is known)
    }
    // A (dual) 3x3 head convolution on the fp32 output of a fused residual block moves to the tensor cores: the block's last
    // epilogue also writes bf16(x) (its free out_a slot, no ReLU) and conv_board_kernel<48> convolves that copy with the bf16
    // filters of both heads, dx-merged (N = 3 x 16).  Same operand precision as every trunk convolution.
#ifndef GAZ_NO_HEAD_TC     // A/B builds only
    for (size_t i = 0; i < n->ops.size(); i++) {
        NetOp &o1 = n->ops[i];
        const gaz_net_op &d1 = o1.d;
        if (d1.type != GAZ_OP_HEADCONV || !o1.head_wide || d1.ksize != 3 || d1.cin != 128 || d1.cout > 8) continue;
        if (gaz_conv::TILE_ROWS % n->P_pad != 0 || 32 % n->Wp != 0 || (n->n_sm & ~1) < 2) continue;
        const gaz_net_op *d2p = o1.dual_partner >= 0 ? &n->ops[(size_t)o1.dual_partner].d : nullptr;
        NetOp *src = nullptr;      // the conv2 op whose (fused SE) epilogue writes the head input
        for (auto &c2 : n->ops) {
            if (c2.d.type != GAZ_OP_CONV_TC || !c2.in_block) continue;
            const gaz_net_op &o = c2.fused_se ? c2.se : c2.d;
            if (o.out_raw == d1.in_buf && o.out_a < 0 && !c2.d_xbf) src = &c2;
        }
        if (!src) continue;
        if (walloc((void **)&src->d_xbf, (size_t)n->rows_alloc * 128 * 2) != 0) { gaz_net_destroy(n); return -1; }
        const size_t ld = (size_t)3 * d1.cin;
        std::vector<uint16_t> wt((size_t)48 * ld, 0);
        auto bf16_bits = [](float f) -> uint16_t { uint32_t u; memcpy(&u, &f, 4); return (uint16_t)((u + 0x7FFFu + ((u >> 16) & 1u)) >> 16); };
        for (int hd = 0; hd < 2; hd++) {
            const gaz_net_op *dd = hd == 0 ? &d1 : d2p;
            if (!dd) continue;
            for (int dy = 0; dy < 3; dy++)
                for (int dx = 0; dx < 3; dx++)
                    for (int k = 0; k < dd->cin; k++)
                        for (int c = 0; c < dd->cout; c++)      // [tap][Cin][Cout] fp32 filters of the head
                            wt[(size_t)(dx * 16 + hd * 8 + c) * ld + (size_t)dy * dd->cin + k] =
                                bf16_bits(desc->wf[dd->w + ((int64_t)(dy * 3 + dx) * dd->cin + k) * dd->cout + c]);
        }
        if (alloc((void **)&o1.d_wt, wt.size() * 2) != 0) { gaz_net_destroy(n); return -1; }
        CKN(cudaMemcpy(o1.d_wt, wt.data(), wt.size() * 2, cudaMemcpyHostToDevice));
        if (make_map(enc, &o1.tmA2, src->d_xbf, 128, (uint64_t)n->rows_alloc, gaz_conv::SLAB_BOX_ROWS) != 0 ||
            make_map(enc, &o1.tmB2, o1.d_wt, (uint64_t)ld, 48, 24) != 0 ||
            make_map_ex(enc, &src->tmOa, src->d_xbf, 128, (uint64_t)n->rows_alloc, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B) != 0) { gaz_net_destroy(n); return -1; }
        memset(&o1.tmOa, 0, sizeof o1.tmOa);
        memset(&o1.tmOb, 0, sizeof o1.tmOb);
        for (int c = 0; c < 640; c++) o1.par[c] = 0.0f;
        for (int c = 0; c < 16; c++) {
            const gaz_net_op *dd = c < 8 ? &d1 : d2p;
            o1.par[c] = (dd && (c & 7) < dd->cout) ? desc->wf[dd->bias + (c & 7)] : 0.0f;
        }
        o1.head_tc = 1;
    }
#endif
    // dense chains: consecutive DENSE ops, each reading the previous one's output, that fit a CTA's shared memory
    for (size_t i = 0; i < n->ops.size(); i++) {
        NetOp &o1 = n->ops[i];
        if (o1.d.type != GAZ_OP_DENSE || o1.dense_tc || o1.chain_skip || o1.chain_len) continue;
        auto fits = [](const gaz_net_op &dd) { return dd.cin <= 512 && dd.cout <= 128; };
        if (!fits(o1.d)) continue;
        int len = 1;
        while (len < 3 && i + (size_t)len < n->ops.size()) {
            const NetOp &nx = n->ops[i + (size_t)len];
            const gaz_net_op &pv = n->ops[i + (size_t)len - 1].d;
            if (nx.d.type != GAZ_OP_DENSE || nx.dense_tc || !fits(nx.d) || (pv.flags & 4) || nx.d.in_buf != pv.out_raw || nx.d.cin != pv.cout) break;
            // the intermediate buffer must have no other reader (the chain never writes it)
            bool other = false;
            for (size_t k = 0; k < n->ops.size(); k++)
                if (k != i + (size_t)len && (n->ops[k].d.in_buf == pv.out_raw || n->ops[k].d.res_buf == pv.out_raw)) other = true;
            if (other || pv.out_raw == n->logits_buf) break;
            len++;
        }
        if (len < 2) continue;
        o1.chain_len = len;
        for (int k = 1; k < len; k++) n->ops[i + (size_t)k].chain_skip = 1;
    }
    // layer 0 of a chain on mma.sync when its shape allows (In a multiple of 16, enough work to matter); a lone fp32 dense layer of
    // that kind (Gomoku's policy_2, 512 -> 225) becomes a one-layer chain
#ifndef GAZ_NO_MLP_MMA     // A/B builds only
    for (auto &o1 : n->ops) {
        const gaz_net_op &d = o1.d;
        if (d.type != GAZ_OP_DENSE || o1.dense_tc || o1.chain_skip || d.cin % 16 != 0 || d.cin < 128 || d.cin > 512) continue;
        if (o1.chain_len == 0) {
            if (d.cout < 64 || d.cout > 256) continue;
            o1.chain_len = 1;
        } else if (d.cout < 64 || d.cout > 128) continue;
        const int KS = d.cin / 16, NT = (((d.cout + 7) / 8) + 7) & ~7;   // n-tiles padded to a multiple of 8 (zero fragments beyond Out)
        std::vector<gaz_small::Frag> fr((size_t)KS * NT * 32);
        for (int ks = 0; ks < KS; ks++)
            for (int nt = 0; nt < NT; nt++)
                for (int lane = 0; lane < 32; lane++) {
                    auto wfun = [&](int k, int nn) -> float { return nn < d.cout ? desc->wf[d.w + (int64_t)k * d.cout + nn] : 0.0f; };   // [In][Out]
                    fr[((size_t)ks * NT + nt) * 32 + lane] = gaz_small::host_frag(lane, wfun, ks * 16, nt * 8);
                }
        if (alloc((void **)&o1.d_frag0, fr.size() * sizeof(gaz_small::Frag)) != 0) { gaz_net_destroy(n); return -1; }
        CKN(cudaMemcpy(o1.d_frag0, fr.data(), fr.size() * sizeof(gaz_small::Frag), cudaMemcpyHostToDevice));
    }
#endif
    // a later chain whose input is complete before this chain's launch (its producer comes earlier in the op list, or is the
    // second head of an earlier dual head convolution) joins the launch
    for (size_t i = 0; i < n->ops.size(); i++) {
        NetOp &o1 = n->ops[i];
        if (o1.d.type != GAZ_OP_DENSE || o1.chain_len == 0 || o1.chain_joined || o1.chain_partner >= 0) continue;
        for (size_t j = i + (size_t)o1.chain_len; j < n->ops.size(); j++) {
            NetOp &o2 = n->ops[j];
            if (o2.d.type != GAZ_OP_DENSE || o2.chain_len == 0 || o2.chain_joined || o2.chain_partner >= 0) continue;
            bool ready = false, clash = false;
            for (size_t k = 0; k < n->ops.size(); k++) {
                const NetOp &pk = n->ops[k];
                if (pk.d.out_raw != o2.d.in_buf) continue;
                size_t exec = k;                       // the op whose launch writes this buffer
                if (pk.dual_skip) { exec = n->ops.size(); for (size_t q = 0; q < k; q++) if (n->ops[q].dual_partner == (int)k) exec = q; }
                if (exec < i) ready = true; else clash = true;
            }
            if (!ready || clash) continue;
            o1.chain_partner = (int)j;
            o2.chain_joined = 1;
            break;
        }
    }
    // stem on the tensor cores: 3x3 on 2 planes -> 256 filters, tile == board, bf16 outputs only
    for (auto &op : n->ops) {
        const gaz_net_op &d = op.d;
        if (d.type != GAZ_OP_STEM) continue;
        if (d.ksize != 3 || d.cin != 2 || d.cout != 256 || n->P_pad != 256 || n->H > 16 || n->W > 16 || d.out_raw >= 0) continue;
        if (d.act != GAZ_ACT_NONE && d.act != GAZ_ACT_RELU) continue;
        if (d.out_a < 0 && d.out_b < 0) continue;
        std::vector<uint16_t> wp((size_t)256 * 64, 0);
        auto bf16_bits = [](float f) -> uint16_t { uint32_t u; memcpy(&u, &f, 4); return (uint16_t)((u + 0x7FFFu + ((u >> 16) & 1u)) >> 16); };
        auto bf16_val = [](uint16_t b) -> float { uint32_t u = (uint32_t)b << 16; float f; memcpy(&f, &u, 4); return f; };
        for (int o = 0; o < 256; o++)
            for (int k = 0; k < 18; k++) {
                const float w = desc->wf[d.w + (int64_t)k * 256 + o];   // [tap][plane][filter]
                const uint16_t hi = bf16_bits(w);
                wp[(size_t)o * 64 + k] = hi;
                wp[(size_t)o * 64 + 18 + k] = bf16_bits(w - bf16_val(hi));
            }
        std::vector<float> par((size_t)4 * 256);
        for (int c = 0; c < 256; c++) {
            const float sc = d.scale_b >= 0 ? desc->wf[d.scale_b + c] : 1.0f, sh = d.shift_b >= 0 ? desc->wf[d.shift_b + c] : 0.0f;
            par[c] = sc;
            par[256 + c] = fmaf(sc, desc->wf[d.bias + c], sh);
            par[512 + c] = d.scale_a >= 0 ? desc->wf[d.scale_a + c] : 1.0f;
            par[768 + c] = d.shift_a >= 0 ? desc->wf[d.shift_a + c] : 0.0f;
        }
        if (alloc((void **)&op.d_stem_w, wp.size() * 2) != 0 || alloc((void **)&op.d_stem_par, par.size() * 4) != 0) { gaz_net_destroy(n); return -1; }
        CKN(cudaMemcpy(op.d_stem_w, wp.data(), wp.size() * 2, cudaMemcpyHostToDevice));
        CKN(cudaMemcpy(op.d_stem_par, par.data(), par.size() * 4, cudaMemcpyHostToDevice));
        memset(&op.tmOa, 0, sizeof op.tmOa);
        memset(&op.tmOb, 0, sizeof op.tmOb);
        bool ok = true;
        for (int k = 0; k < 2 && ok; k++) {
            const int id = k == 0 ? d.out_a : d.out_b;
            if (id < 0) continue;
            const NetBuf &ob = n->bufs[(size_t)id];
            if (ob.kind != GAZ_BUF_ROWS_BF16 || ob.width != 256) { ok = false; break; }
            if (make_map_ex(enc, k == 0 ? &op.tmOa : &op.tmOb, ob.ptr, 256, (uint64_t)n->rows_alloc, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B) != 0) {
                gaz_net_destroy(n);
                return -1;
            }
        }
        op.stem_tc = ok ? 1 : 0;
    }
    // stem followed by the 1x1 projection of the first block's shortcut (C256 -> C128, fp32 out, nothing else reads the stem's
    // raw output): one kernel, the raw stem output never goes to HBM
#ifndef GAZ_NO_STEM_PROJ   // A/B builds only (tools/build_variant.sh)
    for (size_t oi = 0; oi + 1 < n->ops.size(); oi++) {
        NetOp &st = n->ops[oi], &pj = n->ops[oi + 1];
        if (st.d.type != GAZ_OP_STEM || !st.stem_tc || st.d.out_a < 0 || st.d.out_b < 0) continue;
        const gaz_net_op &d = pj.d;
        if (d.type != GAZ_OP_CONV_TC || d.ksize != 1 || d.cin != 256 || d.cout != 128 || d.in_buf != st.d.out_b || d.out_raw < 0 ||
            d.out_a >= 0 || d.out_b >= 0 || d.res_buf >= 0 || d.bias < 0 || pj.fused_se) continue;
        bool other = false;
        for (size_t k = 0; k < n->ops.size(); k++)
            if (k != oi + 1 && (n->ops[k].d.in_buf == st.d.out_b || n->ops[k].d.res_buf == st.d.out_b)) other = true;
        if (other) continue;
        st.stem_proj = 1;
        pj.in_block = 1;
    }
#endif
    // stems with 128 filters on tiles of whole boards (Connect4, TicTacToe): tcgen05 as well (gaz_stem::stem_tile_kernel)
    for (auto &op : n->ops) {
        const gaz_net_op &d = op.d;
        if (d.type != GAZ_OP_STEM || op.stem_tc) continue;
        const bool shape = (d.ksize == 3 && (d.cin == 2 || d.cin == 4)) || (d.ksize == 5 && d.cin == 2);
        if (!shape || d.cout != 128 || gaz_conv::TILE_ROWS % n->P_pad != 0 || d.out_b >= 0 || (d.out_raw < 0 && d.out_a < 0)) continue;
        if (d.act != GAZ_ACT_NONE && d.act != GAZ_ACT_RELU && d.act != GAZ_ACT_GELU) continue;
        const int KK = d.ksize * d.ksize * d.cin;
        std::vector<uint16_t> wp((size_t)128 * 2 * 64, 0);
        auto bf16_bits = [](float f) -> uint16_t { uint32_t u; memcpy(&u, &f, 4); return (uint16_t)((u + 0x7FFFu + ((u >> 16) & 1u)) >> 16); };
        auto bf16_val = [](uint16_t b) -> float { uint32_t u = (uint32_t)b << 16; float f; memcpy(&f, &u, 4); return f; };
        for (int o = 0; o < 128; o++)
            for (int k = 0; k < KK; k++) {
                const float w = desc->wf[d.w + (int64_t)k * 128 + o];   // [tap][plane][filter]
                const uint16_t hi = bf16_bits(w);
                wp[((size_t)o * 2) * 64 + k] = hi;
                wp[((size_t)o * 2 + 1) * 64 + k] = bf16_bits(w - bf16_val(hi));
            }
        std::vector<float> par((size_t)5 * 128);
        for (int c = 0; c < 128; c++) {
            par[c] = desc->wf[d.bias + c];
            par[128 + c] = d.scale_b >= 0 ? desc->wf[d.scale_b + c] : 1.0f;
            par[256 + c] = d.shift_b >= 0 ? desc->wf[d.shift_b + c] : 0.0f;
            par[384 + c] = d.scale_a >= 0 ? desc->wf[d.scale_a + c] : 1.0f;
            par[512 + c] = d.shift_a >= 0 ? desc->wf[d.shift_a + c] : 0.0f;
        }
        if (alloc((void **)&op.d_stem_w, wp.size() * 2) != 0 || alloc((void **)&op.d_stem_par, par.size() * 4) != 0) { gaz_net_destroy(n); return -1; }
        CKN(cudaMemcpy(op.d_stem_w, wp.data(), wp.size() * 2, cudaMemcpyHostToDevice));
        CKN(cudaMemcpy(op.d_stem_par, par.data(), par.size() * 4, cudaMemcpyHostToDevice));
        memset(&op.tmOa, 0, sizeof op.tmOa);
        if (d.out_a >= 0) {
            const NetBuf &ob = n->bufs[(size_t)d.out_a];
            if (ob.kind != GAZ_BUF_ROWS_BF16 || ob.width != 128) continue;
            if (make_map_ex(enc, &op.tmOa, ob.ptr, 128, (uint64_t)n->rows_alloc, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B) != 0) { gaz_net_destroy(n); return -1; }
        }
        if (d.out_raw >= 0 && (n->bufs[(size_t)d.out_raw].kind != GAZ_BUF_ROWS_F32 || n->bufs[(size_t)d.out_raw].width != 128)) continue;
#ifndef GAZ_NO_STEM_TILE   // A/B builds only
        op.stem_tile = 1;
#endif
    }
    for (auto &op : n->ops) {   // every other stem: B fragments (hi | lo) + parameters of gaz_small::stem_mma_kernel
        const gaz_net_op &d = op.d;
        if (d.type != GAZ_OP_STEM || op.stem_tc || op.stem_tile) continue;
        if (d.cout % 8 != 0 || d.cout > 256 || !((d.ksize == 3 && (d.cin == 2 || d.cin == 4)) || (d.ksize == 5 && d.cin == 2))) {
            gaz_net_destroy(n);
            return gaz_fail("stem shape unsupported (k %d cin %d cout %d)", d.ksize, d.cin, d.cout);
        }
        const int KK = d.ksize * d.ksize * d.cin, KS = (KK + 15) / 16, NT = d.cout / 8;
        std::vector<gaz_small::Frag> fr((size_t)KS * NT * 32);
        for (int ks = 0; ks < KS; ks++)
            for (int nt = 0; nt < NT; nt++)
                for (int lane = 0; lane < 32; lane++) {
                    auto wfun = [&](int k, int nn) -> float { return k < KK ? desc->wf[d.w + (int64_t)k * d.cout + nn] : 0.0f; };
                    fr[((size_t)ks * NT + nt) * 32 + lane] = gaz_small::host_frag(lane, wfun, ks * 16, nt * 8);
                }
        std::vector<float> par((size_t)5 * d.cout);
        for (int c = 0; c < d.cout; c++) {
            par[c] = desc->wf[d.bias + c];
            par[(size_t)d.cout + c] = d.scale_b >= 0 ? desc->wf[d.scale_b + c] : 1.0f;
            par[(size_t)2 * d.cout + c] = d.shift_b >= 0 ? desc->wf[d.shift_b + c] : 0.0f;
            par[(size_t)3 * d.cout + c] = d.scale_a >= 0 ? desc->wf[d.scale_a + c] : 1.0f;
            par[(size_t)4 * d.cout + c] = d.shift_a >= 0 ? desc->wf[d.shift_a + c] : 0.0f;
        }
        if (alloc((void **)&op.d_frag, fr.size() * sizeof(gaz_small::Frag)) != 0 || alloc((void **)&op.d_stem_par, par.size() * 4) != 0) { gaz_net_destroy(n); return -1; }
        CKN(cudaMemcpy(op.d_frag, fr.data(), fr.size() * sizeof(gaz_small::Frag), cudaMemcpyHostToDevice));
        CKN(cudaMemcpy(op.d_stem_par, par.data(), par.size() * 4, cudaMemcpyHostToDevice));
        int g0 = 1;
        while ((g0 * n->P_pad) % 16 != 0) g0++;
        int G = g0;
        while ((G + g0) * n->P_pad <= 512) G += g0;    // ~32 m-tiles per iteration: 4 per warp, enough groups to balance the SMs
        op.head_G = G;
    }
#ifndef GAZ_NO_HEAD_STREAMS   // A/B builds only
    {   // separable heads: [head1_begin, head2_begin) ends with POLICY_OUT, [head2_begin, end) reads nothing the first head writes
        int last_block = -1, pout = -1;
        for (size_t i = 0; i < n->ops.size(); i++) {
            const NetOp &o = n->ops[i];
            if (o.block_fused || o.in_block || o.in_trunk || o.skip) last_block = (int)i;
            if (o.d.type == GAZ_OP_POLICY_OUT) pout = (int)i;
        }
        const int h1 = last_block + 1, h2 = pout + 1;
        bool ok = last_block >= 0 && pout > h1 && h2 < (int)n->ops.size();
        for (int i = h2; ok && i < (int)n->ops.size(); i++) {
            const gaz_net_op &d = n->ops[(size_t)i].d;
            for (int j = h1; j < h2; j++) {
                const NetOp &w = n->ops[(size_t)j];
                const int outs[3] = {w.d.out_raw, w.d.out_a, w.d.out_b};
                for (int k = 0; k < 3; k++)
                    if (outs[k] >= 0 && (outs[k] == d.in_buf || outs[k] == d.res_buf || outs[k] == d.out_raw || outs[k] == d.out_a || outs[k] == d.out_b)) ok = false;
                if (w.dual_partner >= i || w.chain_partner >= i) ok = false;   // a launch of the first head that also runs ops of the second
            }
        }
        if (ok) { n->head1_begin = h1; n->head2_begin = h2; }
    }
#endif
    if (share && ws_next != n->ws->ptrs.size()) {
        gaz_net_destroy(n);
        return gaz_fail("shared workspace: %d of its %d activation allocations used", (int)ws_next, (int)share->ws->ptrs.size());
    }
    CKN(cudaDeviceSynchronize());
    *out = n;
    return 0;
}

void gaz_net_destroy(gaz_net *n) {
    if (!n) return;
    cudaStreamSynchronize(n->stream);
    cudaStreamSynchronize(n->stream2);
    // bufs, d_act, d_xbf and the host-path staging belong to the workspace
    for (auto &op : n->ops) { if (op.d_se_b1) cudaFree(op.d_se_b1); if (op.d_wt) cudaFree(op.d_wt); if (op.d_stem_w) cudaFree(op.d_stem_w); if (op.d_stem_par) cudaFree(op.d_stem_par); if (op.d_frag) cudaFree(op.d_frag); if (op.d_hbias) cudaFree(op.d_hbias); if (op.d_frag0) cudaFree(op.d_frag0); }
    cudaFree(n->wf); cudaFree(n->wh); cudaFree(n->d_count); cudaFree(n->d_chunk_count);
    if (n->d_chunk_count16) cudaFree(n->d_chunk_count16);
    if (n->ws && --n->ws->refs == 0) {
        for (void *p : n->ws->ptrs) cudaFree(p);
        delete n->ws;
    }
    for (auto e : n->ev) cudaEventDestroy(e);
    cudaStreamDestroy(n->stream);
    cudaStreamDestroy(n->stream2);
    cudaEventDestroy(n->ev_fork); cudaEventDestroy(n->ev_join);
    delete n->trunk_args;
    delete n;
}

int gaz_net_forward_host(gaz_net *n, const int8_t *states, int cnt, float *policy, float *value, float *logits) {
    if (!n || !states) return gaz_fail("null argument");
    if (cnt < 0 || cnt > n->max_batch) return gaz_fail("batch %d exceeds max_batch %d", cnt, n->max_batch);
    if (cnt == 0) return 0;
    const size_t ss = (size_t)n->H * n->W * n->Cin;
    CKN(cudaMemcpyAsync(n->d_states, states, (size_t)cnt * ss, cudaMemcpyHostToDevice, n->stream));
    set_count_kernel<<<1, 1, 0, n->stream>>>(n->d_count, cnt);
    if (net_forward(n, n->d_states, n->d_count, n->d_policy, n->d_value, n->stream) != 0) return -1;
    if (policy) CKN(cudaMemcpyAsync(policy, n->d_policy, (size_t)cnt * n->P * 4, cudaMemcpyDeviceToHost, n->stream));
    if (value) CKN(cudaMemcpyAsync(value, n->d_value, (size_t)cnt * 4, cudaMemcpyDeviceToHost, n->stream));
    if (logits && n->logits_buf >= 0)
        CKN(cudaMemcpyAsync(logits, n->bufs[(size_t)n->logits_buf].ptr, (size_t)cnt * n->P * 4, cudaMemcpyDeviceToHost, n->stream));
    CKN(cudaStreamSynchronize(n->stream));
    return cnt;
}

static void drop_round_graph(gaz_engine *e) {
    if (e->round_graph) { cudaGraphExecDestroy((cudaGraphExec_t)e->round_graph); e->round_graph = nullptr; }
    e->round_graph_warm = 0;
    e->attach_epoch++;
}

// Packed lists for the first K networks, each of at least `cap` rows (allocated on first use, grown when a symmetry mode
// needs more rows; the round graph bakes in the pointers, so a regrowth drops it).
static int route_reserve(gaz_engine *e, int K, size_t cap) {
    const size_t NT = (size_t)e->v.n_trees, S = (size_t)e->v.ncell * e->v.C, P = (size_t)e->v.P;
    if (!e->route) {
        gaz_route r;
        memset(&r, 0, sizeof r);
        r.cap = NT;
        if (gaz_internal_alloc(e, (void **)&r.count, GAZ_MAX_NETS * sizeof(int32_t)) != 0 ||
            gaz_internal_alloc(e, (void **)&r.rows, GAZ_MAX_NETS * sizeof(int32_t)) != 0 ||
            gaz_internal_alloc(e, (void **)&e->d_tree_net, NT) != 0)   // zero: every tree on network 0
            return -1;
        e->route = new gaz_route(r);
    }
    gaz_route &r = *e->route;
    if (cap > r.cap) {   // new lists first: a failed allocation leaves the old ones in place
        int8_t *st[GAZ_MAX_NETS] = {};
        float *po[GAZ_MAX_NETS] = {}, *va[GAZ_MAX_NETS] = {};
        auto undo = [&]() {
            for (int k = 0; k < r.n_alloc; k++) {
                if (st[k]) gaz_internal_free(e, st[k], cap * S);
                if (po[k]) gaz_internal_free(e, po[k], cap * P * sizeof(float));
                if (va[k]) gaz_internal_free(e, va[k], cap * sizeof(float));
            }
            return -1;
        };
        for (int k = 0; k < r.n_alloc; k++)
            if (gaz_internal_alloc(e, (void **)&st[k], cap * S) != 0 || gaz_internal_alloc(e, (void **)&po[k], cap * P * sizeof(float)) != 0 ||
                gaz_internal_alloc(e, (void **)&va[k], cap * sizeof(float)) != 0)
                return undo();
        CKN(cudaStreamSynchronize(e->stream));
        drop_round_graph(e);
        for (int k = 0; k < r.n_alloc; k++) {
            gaz_internal_free(e, r.state[k], r.cap * S);
            gaz_internal_free(e, r.pol[k], r.cap * P * sizeof(float));
            gaz_internal_free(e, r.val[k], r.cap * sizeof(float));
            r.state[k] = st[k]; r.pol[k] = po[k]; r.val[k] = va[k];
        }
        r.cap = cap;
    }
    for (int k = r.n_alloc; k < K; k++) {   // packed lists of the networks not seen before
        if (gaz_internal_alloc(e, (void **)&r.idx[k], NT * sizeof(int32_t)) != 0 ||
            gaz_internal_alloc(e, (void **)&r.sym[k], NT) != 0 ||
            gaz_internal_alloc(e, (void **)&r.state[k], r.cap * S) != 0 ||
            gaz_internal_alloc(e, (void **)&r.pol[k], r.cap * P * sizeof(float)) != 0 ||
            gaz_internal_alloc(e, (void **)&r.val[k], r.cap * sizeof(float)) != 0)
            return -1;
        r.n_alloc = k + 1;
    }
    return 0;
}

static bool sym_on(const gaz_engine *e) { return e->sym && e->sym->mode != GAZ_SYM_NONE; }
static int sym_rows_per_leaf(const gaz_engine *e) { return sym_on(e) && e->sym->mode == GAZ_SYM_ENSEMBLE ? e->sym->n : 1; }

int gaz_attach_net(gaz_engine *e, gaz_net *n) {
    if (!e) return gaz_fail("null engine");
    if (n) {
        if (n->game != e->cfg.game) return gaz_fail("network game %d != engine game %d", n->game, e->cfg.game);
    }
    if (e->route && e->tree_net_max > 0) {   // the routed symmetric path reads the table: back to network 0
        CKN(cudaMemsetAsync(e->d_tree_net, 0, (size_t)e->v.n_trees, e->stream));
        e->tree_net_max = 0;
    }
    for (int k = 0; k < GAZ_MAX_NETS; k++) e->nets[k] = k == 0 ? n : nullptr;
    e->n_nets = n ? 1 : 0;
    drop_round_graph(e);
    return 0;
}

int gaz_attach_nets(gaz_engine *e, gaz_net *const *nets, int n_nets) {
    if (!e || !nets) return gaz_fail("null argument");
    if (n_nets < 1 || n_nets > GAZ_MAX_NETS) return gaz_fail("gaz_attach_nets: %d networks (1 to %d)", n_nets, GAZ_MAX_NETS);
    for (int k = 0; k < n_nets; k++)
        if (!nets[k]) return gaz_fail("gaz_attach_nets: network %d is null", k);
    if (n_nets == 1) return gaz_attach_net(e, nets[0]);
    for (int k = 1; k < n_nets; k++)
        if (nets[k]->game != nets[0]->game)
            return gaz_fail("networks 0 and %d are for different games (%d, %d)", k, nets[0]->game, nets[k]->game);
    if (nets[0]->game != e->cfg.game) return gaz_fail("network game %d != engine game %d", nets[0]->game, e->cfg.game);
    for (int k = 0; k < n_nets; k++)
        if (nets[k]->P != e->v.P)
            return gaz_fail("network %d has policy size %d (network 0: %d, engine: %d)", k, nets[k]->P, nets[0]->P, e->v.P);
    if (e->cache) return gaz_fail("%d networks cannot share the evaluation cache: its key does not include the network", n_nets);
    if (route_reserve(e, n_nets, (size_t)e->v.n_trees * sym_rows_per_leaf(e)) != 0) return -1;
    const size_t NT = (size_t)e->v.n_trees;
    if (e->tree_net_max >= n_nets) {   // the table names a network that is no longer attached: back to network 0
        CKN(cudaMemsetAsync(e->d_tree_net, 0, NT, e->stream));
        e->tree_net_max = 0;
    }
    for (int k = 0; k < GAZ_MAX_NETS; k++) e->nets[k] = k < n_nets ? nets[k] : nullptr;
    e->n_nets = n_nets;
    drop_round_graph(e);
    return 0;
}

int gaz_set_tree_nets(gaz_engine *e, const uint8_t *tree_net) {
    if (!e || !tree_net) return gaz_fail("null argument");
    const int lim = e->n_nets > 1 ? e->n_nets : 1;
    int mx = 0;
    for (int t = 0; t < e->v.n_trees; t++) {
        if (tree_net[t] >= lim) return gaz_fail("tree_net[%d] = %d, but %d network(s) attached", t, (int)tree_net[t], e->n_nets);
        mx = tree_net[t] > mx ? tree_net[t] : mx;
    }
    if (!e->d_tree_net) return 0;   // no second network was ever attached: every tree is on network 0 already
    CKN(cudaMemcpyAsync(e->d_tree_net, tree_net, (size_t)e->v.n_trees, cudaMemcpyHostToDevice, e->stream));
    e->tree_net_max = mx;
    return 0;
}

int gaz_set_eval_symmetry(gaz_engine *e, int mode, int n_sym, const int32_t *perm_state, const int32_t *perm_policy,
                          uint64_t seed) {
    if (!e) return gaz_fail("null engine");
    if (mode != GAZ_SYM_NONE && mode != GAZ_SYM_RANDOM && mode != GAZ_SYM_ENSEMBLE)
        return gaz_fail("unknown symmetry mode %d (GAZ_SYM_NONE 0, GAZ_SYM_RANDOM 1, GAZ_SYM_ENSEMBLE 2)", mode);
    if (mode == GAZ_SYM_NONE) {
        if (sym_on(e)) { e->sym->mode = GAZ_SYM_NONE; drop_round_graph(e); }
        return 0;
    }
    if (n_sym < 1 || n_sym > GAZ_MAX_SYM) return gaz_fail("n_sym = %d (1 to %d symmetries)", n_sym, GAZ_MAX_SYM);
    if (!perm_state || !perm_policy) return gaz_fail("null symmetry table");
    if (e->cache) return gaz_fail("symmetric evaluation cannot be used with the evaluation cache");
    const int S = e->v.ncell * e->v.C, P = e->v.P;
    std::vector<int16_t> ps((size_t)n_sym * S), pp((size_t)n_sym * P);
    for (int t = 0; t < 2; t++) {
        const int len = t == 0 ? S : P;
        const int32_t *tab = t == 0 ? perm_state : perm_policy;
        std::vector<char> seen((size_t)len);
        for (int g = 0; g < n_sym; g++) {
            std::fill(seen.begin(), seen.end(), 0);
            for (int j = 0; j < len; j++) {
                const int32_t x = tab[(size_t)g * len + j];
                if (x < 0 || x >= len || seen[(size_t)x])
                    return gaz_fail("%s row %d is not a permutation of 0..%d (entry %d = %d)", t == 0 ? "perm_state" : "perm_policy",
                                    g, len - 1, j, (int)x);
                seen[(size_t)x] = 1;
                (t == 0 ? ps : pp)[(size_t)g * len + j] = (int16_t)x;
            }
        }
    }
    if (!e->sym) {
        gaz_sym s;
        memset(&s, 0, sizeof s);
        if (gaz_internal_alloc(e, (void **)&s.perm_state, (size_t)GAZ_MAX_SYM * S * sizeof(int16_t)) != 0 ||
            gaz_internal_alloc(e, (void **)&s.perm_policy, (size_t)GAZ_MAX_SYM * P * sizeof(int16_t)) != 0)
            return -1;
        e->sym = new gaz_sym(s);
    }
    const int K = e->n_nets > 1 ? e->n_nets : 1;
    if (route_reserve(e, K, (size_t)e->v.n_trees * (mode == GAZ_SYM_ENSEMBLE ? n_sym : 1)) != 0) return -1;
    if (e->tree_net_max >= K) {   // the table names a network that is no longer attached: back to network 0
        CKN(cudaMemsetAsync(e->d_tree_net, 0, (size_t)e->v.n_trees, e->stream));
        e->tree_net_max = 0;
    }
    // the tables are read from device memory: a captured round graph stays valid when only they change
    CKN(cudaMemcpyAsync(e->sym->perm_state, ps.data(), ps.size() * sizeof(int16_t), cudaMemcpyHostToDevice, e->stream));
    CKN(cudaMemcpyAsync(e->sym->perm_policy, pp.data(), pp.size() * sizeof(int16_t), cudaMemcpyHostToDevice, e->stream));
    CKN(cudaStreamSynchronize(e->stream));
    gaz_sym &s = *e->sym;
    if (s.mode != mode || s.n != n_sym || s.seed != seed) drop_round_graph(e);
    s.mode = mode; s.n = n_sym; s.seed = seed;
    return 0;
}

// forward chunks of network n over a packed request list of at most rows_per_leaf x leaf_bound rows (the count itself is
// on the device)
static int forward_chunks(gaz_engine *e, gaz_net *n, int rows_per_leaf, const int32_t *total, const int8_t *states, float *pol,
                          float *val) {
    const gaz::View &v = e->v;
    const int bound = (e->leaf_bound > 0 ? e->leaf_bound : v.n_trees) * rows_per_leaf;
    const int chunks = (bound + n->max_batch - 1) / n->max_batch;
    if (chunks > n->chunk_cap) return gaz_fail("a bound of %d rows needs more than %d chunks of %d", bound, n->chunk_cap, n->max_batch);
    const size_t ss = (size_t)v.ncell * v.C;
    for (int ck = 0; ck < chunks; ck++) {
        const int off = ck * n->max_batch;
        chunk_count_kernel<<<1, 1, 0, e->stream>>>(total, off, n->max_batch, n->d_chunk_count + ck);
        if (net_forward(n, states + (size_t)off * ss, n->d_chunk_count + ck, pol + (size_t)off * v.P, val + off, e->stream) != 0) return -1;
    }
    return 0;
}

// Serves the engine's outstanding leaf requests; the request list is cut into chunks of max_batch
// leaves (the host-side bound e->leaf_bound says how many chunks can be non-empty).
static int engine_forward(gaz_engine *e) {
    const gaz::View &v = e->v;
    if (sym_on(e)) {
        // route (K = 1 too) -> pack (leaf, g) rows -> each network's chunks over rows_per_leaf x the leaf bound -> map back
        const gaz_route &r = *e->route;
        const gaz_sym &s = *e->sym;
        const int K = e->n_nets, S = v.ncell * v.C, per = sym_rows_per_leaf(e);
        const SymArgs pack{s.perm_state, s.n, per > 1, s.seed, v.tree_keys, 1.0f / (float)s.n};
        const SymArgs back{s.perm_policy, s.n, per > 1, s.seed, v.tree_keys, 1.0f / (float)s.n};
        auto blocks = [](size_t warps) { const size_t b = (warps + 7) / 8; return (unsigned)(b < 148 * 8 ? b : 148 * 8); };
        route_leaves_kernel<<<1, 1024, 0, e->stream>>>(v.leaves, v.leaf_count, e->d_tree_net, K, r);
        sym_states_kernel<<<blocks((size_t)v.n_trees * per), 256, (size_t)s.n * S * sizeof(int16_t), e->stream>>>(
            v.leaves, v.leaf_state, S, K, r, pack);
        CKN(cudaGetLastError());
        for (int k = 0; k < K; k++)
            if (forward_chunks(e, e->nets[k], per, r.rows + k, r.state[k], r.pol[k], r.val[k]) != 0) return -1;
        sym_scatter_kernel<<<blocks((size_t)v.n_trees), 256, (size_t)s.n * v.P * sizeof(int16_t), e->stream>>>(
            v.P, K, r, back, v.policy, v.value);
        CKN(cudaGetLastError());
        return 0;
    }
    if (e->n_nets > 1) {
        // route -> each network's chunks in turn -> scatter.  Any packed list can hold every leaf, so each network gets the
        // chunks of the whole bound and a changed tree_net needs no new round graph.
        const gaz_route &r = *e->route;
        const int K = e->n_nets;
        const unsigned rows = (unsigned)(((size_t)v.n_trees * 32 + 127) / 128);
        route_leaves_kernel<<<1, 1024, 0, e->stream>>>(v.leaves, v.leaf_count, e->d_tree_net, K, r);
        route_states_kernel<<<rows, 128, 0, e->stream>>>(v.leaf_state, v.ncell * v.C, K, r);
        CKN(cudaGetLastError());
        for (int k = 0; k < K; k++)
            if (forward_chunks(e, e->nets[k], 1, r.count + k, r.state[k], r.pol[k], r.val[k]) != 0) return -1;
        scatter_evals_kernel<<<rows, 128, 0, e->stream>>>(v.P, K, r, v.policy, v.value);
        CKN(cudaGetLastError());
        return 0;
    }
    // with the evaluation cache on, the network sees the packed misses of the look-up pass instead of the leaf list
    gaz_eval_cache *c = e->cache;
    if (c && gaz_internal_cache_lookup(e) != 0) return -1;
    const int32_t *total = c ? c->miss_count : v.leaf_count;
    const int8_t *states = c ? c->packed_state : v.leaf_state;
    float *pol = c ? c->packed_pol : v.policy, *val = c ? c->packed_val : v.value;
    if (forward_chunks(e, e->nets[0], 1, total, states, pol, val) != 0) return -1;
    if (c && gaz_internal_cache_fill(e) != 0) return -1;
    return 0;
}

// Every network has 16 per-chunk counters, as many forward chunks as one evaluation of the leaf list takes; ENSEMBLE
// evaluation serves n_sym rows per leaf and can take up to MAX_CHUNKS.  The larger buffer is allocated here, outside any
// graph capture, on the first ENSEMBLE evaluation; the 16-entry one stays allocated with the network, since a round graph
// captured before (by this or another engine) still reads it.
static int reserve_chunk_counts(gaz_engine *e) {
    if (sym_rows_per_leaf(e) == 1) return 0;
    for (int k = 0; k < e->n_nets; k++) {
        gaz_net *n = e->nets[k];
        if (n->chunk_cap >= MAX_CHUNKS) continue;
        int32_t *p = nullptr;
        CKN(cudaMalloc((void **)&p, MAX_CHUNKS * 4));
        CKN(cudaMemset(p, 0, MAX_CHUNKS * 4));
        n->bytes += MAX_CHUNKS * 4;
        n->d_chunk_count16 = n->d_chunk_count;
        n->d_chunk_count = p;
        n->chunk_cap = MAX_CHUNKS;
        drop_round_graph(e);
    }
    return 0;
}

int gaz_eval_net(gaz_engine *e) {
    if (!e || !e->n_nets) return gaz_fail("no network attached");
    if (reserve_chunk_counts(e) != 0) return -1;
    return engine_forward(e);
}

static int one_round_eager(gaz_engine *e) {
    if (gaz_internal_launch_select(e) != 0) return -1;
    if (engine_forward(e) != 0) return -1;
    return gaz_internal_launch_expand(e);
}

// n_rounds x (select -> network -> expand).  One round is ~30-45 kernel launches; for small networks (TicTacToe: 0.2 ms of
// GPU work per round) the launch path is the bottleneck, so the round is captured once into a CUDA graph and replayed.
// Every kernel reads its leaf count from device memory, so the graph does not depend on the data; it is rebuilt when
// the number of forward chunks or the attached network set changes.  Disabled while conv launches are being event-timed.
static int run_rounds(gaz_engine *e, int n_rounds) {
    if (reserve_chunk_counts(e) != 0) return -1;
    bool profiling = false;
    uint64_t chunks = 0;   // forward chunks of every attached network, 8 bits each (at most MAX_CHUNKS, 8 networks)
    const int bound = (e->leaf_bound > 0 ? e->leaf_bound : e->v.n_trees) * sym_rows_per_leaf(e);
    for (int k = 0; k < e->n_nets; k++) {
        profiling = profiling || e->nets[k]->profile;
        chunks |= (uint64_t)((bound + e->nets[k]->max_batch - 1) / e->nets[k]->max_batch) << (8 * k);
    }
    const bool use_graph = !profiling;   // per-launch event timers need eager launches
    for (int r = 0; r < n_rounds; r++) {
        if (!use_graph) { if (one_round_eager(e) != 0) return -1; continue; }
        if (!e->round_graph || e->round_graph_chunks != chunks || e->round_graph_attach != e->attach_epoch ||
            e->round_graph_epoch != e->view_epoch) {
            if (e->round_graph_warm < 1) { // first round eagerly: one-time function attributes are set outside a capture
                if (one_round_eager(e) != 0) return -1;
                e->round_graph_warm = 1;
                continue;
            }
            if (e->round_graph) { cudaGraphExecDestroy((cudaGraphExec_t)e->round_graph); e->round_graph = nullptr; }
            cudaGraph_t g = nullptr;
            CKN(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
            const int rc = one_round_eager(e);
            cudaError_t ce = cudaStreamEndCapture(e->stream, &g);
            if (rc != 0 || ce != cudaSuccess || !g) return gaz_fail("CUDA graph capture of a search round failed (%s)", cudaGetErrorString(ce));
            cudaGraphExec_t ex = nullptr;
            ce = cudaGraphInstantiate(&ex, g, 0);
            cudaGraphDestroy(g);
            if (ce != cudaSuccess) return gaz_fail("cudaGraphInstantiate: %s", cudaGetErrorString(ce));
            e->round_graph = (void *)ex;
            e->round_graph_chunks = chunks;
            e->round_graph_attach = e->attach_epoch;
            e->round_graph_epoch = e->view_epoch;
        }
        CKN(cudaGraphLaunch((cudaGraphExec_t)e->round_graph, e->stream));
    }
    return 0;
}

int gaz_rounds_net(gaz_engine *e, int n_rounds) {
    if (!e || !e->n_nets) return gaz_fail("no network attached");
    if (run_rounds(e, n_rounds) != 0) return -1;
    CKN(cudaStreamSynchronize(e->stream));
    return 0;
}

// same without the trailing synchronise (bench: events bracket many calls)
int gaz_rounds_net_async(gaz_engine *e, int n_rounds) {
    if (!e || !e->n_nets) return gaz_fail("no network attached");
    return run_rounds(e, n_rounds);
}

int64_t gaz_net_bytes(gaz_net *n) { return n ? n->bytes : 0; }

int gaz_net_launches_per_forward(gaz_net *n) { // kernels actually launched: ops folded into another op's kernel do not count
    if (!n) return 0;
    int k = 0;
    for (auto &op : n->ops) {
        if (op.skip || op.in_block || op.in_trunk || op.dual_skip || op.chain_skip || op.chain_joined) continue;
        k += 1;
    }
    return k;
}

int gaz_net_op_blocks(gaz_net *n, int op) { // residual blocks run by the launch of op `op` (0: the op launches no block kernel)
    if (!n || op < 0 || (size_t)op >= n->ops.size()) return 0;
    return n->ops[(size_t)op].in_trunk ? 0 : n->ops[(size_t)op].trunk_len;
}

/* profile = number of conv launches to keep events for (0 disables).  While enabled every tcgen05 conv
 * launch is bracketed by CUDA events on the launching stream. */
int gaz_net_profile(gaz_net *n, int max_launches) {
    if (!n) return gaz_fail("null net");
    n->profile = max_launches > 0;
    n->ev_used = 0;
    n->ev_op.clear();
    while ((int)n->ev.size() < 2 * max_launches) {
        cudaEvent_t ev;
        CKN(cudaEventCreate(&ev));
        n->ev.push_back(ev);
    }
    return 0;
}

/* Sum / count of the bracketed conv launches since gaz_net_profile(); per_op_ms (n_ops floats, optional)
 * receives the per-op totals.  Call after synchronising the stream. */
int gaz_net_profile_read(gaz_net *n, float *total_ms, int *n_launches, float *per_op_ms) {
    if (!n) return gaz_fail("null net");
    float tot = 0.0f;
    int cnt = 0;
    if (per_op_ms) for (size_t i = 0; i < n->ops.size(); i++) per_op_ms[i] = 0.0f;
    for (size_t i = 0; i + 1 < n->ev_used; i += 2) {
        float ms = 0.0f;
        CKN(cudaEventElapsedTime(&ms, n->ev[i], n->ev[i + 1]));
        tot += ms;
        if (per_op_ms && i / 2 < n->ev_op.size()) per_op_ms[n->ev_op[i / 2]] += ms;
        cnt++;
    }
    if (total_ms) *total_ms = tot;
    if (n_launches) *n_launches = cnt;
    return cnt;
}

int gaz_net_time_forward(gaz_net *n, int cnt, int iters, float *ms_out) {
    if (!n || !ms_out) return gaz_fail("null argument");
    if (cnt <= 0 || cnt > n->max_batch) return gaz_fail("bad batch %d", cnt);
    set_count_kernel<<<1, 1, 0, n->stream>>>(n->d_count, cnt);
    for (int i = 0; i < 3; i++)
        if (net_forward(n, n->d_states, n->d_count, n->d_policy, n->d_value, n->stream) != 0) return -1;
    cudaEvent_t e0, e1;
    CKN(cudaEventCreate(&e0));
    CKN(cudaEventCreate(&e1));
    CKN(cudaStreamSynchronize(n->stream));
    CKN(cudaEventRecord(e0, n->stream));
    for (int i = 0; i < iters; i++)
        if (net_forward(n, n->d_states, n->d_count, n->d_policy, n->d_value, n->stream) != 0) return -1;
    CKN(cudaEventRecord(e1, n->stream));
    CKN(cudaStreamSynchronize(n->stream));
    float ms = 0.0f;
    CKN(cudaEventElapsedTime(&ms, e0, e1));
    ms_out[0] = ms / (float)iters;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return 0;
}

} // extern "C"
