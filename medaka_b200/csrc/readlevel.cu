// Read-level consensus network: LatentSpaceLSTM.forward (medaka/architectures/latent_space_lstm.py:154-207) with
// ReadLevelConv (read_level_modules.py:45-78) and MeanPooler (:81-100), fp32 on the CUDA cores - the first correct
// version of SURVEY.md row f4's network half (the feature tensor comes from mdk_read_matrix, pileup.cu).
//
//   x int8 [B][P][D][F]  (base, quality, strand, mapQ [, dwell])                      latent_space_lstm.py:163-183
//   e = base_embedder[base] + strand_embedder[strand + 1]  (6) ++ q / 25 - 1 (++ dwell)          :168-183
//   y1 = BN1(ReLU(Conv1d k=1 (7|8 -> C)))          per read, along positions                       read_level_modules.py:31-40
//   y2 = BN2(ReLU(Conv1d k=17, zero padding 8 (C -> C)))
//   z  = mean over the non-empty reads of Linear(C -> H)(y2)                                        :192-197, MeanPooler
//   two bidirectional LSTM layers (H), Linear(2H -> 5), softmax                                    :198-205
// Sizes: C = cnn_size = H = lstm_size = 128 (the class defaults); other sizes are refused.  BatchNorm runs in inference
// mode (running statistics), in torch's operation order ((x - mean) * invstd * weight + bias).
//
// Kernels:
//   rl_mask_kernel        which (window, read) rows are non-empty (x.sum((1, -1)) != 0, :163-165)
//   rl_embed_conv1_kernel embedding lookups + the k = 1 convolution + ReLU + BN1 -> y1 [B][D][P][C]  (non-empty rows only)
//   rl_conv17_pool_kernel the k = 17 convolution as an implicit GEMM (64 positions x 128 channels per CTA, K = 17 x 128,
//                         8 x 4 register tiles, weights streamed through shared memory), ReLU + BN2 and the masked SUM
//                         over a group of reads, all in one pass: y2 never exists in memory
//   rl_pool_linear_kernel sum of the read groups / number of reads, then Linear(C -> H).  (The reference applies the
//                         Linear before the mean; the mean of an affine map is the affine map of the mean.)
//   rl_gemm_kernel        LSTM input projections  gi = X W_ih^T + b_ih + b_hh   (both directions in one launch)
//   rl_lstm_kernel        the LSTM recurrence: one CTA = 4 windows of one direction, 256 threads (gate pair, unit j);
//                         W_hh^T of gates i, f, g resident in shared memory (192 KiB), gate o's rows in registers (128
//                         per thread of the second half); c and h stay on chip for all P steps
//   head_kernel (misc.cu) Linear(2H -> 5) + softmax, shared with the counts models
// All of it is CUDA-core fp32: parity first (tests/test_read_level.py against the reference's own class); the convolution
// is 99 % of the FLOPs (557 kFLOP per read and position) and belongs on tcgen05 next.
#include <cstdlib>
#include <string>
#include <unordered_map>
#include <vector>

#include "common.cuh"
#include "ptx.cuh"

namespace mdk {

constexpr int RL_C = 128;        // cnn_size
constexpr int RL_H = 128;        // lstm_size
constexpr int RL_EMB = 6;        // bases_embedding_size
constexpr int RL_TAPS = 17;
constexpr int RL_PAD = 8;
constexpr int RL_G4 = 4 * RL_H;

__device__ __forceinline__ float rl_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

// ---------------------------------------------------------------------------------------------- mask
__global__ void __launch_bounds__(256) rl_mask_kernel(const int8_t *__restrict__ x, int64_t P, int D, int F,
                                                      uint8_t *__restrict__ mask) {
    // one block per (b, d): sum over positions and features != 0  (int sum like torch's int64 reduction of int8 input)
    const int64_t b = blockIdx.x / D;
    const int d = (int)(blockIdx.x % D);
    long long s = 0;
    for (int64_t i = threadIdx.x; i < P * F; i += blockDim.x) {
        const int64_t p = i / F;
        const int f = (int)(i % F);
        s += x[((b * P + p) * D + d) * F + f];
    }
    __shared__ long long red[256];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) mask[blockIdx.x] = red[0] != 0;
}

// ---------------------------------------------------------------------------------------------- embedding + conv k=1
struct RlConv1 {
    const float *emb_base;      // [6][6]
    const float *emb_strand;    // [3][6]
    const float *w;             // [C][in]   in = 7 (+1 dwell)
    const float *b;             // [C]
    const float *bn_mean, *bn_invstd, *bn_w, *bn_b;   // [C]
};

__global__ void __launch_bounds__(RL_C) rl_embed_conv1_kernel(const int8_t *__restrict__ x, const uint8_t *__restrict__ mask,
                                                              RlConv1 a, int64_t P, int D, int F, int use_dwells,
                                                              float *__restrict__ y1) {
    // grid: (B * D, position chunks of 32, at most 65 535 of them: a CTA strides over the rest); thread = output channel.
    // B * D goes in x: 100 reads per window put it past y's limit of 65 535 at 656 windows per call
    const int64_t bd = blockIdx.x;
    if (!mask[bd]) return;
    const int64_t b = bd / D;
    const int d = (int)(bd % D);
    const int c = threadIdx.x;
    const int nin = RL_EMB + 1 + (use_dwells ? 1 : 0);
    float w[RL_EMB + 2];
    for (int i = 0; i < nin; ++i) w[i] = a.w[c * nin + i];
    const float bias = a.b[c], mean = a.bn_mean[c], invstd = a.bn_invstd[c], bw = a.bn_w[c], bb = a.bn_b[c];
    __shared__ float in[32][RL_EMB + 2];
    for (int64_t p0 = (int64_t)blockIdx.y * 32; p0 < P; p0 += (int64_t)gridDim.y * 32) {
        __syncthreads();                                       // the previous chunk's rows are consumed
        if (threadIdx.x < 32) {
            const int64_t p = p0 + threadIdx.x;
            if (p < P) {
                const int8_t *v = x + ((b * P + p) * D + d) * F;
                const int base = min(max((int)v[0], 0), 5), strand = min(max((int)v[2] + 1, 0), 2);
                for (int i = 0; i < RL_EMB; ++i) in[threadIdx.x][i] = a.emb_base[base * RL_EMB + i] + a.emb_strand[strand * RL_EMB + i];
                in[threadIdx.x][RL_EMB] = (float)v[1] / 25.0f - 1.0f;
                if (use_dwells) in[threadIdx.x][RL_EMB + 1] = (float)v[4];
            }
        }
        __syncthreads();
        for (int i = 0; i < 32; ++i) {
            const int64_t p = p0 + i;
            if (p >= P) break;
            float acc = bias;
            for (int k = 0; k < nin; ++k) acc = fmaf(w[k], in[i][k], acc);
            acc = fmaxf(acc, 0.f);
            y1[(bd * P + p) * RL_C + c] = (acc - mean) * invstd * bw + bb;
        }
    }
}

// ---------------------------------------------------------------------------------------------- conv k=17 + pooling
struct RlConv17 {
    const float *w_t;           // [17][C in][C out]  (transposed from torch's [out][in][tap])
    const float *b;             // [C]
    const float *bn_mean, *bn_invstd, *bn_w, *bn_b;
};
constexpr int RL_PT = 64;                        // positions per CTA
constexpr int RL_ROWS = RL_PT + 2 * RL_PAD;      // 80 staged input rows
constexpr int RL_YS = RL_C + 4;                  // padded row stride of the staged input
constexpr int RL_KC = 32;                        // input channels per weight chunk
constexpr int RL_CONV_SMEM = (RL_ROWS * RL_YS + RL_KC * RL_C) * 4;

__global__ void __launch_bounds__(256) rl_conv17_pool_kernel(const float *__restrict__ y1, const uint8_t *__restrict__ mask,
                                                             RlConv17 a, int64_t P, int D, int dgroup,
                                                             float *__restrict__ partial) {
    // grid: (position tiles, read groups, B).  partial [B][n_groups][P][C]
    extern __shared__ __align__(16) float smem_rl[];
    float *ys = smem_rl;                      // [80][132]
    float *ws = smem_rl + RL_ROWS * RL_YS;    // [32][128]
    const int tid = threadIdx.x;
    const int tx = tid % 16, ty = tid / 16;   // 16 channel groups of 8, 16 position groups of 4
    const int64_t b = blockIdx.z;
    const int g = blockIdx.y;
    const int64_t p0 = (int64_t)blockIdx.x * RL_PT;
    float bias[8], mean[8], invstd[8], bw[8], bb[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int c = tx * 8 + j;
        bias[j] = a.b[c]; mean[j] = a.bn_mean[c]; invstd[j] = a.bn_invstd[c]; bw[j] = a.bn_w[c]; bb[j] = a.bn_b[c];
    }
    float pooled[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) pooled[i][j] = 0.f;
    const int d0 = g * dgroup, d1 = min(D, d0 + dgroup);
    for (int d = d0; d < d1; ++d) {
        const int64_t bd = b * D + d;
        if (!mask[bd]) continue;                                   // (uniform over the CTA)
        __syncthreads();
        // stage rows p0-8 .. p0+71 of this read's y1, zeros outside [0, P)  (Conv1d zero padding)
        for (int i = tid; i < RL_ROWS * (RL_C / 4); i += 256) {
            const int r = i / (RL_C / 4), q = i % (RL_C / 4);
            const int64_t p = p0 - RL_PAD + r;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p >= 0 && p < P) v = *reinterpret_cast<const float4 *>(y1 + (bd * P + p) * RL_C + q * 4);
            *reinterpret_cast<float4 *>(ys + r * RL_YS + q * 4) = v;
        }
        float acc[4][8];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
        for (int t = 0; t < RL_TAPS; ++t) {
            for (int cc = 0; cc < RL_C / RL_KC; ++cc) {
                __syncthreads();                                   // previous chunk consumed (and ys staged)
                const float *wsrc = a.w_t + ((size_t)t * RL_C + cc * RL_KC) * RL_C;
                for (int i = tid; i < RL_KC * RL_C / 4; i += 256)
                    reinterpret_cast<float4 *>(ws)[i] = reinterpret_cast<const float4 *>(wsrc)[i];
                __syncthreads();
#pragma unroll 4
                for (int k = 0; k < RL_KC; ++k) {
                    float av[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) av[i] = ys[(ty * 4 + i + t) * RL_YS + cc * RL_KC + k];
                    const float4 b0 = *reinterpret_cast<const float4 *>(ws + k * RL_C + tx * 8);
                    const float4 b1 = *reinterpret_cast<const float4 *>(ws + k * RL_C + tx * 8 + 4);
                    const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float v = fmaxf(acc[i][j] + bias[j], 0.f);
                pooled[i][j] += (v - mean[j]) * invstd[j] * bw[j] + bb[j];
            }
    }
    const int n_groups = gridDim.y;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t p = p0 + ty * 4 + i;
        if (p >= P) continue;
        float *dst = partial + (((b * n_groups + g) * P + p) * RL_C) + tx * 8;
        *reinterpret_cast<float4 *>(dst) = make_float4(pooled[i][0], pooled[i][1], pooled[i][2], pooled[i][3]);
        *reinterpret_cast<float4 *>(dst + 4) = make_float4(pooled[i][4], pooled[i][5], pooled[i][6], pooled[i][7]);
    }
}

// ---------------------------------------------------------------------------------------------- conv k=17 on tcgen05
// The same convolution as an implicit GEMM on the tensor cores:  D[co][p] = sum_t sum_ci W[co][ci][t] . y1[p + t - 8][ci].
//   A = one tap's weights [128 co][128 ci]  (K-major fp16 hi | lo planes, pre-tiled in HBM, streamed through a two-stage
//       shared-memory ring with bulk copies; SS mode: 17 x 64 KiB of weights fit neither tensor memory nor shared memory)
//   B = ONE staged activation tile [144 positions][128 ci] (hi | lo) serves all 17 taps: tap t is the same buffer with the
//       descriptor's start address moved down t rows (K-major SWIZZLE_NONE: a row is 16 bytes inside its k-group block)
//   D = 128 columns of tensor memory (lane = output channel, column = position), three fp16 products per contraction like
//       the GRU kernels (fp32-faithful)
// A CTA owns (window b, 128 positions, a group of reads): for TWO reads at a time it builds the activation tiles in shared
// memory straight from the int8 features (embedding + k = 1 convolution + ReLU + BN1, never written to HBM), runs
// 17 x 24 MMAs per read against one pass of the weights, drains the two accumulators through ReLU + BN2 into per-thread
// sums (one output channel x 128 positions per thread), and writes the group's sum once.  Warp 0: weight producer; warp 1: MMA issuer, TMEM owner; warps 4-7: epilogue; all eight
// warps build the activation tile.
constexpr int CT_NPOS = 128;
constexpr int CT_ROWS = CT_NPOS + 2 * RL_PAD;            // 144 staged positions
constexpr int CT_BPLANE = (RL_C / 8) * CT_ROWS * 16;     // 36 864 B
constexpr int CT_BTILE = 2 * CT_BPLANE;                  // hi + lo of one read's activation tile
constexpr int CT_PAIR = 2;                               // reads that share one pass over the weights
constexpr int CT_WPLANE = (RL_C / 8) * RL_C * 16;        // 32 768 B: one plane of one tap = one ring stage
constexpr int CT_STAGES = 2;
constexpr int CT_OFF_W = CT_PAIR * CT_BTILE;
constexpr int CT_OFF_IN = CT_OFF_W + CT_STAGES * CT_WPLANE;
constexpr int CT_OFF_BAR = CT_OFF_IN + CT_PAIR * CT_ROWS * 8 * 4;
constexpr int CT_SMEM = CT_OFF_BAR + 128;

__global__ void __launch_bounds__(256, 1) rl_conv17_tc_kernel(const int8_t *__restrict__ x, const uint8_t *__restrict__ mask,
                                                              RlConv1 c1, RlConv17 c17, const uint8_t *__restrict__ w_tc,
                                                              int64_t P, int D, int F, int use_dwells, int dgroup,
                                                              float *__restrict__ partial) {
    extern __shared__ __align__(128) uint8_t smem_ct[];
    uint8_t *sb = smem_ct;                                             // [pair][hi | lo][k-group][144][8 halfs]
    uint8_t *sw = smem_ct + CT_OFF_W;                                  // [stage][k-group][128][8 halfs]
    float *sin = reinterpret_cast<float *>(smem_ct + CT_OFF_IN);       // [pair][144][8]
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_ct + CT_OFF_BAR);
    uint64_t *empty = full + CT_STAGES;
    uint64_t *acc_full = empty + CT_STAGES;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_full + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t b = blockIdx.z;
    const int g = blockIdx.y;
    const int64_t p0 = (int64_t)blockIdx.x * CT_NPOS;
    const int nin = RL_EMB + 1 + (use_dwells ? 1 : 0);

    if (tid == 0) {
        for (int i = 0; i < CT_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(acc_full, 1);
        fence_mbar_init();
    }
    if (warp == 1) { tmem_alloc(tmem_slot, 256); tmem_relinquish(); }
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    // builder constants: this thread's k = 1 convolution channel
    const int bc = tid & 127;
    float w1[RL_EMB + 2];
    for (int i = 0; i < nin; ++i) w1[i] = c1.w[bc * nin + i];
    const float b1 = c1.b[bc], m1 = c1.bn_mean[bc], s1 = c1.bn_invstd[bc], g1 = c1.bn_w[bc], o1 = c1.bn_b[bc];
    // epilogue constants: this thread's output channel (TMEM lane)
    const int co = (warp & 3) * 32 + lane;
    const float b2 = c17.b[co], m2 = c17.bn_mean[co], s2 = c17.bn_invstd[co], g2 = c17.bn_w[co], o2 = c17.bn_b[co];
    float pooled[CT_NPOS];
    if (warp >= 4) {
#pragma unroll
        for (int i = 0; i < CT_NPOS; ++i) pooled[i] = 0.f;
    }
    const uint32_t idesc = make_idesc_f16(128, CT_NPOS);
    const int d0 = g * dgroup, d1 = min(D, d0 + dgroup);
    uint32_t it = 0;             // weight-plane stages handed over so far (producer and issuer count alike)
    uint32_t n_done = 0;         // passes over the weights
    int d = d0;
    while (true) {
        // ---- the next one or two non-empty reads of the group share one pass over the 17 taps' weights (the weights
        //      come from L2 each time: with one read per pass all SMs together ask for more than L2 delivers)
        int dq[CT_PAIR], n_pair = 0;
        while (d < d1 && n_pair < CT_PAIR) {
            if (mask[b * D + d]) dq[n_pair++] = d;
            ++d;
        }
        if (n_pair == 0) break;                                    // uniform over the CTA
        // ---- build the activation tiles (the previous pass's MMAs are complete: everybody waited on acc_full below)
        for (int q = 0; q < n_pair; ++q) {
            if (tid < CT_ROWS) {
                const int64_t p = p0 - RL_PAD + tid;
                float *row = sin + (q * CT_ROWS + tid) * 8;
                if (p >= 0 && p < P) {
                    const int8_t *v = x + ((b * P + p) * D + dq[q]) * F;
                    const int base = min(max((int)v[0], 0), 5), strand = min(max((int)v[2] + 1, 0), 2);
                    for (int i = 0; i < RL_EMB; ++i) row[i] = c1.emb_base[base * RL_EMB + i] + c1.emb_strand[strand * RL_EMB + i];
                    row[RL_EMB] = (float)v[1] / 25.0f - 1.0f;
                    row[RL_EMB + 1] = use_dwells ? (float)v[4] : 0.f;
                } else {
                    row[0] = __int_as_float(0x7fc00000);          // marker: outside the window -> zero row (conv padding)
                }
            }
        }
        __syncthreads();
        for (int q = 0; q < n_pair; ++q) {
            uint8_t *tile = sb + q * CT_BTILE;
            for (int r = tid >> 7; r < CT_ROWS; r += 2) {
                const float *row = sin + (q * CT_ROWS + r) * 8;
                float y = 0.f;
                if (!(row[0] != row[0])) {
                    float acc = b1;
                    for (int k = 0; k < nin; ++k) acc = fmaf(w1[k], row[k], acc);
                    acc = fmaxf(acc, 0.f);
                    y = (acc - m1) * s1 * g1 + o1;
                }
                __half hi, lo;
                split_f16(y, hi, lo);
                const int off = (bc >> 3) * (CT_ROWS * 16) + r * 16 + (bc & 7) * 2;
                *reinterpret_cast<__half *>(tile + off) = hi;
                *reinterpret_cast<__half *>(tile + CT_BPLANE + off) = lo;
            }
        }
        fence_proxy_async_smem();
        tc_fence_before_sync();
        __syncthreads();
        tc_fence_after_sync();
        // ---- 17 taps x (hi plane, lo plane)
        if (warp == 0) {
            if (lane == 0) {
                for (int ps = 0; ps < 2 * RL_TAPS; ++ps, ++it) {
                    const uint32_t st = it % CT_STAGES;
                    mbar_wait(&empty[st], ((it / CT_STAGES) & 1) ^ 1);
                    mbar_arrive_expect_tx(&full[st], CT_WPLANE);
                    const uint8_t *src = w_tc + (size_t)ps * CT_WPLANE;           // [tap][hi | lo] back to back
#pragma unroll
                    for (int c = 0; c < 2; ++c) bulk_g2s(sw + st * CT_WPLANE + c * (CT_WPLANE / 2), src + c * (CT_WPLANE / 2), CT_WPLANE / 2, &full[st]);
                }
            } else {
                it += 2 * RL_TAPS;
            }
        } else if (warp == 1) {
            for (int ps = 0; ps < 2 * RL_TAPS; ++ps, ++it) {
                const uint32_t st = it % CT_STAGES;
                const int t = ps >> 1, lo_plane = ps & 1;
                mbar_wait(&full[st], (it / CT_STAGES) & 1);
                tc_fence_after_sync();
                if (elect_one()) {
                    const uint32_t a0 = smem_u32(sw + st * CT_WPLANE);
                    for (int q = 0; q < n_pair; ++q) {
                        const uint32_t dcol = tmem_base + (uint32_t)(q * CT_NPOS);
                        const uint32_t bb0 = smem_u32(sb + q * CT_BTILE) + (uint32_t)t * 16u;
                        // hi plane of the weights: x activation hi, then x activation lo;  lo plane: x activation hi
                        const int n_prod = lo_plane ? 1 : 2;
                        for (int prod = 0; prod < n_prod; ++prod) {
                            const int pb = lo_plane ? 0 : prod;
#pragma unroll
                            for (int ks = 0; ks < RL_C / 16; ++ks) {
                                const uint64_t ad = make_smem_desc(a0 + ks * 2 * (RL_C * 16), RL_C * 16, 128);
                                const uint64_t bdsc = make_smem_desc(bb0 + pb * CT_BPLANE + ks * 2 * (CT_ROWS * 16), CT_ROWS * 16, 128);
                                umma_f16(dcol, ad, bdsc, idesc, (ps | prod | ks) ? 1u : 0u);
                            }
                        }
                    }
                    umma_commit(&empty[st]);
                    if (ps == 2 * RL_TAPS - 1) umma_commit(acc_full);
                }
                __syncwarp();
            }
        } else {
            it += 2 * RL_TAPS;
        }
        // ---- everybody waits for the pass's accumulators (the activation tiles may then be rebuilt)
        mbar_wait(acc_full, n_done & 1);
        tc_fence_after_sync();
        if (warp >= 4) {
            for (int q = 0; q < n_pair; ++q) {
                const uint32_t t_lane = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(q * CT_NPOS);
#pragma unroll
                for (int c32 = 0; c32 < CT_NPOS; c32 += 32) {
                    uint32_t v[32];
                    tmem_ld_x32(t_lane + c32, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const float av = fmaxf(__uint_as_float(v[i]) + b2, 0.f);
                        pooled[c32 + i] += (av - m2) * s2 * g2 + o2;
                    }
                }
            }
        }
        tc_fence_before_sync();
        __syncthreads();                                           // accumulators drained, tiles free
        tc_fence_after_sync();
        ++n_done;
    }
    if (warp >= 4) {
        const int n_groups = gridDim.y;
        float *dst = partial + ((b * n_groups + g) * P + p0) * RL_C + co;
#pragma unroll
        for (int i = 0; i < CT_NPOS; ++i)
            if (p0 + i < P) dst[(int64_t)i * RL_C] = pooled[i];
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 1) { tc_fence_after_sync(); tmem_dealloc(tmem_base, 256); }
}

// ---------------------------------------------------------------------------------------------- mean + Linear(C -> H)
constexpr int RL_PLT = 16;        // positions per CTA of the pooling kernel
__global__ void __launch_bounds__(RL_H) rl_pool_linear_kernel(const float *__restrict__ partial, const uint8_t *__restrict__ mask,
                                                              const float *__restrict__ w_t, const float *__restrict__ bias,
                                                              int64_t P, int D, int n_groups, float *__restrict__ out) {
    // grid: (position tiles of 16, B); thread = channel while summing, output unit afterwards.  w_t [C k][H] (transposed)
    const int64_t b = blockIdx.y, p0 = (int64_t)blockIdx.x * RL_PLT;
    __shared__ float v[RL_PLT][RL_C];
    __shared__ int n_reads;
    if (threadIdx.x == 0) {
        int n = 0;
        for (int d = 0; d < D; ++d) n += mask[b * D + d];
        n_reads = n;
    }
    __syncthreads();
    for (int i = 0; i < RL_PLT; ++i) {
        const int64_t p = p0 + i;
        float s = 0.f;
        if (p < P)
            for (int g = 0; g < n_groups; ++g) s += partial[((b * n_groups + g) * P + p) * RL_C + threadIdx.x];
        v[i][threadIdx.x] = s / (float)n_reads;            // 0 / 0 = nan when a window has no reads, like the reference
    }
    __syncthreads();
    const int h = threadIdx.x;
    float acc[RL_PLT];
#pragma unroll
    for (int i = 0; i < RL_PLT; ++i) acc[i] = bias[h];
    for (int k = 0; k < RL_C; ++k) {
        const float w = w_t[k * RL_H + h];
#pragma unroll
        for (int i = 0; i < RL_PLT; ++i) acc[i] = fmaf(w, v[i][k], acc[i]);
    }
#pragma unroll
    for (int i = 0; i < RL_PLT; ++i)
        if (p0 + i < P) out[(b * P + p0 + i) * RL_H + h] = acc[i];
}

// ---------------------------------------------------------------------------------------------- generic fp32 GEMM
// C[M][N] = A[M][K] . W[N][K]^T + bias[N];  K % 16 == 0, N % 128 == 0.  128 x 128 x 16 tiles, 8 x 8 per thread.
__global__ void __launch_bounds__(256) rl_gemm_kernel(const float *__restrict__ A, const float *__restrict__ W,
                                                      const float *__restrict__ bias, float *__restrict__ C, int64_t M,
                                                      int K, int N) {
    __shared__ float As[16][128 + 4];
    __shared__ float Ws[16][128 + 4];
    const int tid = threadIdx.x;
    const int64_t m0 = (int64_t)blockIdx.x * 128;
    const int n0 = blockIdx.y * 128;
    const int tx = tid % 16, ty = tid / 16;
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    const int lrow = tid / 4, lk = (tid % 4) * 4;
    for (int k0 = 0; k0 < K; k0 += 16) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int r = lrow + half * 64;
            const int64_t gm = m0 + r;
            float4 av = make_float4(0.f, 0.f, 0.f, 0.f);
            if (gm < M) av = *reinterpret_cast<const float4 *>(A + gm * K + k0 + lk);
            As[lk + 0][r] = av.x; As[lk + 1][r] = av.y; As[lk + 2][r] = av.z; As[lk + 3][r] = av.w;
            const float4 wv = *reinterpret_cast<const float4 *>(W + (int64_t)(n0 + r) * K + k0 + lk);
            Ws[lk + 0][r] = wv.x; Ws[lk + 1][r] = wv.y; Ws[lk + 2][r] = wv.z; Ws[lk + 3][r] = wv.w;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&As[k][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4 *>(&As[k][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Ws[k][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4 *>(&Ws[k][64 + tx * 4]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
    float bv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) bv[j] = bias[n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + j - 4)];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t gm = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + i - 4);
        if (gm >= M) continue;
        float *dst = C + gm * N + n0;
        *reinterpret_cast<float4 *>(dst + tx * 4) = make_float4(acc[i][0] + bv[0], acc[i][1] + bv[1], acc[i][2] + bv[2], acc[i][3] + bv[3]);
        *reinterpret_cast<float4 *>(dst + 64 + tx * 4) = make_float4(acc[i][4] + bv[4], acc[i][5] + bv[5], acc[i][6] + bv[6], acc[i][7] + bv[7]);
    }
}

// ---------------------------------------------------------------------------------------------- LSTM recurrence
// gi  [B*P][2 dirs][4H]  (torch gate order i, f, g, o; b_ih + b_hh folded in)
// out [B*P][2H]          (columns dir*H + j)
// w3t [dir][H k][3H]     W_hh^T of gates i, f, g;   wo [dir][H j][H k]  W_hh rows of gate o
// One CTA = 4 windows of one direction, 256 threads = (half, unit j).  Half 0 computes gates i and f of unit j, half 1
// gates g and o; W_hh^T of i, f, g is resident in shared memory (192 KiB), gate o's row j lives in the 128 registers of
// thread (1, j).  The step is bound by shared-memory wavefronts (weights: 3 x 128 per warp pair; h: one broadcast
// 16-byte load per window and 4 k), so every load of h feeds two gates.
constexpr int RL_NB = 4;
constexpr int RL_LSTM_SMEM = (RL_H * 3 * RL_H + 2 * RL_NB * RL_H + 4 * RL_NB * RL_H) * 4;      // 208 KiB

__global__ void __launch_bounds__(256, 1) rl_lstm_kernel(const float *__restrict__ gi, const float *__restrict__ w3t,
                                                         const float *__restrict__ wo, float *__restrict__ out, int64_t B,
                                                         int64_t P) {
    extern __shared__ __align__(16) float smem_rl[];
    float *wt = smem_rl;                                  // [128 k][384]
    float *hs = wt + RL_H * 3 * RL_H;                     // [2][NB][128]
    float *pre = hs + 2 * RL_NB * RL_H;                   // [4 gates][NB][128]
    const int tid = threadIdx.x;
    const int half = tid >> 7, j = tid & 127;
    const int dir = blockIdx.y;
    const int64_t b0 = (int64_t)blockIdx.x * RL_NB;
    const int nb = (int)min((int64_t)RL_NB, B - b0);
    {
        const float *src = w3t + (size_t)dir * RL_H * 3 * RL_H;
        for (int i = tid; i < RL_H * 3 * RL_H / 4; i += 256) reinterpret_cast<float4 *>(wt)[i] = reinterpret_cast<const float4 *>(src)[i];
        for (int i = tid; i < 2 * RL_NB * RL_H; i += 256) hs[i] = 0.f;
    }
    float wq[RL_H];                                       // gate o, row j (half 1 only)
    if (half == 1) {
#pragma unroll
        for (int k = 0; k < RL_H; k += 4) {
            const float4 v = *reinterpret_cast<const float4 *>(wo + ((size_t)dir * RL_H + j) * RL_H + k);
            wq[k] = v.x; wq[k + 1] = v.y; wq[k + 2] = v.z; wq[k + 3] = v.w;
        }
    }
    // update phase: thread (half, j) owns windows n = half, half + 2 of unit j
    float c_state[RL_NB / 2];
#pragma unroll
    for (int q = 0; q < RL_NB / 2; ++q) c_state[q] = 0.f;
    __syncthreads();
    int cur = 0;
    float gnext[RL_NB / 2][4];
    auto fetch = [&](int64_t t, float (&dst)[RL_NB / 2][4]) {
#pragma unroll
        for (int q = 0; q < RL_NB / 2; ++q) {
            const int n = half + 2 * q;
            const bool ok = n < nb;
            const float *row = gi + (((b0 + (ok ? n : 0)) * P + t) * 2 + dir) * RL_G4;
#pragma unroll
            for (int gate = 0; gate < 4; ++gate) dst[q][gate] = ok ? __ldg(row + gate * RL_H + j) : 0.f;
        }
    };
    fetch(dir ? (P - 1) : 0, gnext);
    for (int64_t step = 0; step < P; ++step) {
        const int64_t t = dir ? (P - 1 - step) : step;
        const float *hc = hs + cur * RL_NB * RL_H;
        float gcur[RL_NB / 2][4];
#pragma unroll
        for (int q = 0; q < RL_NB / 2; ++q)
#pragma unroll
            for (int gate = 0; gate < 4; ++gate) gcur[q][gate] = gnext[q][gate];
        if (step + 1 < P) fetch(dir ? (t - 1) : (t + 1), gnext);
        float a0[RL_NB], a1[RL_NB];                       // half 0: i, f     half 1: g, o
#pragma unroll
        for (int n = 0; n < RL_NB; ++n) { a0[n] = 0.f; a1[n] = 0.f; }
        if (half == 0) {
#pragma unroll 4
            for (int k = 0; k < RL_H; k += 4) {
                float4 hv[RL_NB];
#pragma unroll
                for (int n = 0; n < RL_NB; ++n) hv[n] = *reinterpret_cast<const float4 *>(hc + n * RL_H + k);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const float wi = wt[(k + kk) * 3 * RL_H + j];
                    const float wf = wt[(k + kk) * 3 * RL_H + RL_H + j];
#pragma unroll
                    for (int n = 0; n < RL_NB; ++n) {
                        const float hvk = kk == 0 ? hv[n].x : kk == 1 ? hv[n].y : kk == 2 ? hv[n].z : hv[n].w;
                        a0[n] = fmaf(wi, hvk, a0[n]);
                        a1[n] = fmaf(wf, hvk, a1[n]);
                    }
                }
            }
        } else {
#pragma unroll
            for (int k = 0; k < RL_H; k += 4) {            // fully unrolled: wq[] must stay in registers
                float4 hv[RL_NB];
#pragma unroll
                for (int n = 0; n < RL_NB; ++n) hv[n] = *reinterpret_cast<const float4 *>(hc + n * RL_H + k);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const float wg = wt[(k + kk) * 3 * RL_H + 2 * RL_H + j];
                    const float wov = wq[k + kk];
#pragma unroll
                    for (int n = 0; n < RL_NB; ++n) {
                        const float hvk = kk == 0 ? hv[n].x : kk == 1 ? hv[n].y : kk == 2 ? hv[n].z : hv[n].w;
                        a0[n] = fmaf(wg, hvk, a0[n]);
                        a1[n] = fmaf(wov, hvk, a1[n]);
                    }
                }
            }
        }
#pragma unroll
        for (int n = 0; n < RL_NB; ++n) {
            pre[((2 * half) * RL_NB + n) * RL_H + j] = a0[n];
            pre[((2 * half + 1) * RL_NB + n) * RL_H + j] = a1[n];
        }
        __syncthreads();
        float *hn = hs + (cur ^ 1) * RL_NB * RL_H;
#pragma unroll
        for (int q = 0; q < RL_NB / 2; ++q) {
            const int n = half + 2 * q;
            const bool ok = n < nb;
            const float ig = rl_sigmoid(gcur[q][0] + pre[(0 * RL_NB + n) * RL_H + j]);
            const float fg = rl_sigmoid(gcur[q][1] + pre[(1 * RL_NB + n) * RL_H + j]);
            const float gg = tanhf(gcur[q][2] + pre[(2 * RL_NB + n) * RL_H + j]);
            const float og = rl_sigmoid(gcur[q][3] + pre[(3 * RL_NB + n) * RL_H + j]);
            const float c = fg * c_state[q] + ig * gg;
            c_state[q] = c;
            const float h = og * tanhf(c);
            hn[n * RL_H + j] = h;
            if (ok) out[((b0 + n) * P + t) * (2 * RL_H) + dir * RL_H + j] = h;
        }
        __syncthreads();
        cur ^= 1;
    }
}

// ---------------------------------------------------------------------------------------------- LSTM on tcgen05
// The recurrence with the matvec on the tensor cores:  G^T[4H][16 windows] = W_hh[4H][H] . h^T[H][16]  per time step.
//   A = W_hh: the fp16 hi plane of all four gates lives in TENSOR MEMORY (4 x 64 columns, TS mode) and so does the lo
//       plane of gates i and f (2 x 64 columns behind the accumulators); the lo plane of gates g and o comes from shared
//       memory as K-major operand tiles (SS mode) - hi + lo of all four gates would fill all 512 columns
//   B = the h tile [16 windows][128] the gate warps publish every step (fp16 hi | lo, K-major)
//   D = four 16-column accumulators (lane = hidden unit, column = window); three products per contraction:
//       W_hi.h_hi and W_hi.h_lo from tensor memory, W_lo.h_hi from shared memory
// One CTA = 16 windows of one direction; warps 0-7: gate warps (thread = hidden unit x 8 windows: c and h stay in
// registers, the input pre-activations are fetched one step ahead), warp 8: MMA issuer.  A step is the dependent chain
// publish h -> 96 MMAs -> gate arithmetic, like the one-tile GRU kernel.
constexpr int LT_N = 16;
constexpr int LT_WLO_GATE = (RL_H / 8) * RL_H * 16;          // 32 768 B: one gate's lo plane as A operand tiles
constexpr int LT_HPLANE = (RL_H / 8) * LT_N * 16;            // 4 096 B
constexpr int LT_OFF_H = 4 * LT_WLO_GATE;
constexpr int LT_OFF_BAR = LT_OFF_H + 2 * LT_HPLANE;
constexpr int LT_SMEM = LT_OFF_BAR + 64;
constexpr uint32_t LT_ACC_COL = 256;                         // accumulators behind the four 64-column weight blocks
constexpr uint32_t LT_LO_COL = 320;                          // lo plane of the first LT_LO_TMEM_GATES gates
constexpr int LT_LO_TMEM_GATES = 2;
constexpr int LT_W = LT_N / 2;                               // windows per gate thread
constexpr int LT_ISSUER = 8;                                 // warps 0-7 gate warps, warp 8 issues
constexpr int LT_THREADS = 32 * (LT_ISSUER + 1);
// MUFU-based gate functions (ex2.approx / rcp.approx, ~2 ulp): the gate phase is instruction bound
__device__ __forceinline__ float lt_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lt_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lt_sigmoid(float x) { return lt_rcp(1.0f + lt_ex2(-1.4426950408889634f * x)); }
__device__ __forceinline__ float lt_tanh(float x) { return fmaf(-2.0f, lt_rcp(1.0f + lt_ex2(2.8853900817779268f * x)), 1.0f); }

__global__ void __launch_bounds__(LT_THREADS, 1) rl_lstm_tc_kernel(const float *__restrict__ gi, const __half *__restrict__ w_hi,
                                                            const __half *__restrict__ w_lo_rm,
                                                            const uint8_t *__restrict__ w_lo_tiles, float *__restrict__ out,
                                                            int64_t B, int64_t P) {
    extern __shared__ __align__(128) uint8_t smem_lt[];
    uint8_t *swlo = smem_lt;
    uint8_t *sh = smem_lt + LT_OFF_H;
    uint64_t *acc_full = reinterpret_cast<uint64_t *>(smem_lt + LT_OFF_BAR);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_full + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int dir = blockIdx.y;
    const int64_t b0 = (int64_t)blockIdx.x * LT_N;
    const int nb = (int)min((int64_t)LT_N, B - b0);
    if (tid == 0) { mbar_init(acc_full, 1); fence_mbar_init(); }
    if (warp == LT_ISSUER) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
    // lo plane of W_hh -> shared memory (pre-tiled per direction: [gate][k-group][row][8 halfs]); h tile = 0
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(w_lo_tiles + (size_t)dir * 4 * LT_WLO_GATE);
        for (int i = tid; i < 4 * LT_WLO_GATE / 16; i += LT_THREADS) reinterpret_cast<uint4 *>(swlo)[i] = src[i];
        for (int i = tid; i < 2 * LT_HPLANE / 16; i += LT_THREADS) reinterpret_cast<uint4 *>(sh)[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    const int j = tid & 127;                                 // hidden unit of a gate thread
    if (warp < 4) {
        // (one warp per lane quarter) hi plane of W_hh (row-major fp16 [dir][4H][H]) -> tensor memory: gate g, k-step ks at column g*64 + ks*8
        const uint32_t t_w = tmem_base + ((uint32_t)(warp * 32) << 16);
        for (int g = 0; g < 4; ++g) {
            const uint4 *src = reinterpret_cast<const uint4 *>(w_hi + (((size_t)dir * 4 + g) * RL_H + j) * RL_H);
#pragma unroll
            for (int ks = 0; ks < RL_H / 16; ++ks) {
                const uint4 lo4 = src[2 * ks], hi4 = src[2 * ks + 1];
                const uint32_t v[8] = {lo4.x, lo4.y, lo4.z, lo4.w, hi4.x, hi4.y, hi4.z, hi4.w};
                tmem_st_x8(t_w + (uint32_t)(g * 64 + ks * 8), v);
            }
        }
        // the lo plane of gates i and f fits behind the accumulators (columns 320..447): their third product runs in
        // TS mode too (10 instead of 40 cycles per MMA); gates g and o take theirs from shared memory
        for (int g = 0; g < LT_LO_TMEM_GATES; ++g) {
            const uint4 *src = reinterpret_cast<const uint4 *>(w_lo_rm + (((size_t)dir * 4 + g) * RL_H + j) * RL_H);
#pragma unroll
            for (int ks = 0; ks < RL_H / 16; ++ks) {
                const uint4 lo4 = src[2 * ks], hi4 = src[2 * ks + 1];
                const uint32_t v[8] = {lo4.x, lo4.y, lo4.z, lo4.w, hi4.x, hi4.y, hi4.z, hi4.w};
                tmem_st_x8(t_w + LT_LO_COL + (uint32_t)(g * 64 + ks * 8), v);
            }
        }
        tmem_st_wait();
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();

    if (warp == LT_ISSUER) {
        const uint32_t idesc = make_idesc_f16(128, LT_N);
        const uint32_t h_hi = smem_u32(sh), h_lo = smem_u32(sh + LT_HPLANE), wl = smem_u32(swlo);
        for (int64_t step = 0; step < P; ++step) {
            if (elect_one()) {
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const uint32_t d = tmem_base + LT_ACC_COL + (uint32_t)(g * LT_N);
#pragma unroll
                    for (int ks = 0; ks < RL_H / 16; ++ks) {
                        const uint64_t bh = make_smem_desc(h_hi + ks * 2 * (LT_N * 16), LT_N * 16, 128);
                        umma_f16_ts(d, tmem_base + (uint32_t)(g * 64 + ks * 8), bh, idesc, ks ? 1u : 0u);
                    }
#pragma unroll
                    for (int ks = 0; ks < RL_H / 16; ++ks) {
                        const uint64_t bl = make_smem_desc(h_lo + ks * 2 * (LT_N * 16), LT_N * 16, 128);
                        umma_f16_ts(d, tmem_base + (uint32_t)(g * 64 + ks * 8), bl, idesc, 1u);
                    }
#pragma unroll
                    for (int ks = 0; ks < RL_H / 16; ++ks) {
                        const uint64_t bh = make_smem_desc(h_hi + ks * 2 * (LT_N * 16), LT_N * 16, 128);
                        if (g < LT_LO_TMEM_GATES) {
                            umma_f16_ts(d, tmem_base + LT_LO_COL + (uint32_t)(g * 64 + ks * 8), bh, idesc, 1u);
                        } else {
                            const uint64_t ad = make_smem_desc(wl + g * LT_WLO_GATE + ks * 2 * (RL_H * 16), RL_H * 16, 128);
                            umma_f16(d, ad, bh, idesc, 1u);
                        }
                    }
                }
                umma_commit(acc_full);
            }
            __syncwarp();
            tc_fence_before_sync();
            __syncthreads();                                   // the gate warps have published the next h tile
            tc_fence_after_sync();
        }
    } else {
        // warps w and w + 4 share TMEM lane quarter w (hidden units 32 w .. 32 w + 31) and split the 16 windows.
        // the input pre-activations of the NEXT step are loaded right after this step's arithmetic has consumed the
        // current ones: the loads fly under the publish and the next step's MMAs (one register set, not two)
        const int half = warp >> 2;
        float c_state[LT_W], gcur[4][LT_W];
#pragma unroll
        for (int n = 0; n < LT_W; ++n) c_state[n] = 0.f;
        auto fetch = [&](int64_t t) {
#pragma unroll
            for (int n = 0; n < LT_W; ++n) {
                const int wdw = half * LT_W + n;
                const bool ok = wdw < nb;
                const float *row = gi + (((b0 + (ok ? wdw : 0)) * P + t) * 2 + dir) * RL_G4 + j;
#pragma unroll
                for (int g = 0; g < 4; ++g) gcur[g][n] = ok ? __ldg(row + g * RL_H) : 0.f;
            }
        };
        fetch(dir ? (P - 1) : 0);
        const uint32_t t_lane = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + LT_ACC_COL + (uint32_t)(half * LT_W);
        const int hoff = (j >> 3) * (LT_N * 16) + (j & 7) * 2 + half * LT_W * 16;
        for (int64_t step = 0; step < P; ++step) {
            const int64_t t = dir ? (P - 1 - step) : step;
            mbar_wait(acc_full, (uint32_t)(step & 1));
            tc_fence_after_sync();
            uint32_t a[4][LT_W];
#pragma unroll
            for (int g = 0; g < 4; ++g) tmem_ld_x8(t_lane + (uint32_t)(g * LT_N), a[g]);
            tmem_ld_wait();
#pragma unroll
            for (int n = 0; n < LT_W; ++n) {
                const float ig = lt_sigmoid(gcur[0][n] + __uint_as_float(a[0][n]));
                const float fg = lt_sigmoid(gcur[1][n] + __uint_as_float(a[1][n]));
                const float gg = lt_tanh(gcur[2][n] + __uint_as_float(a[2][n]));
                const float og = lt_sigmoid(gcur[3][n] + __uint_as_float(a[3][n]));
                const float c = fmaf(fg, c_state[n], ig * gg);
                c_state[n] = c;
                const float h = og * lt_tanh(c);
                const int wdw = half * LT_W + n;
                if (wdw < nb) out[((b0 + wdw) * P + t) * (2 * RL_H) + dir * RL_H + j] = h;
                __half hi, lo;
                split_f16(h, hi, lo);
                *reinterpret_cast<__half *>(sh + hoff + n * 16) = hi;
                *reinterpret_cast<__half *>(sh + LT_HPLANE + hoff + n * 16) = lo;
            }
            if (step + 1 < P) fetch(dir ? (t - 1) : (t + 1));
            fence_proxy_async_smem();
            tc_fence_before_sync();
            __syncthreads();
            tc_fence_after_sync();
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == LT_ISSUER) { tc_fence_after_sync(); tmem_dealloc(tmem_base, 512); }
}

// ---------------------------------------------------------------------------------------------- engine
struct RlLstmLayer {
    __half *w_hi = nullptr;     // [2][4H][H] fp16 hi plane of W_hh (tensor-core kernel: -> tensor memory)
    __half *w_lo_rm = nullptr;  // [2][4H][H] fp16 lo plane, row-major (gates i, f: -> tensor memory)
    uint8_t *w_lo = nullptr;    // [2][4 gates][k-group 16][row 128][8 halfs] lo plane as shared-memory A operand tiles
    float *w_ih = nullptr;      // [2 dirs * 4H][in]   (both directions stacked: one GEMM)
    float *bias = nullptr;      // [2 * 4H]  b_ih + b_hh
    float *w3t = nullptr;       // [2][H][3H]
    float *wo = nullptr;        // [2][H][H]
};

}  // namespace mdk

using namespace mdk;

struct mdk_rl_engine {
    int device = 0;
    int use_dwells = 0;
    std::unordered_map<std::string, std::vector<float>> host;     // state-dict tensors as loaded
    bool prepared = false;
    // device parameters
    float *emb_base = nullptr, *emb_strand = nullptr;
    float *c1_w = nullptr, *c1_b = nullptr, *bn1[4] = {nullptr, nullptr, nullptr, nullptr};
    float *c17_wt = nullptr, *c17_b = nullptr, *bn2[4] = {nullptr, nullptr, nullptr, nullptr};
    uint8_t *c17_tc = nullptr;     // [17 taps][hi | lo][k-group 16][co 128][8 halfs]: the tensor-core kernel's A operand tiles
    int conv_tc = 1;               // 1: k = 17 convolution on tcgen05 (default), 0: fp32 CUDA cores
    int lstm_tc = 1;               // 1: LSTM recurrence on tcgen05 (default), 0: fp32 CUDA cores
    float *pool_w = nullptr, *pool_b = nullptr;
    RlLstmLayer lstm[2];
    float *lin_w = nullptr, *lin_b = nullptr;
    std::vector<void *> allocs;
    uint8_t *scratch = nullptr;    // per-call intermediates, grown on demand and kept
    size_t scratch_bytes = 0;
    cudaStream_t stream = nullptr;
};

namespace {

int rl_upload(mdk_rl_engine *e, const std::vector<float> &v, float **out) {
    void *p = nullptr;
    MDK_CUDA(cudaMalloc(&p, std::max<size_t>(v.size(), 1) * sizeof(float)));
    e->allocs.push_back(p);
    if (!v.empty()) MDK_CUDA(cudaMemcpy(p, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
    *out = static_cast<float *>(p);
    return MDK_OK;
}

const std::vector<float> *rl_get(mdk_rl_engine *e, const std::string &name, size_t want) {
    auto it = e->host.find(name);
    if (it == e->host.end()) { set_error("read-level model: tensor '" + name + "' was not loaded"); return nullptr; }
    if (it->second.size() != want) {
        set_error("read-level model: tensor '" + name + "' has " + std::to_string(it->second.size()) + " values, expected " +
                  std::to_string(want));
        return nullptr;
    }
    return &it->second;
}

int rl_prepare(mdk_rl_engine *e) {
    if (e->prepared) return MDK_OK;
    const int nin = RL_EMB + 1 + (e->use_dwells ? 1 : 0);
    int rc;
#define RL_NEED(var, name, n) const std::vector<float> *var = rl_get(e, name, (size_t)(n)); if (!var) return MDK_ERR_STATE;
    RL_NEED(eb, "base_embedder.weight", 6 * RL_EMB)
    RL_NEED(es, "strand_embedder.weight", 3 * RL_EMB)
    RL_NEED(c1w, "read_level_conv.convs.0.weight", RL_C * nin)
    RL_NEED(c1b, "read_level_conv.convs.0.bias", RL_C)
    RL_NEED(c17w, "read_level_conv.convs.3.weight", RL_C * RL_C * RL_TAPS)
    RL_NEED(c17b, "read_level_conv.convs.3.bias", RL_C)
    RL_NEED(pw, "pre_pool_expansion_layer.weight", RL_H * RL_C)
    RL_NEED(pb, "pre_pool_expansion_layer.bias", RL_H)
    RL_NEED(lw, "linear.weight", NCLS * 2 * RL_H)
    RL_NEED(lb, "linear.bias", NCLS)
    if ((rc = rl_upload(e, *eb, &e->emb_base)) || (rc = rl_upload(e, *es, &e->emb_strand)) || (rc = rl_upload(e, *c1w, &e->c1_w)) ||
        (rc = rl_upload(e, *c1b, &e->c1_b)) || (rc = rl_upload(e, *c17b, &e->c17_b)) ||
        (rc = rl_upload(e, *pb, &e->pool_b)) || (rc = rl_upload(e, *lw, &e->lin_w)) || (rc = rl_upload(e, *lb, &e->lin_b)))
        return rc;
    {   // Linear(C -> H) weights transposed to [k][h]: coalesced across the output units
        std::vector<float> wt((size_t)RL_C * RL_H);
        for (int h = 0; h < RL_H; ++h)
            for (int k = 0; k < RL_C; ++k) wt[(size_t)k * RL_H + h] = (*pw)[(size_t)h * RL_C + k];
        if ((rc = rl_upload(e, wt, &e->pool_w))) return rc;
    }
    // conv k = 17 weights: torch [out][in][tap] -> [tap][in][out]
    {
        std::vector<float> wt((size_t)RL_TAPS * RL_C * RL_C);
        for (int o = 0; o < RL_C; ++o)
            for (int i = 0; i < RL_C; ++i)
                for (int t = 0; t < RL_TAPS; ++t) wt[((size_t)t * RL_C + i) * RL_C + o] = (*c17w)[((size_t)o * RL_C + i) * RL_TAPS + t];
        if ((rc = rl_upload(e, wt, &e->c17_wt))) return rc;
        // the same weights as K-major fp16 hi / lo operand tiles, one 64 KiB block per tap
        std::vector<__half> tc((size_t)RL_TAPS * 2 * RL_C * RL_C);
        for (int t = 0; t < RL_TAPS; ++t)
            for (int o = 0; o < RL_C; ++o)
                for (int i = 0; i < RL_C; ++i) {
                    const float v = (*c17w)[((size_t)o * RL_C + i) * RL_TAPS + t];
                    const __half hi = __float2half_rn(v);
                    const __half lo = __float2half_rn(v - __half2float(hi));
                    const size_t off = (size_t)(i / 8) * (RL_C * 8) + (size_t)o * 8 + (i % 8);
                    tc[((size_t)t * 2 + 0) * RL_C * RL_C + off] = hi;
                    tc[((size_t)t * 2 + 1) * RL_C * RL_C + off] = lo;
                }
        void *p = nullptr;
        MDK_CUDA(cudaMalloc(&p, tc.size() * sizeof(__half)));
        e->allocs.push_back(p);
        MDK_CUDA(cudaMemcpy(p, tc.data(), tc.size() * sizeof(__half), cudaMemcpyHostToDevice));
        e->c17_tc = static_cast<uint8_t *>(p);
    }
    // BatchNorm (inference): mean, 1 / sqrt(var + eps), weight, bias
    for (int l = 0; l < 2; ++l) {
        const std::string base = std::string("read_level_conv.convs.") + (l == 0 ? "2" : "5") + ".";
        RL_NEED(mean, base + "running_mean", RL_C)
        RL_NEED(var, base + "running_var", RL_C)
        RL_NEED(w, base + "weight", RL_C)
        RL_NEED(b, base + "bias", RL_C)
        std::vector<float> invstd(RL_C);
        for (int c = 0; c < RL_C; ++c) invstd[c] = 1.0f / sqrtf((*var)[c] + 1e-5f);
        float **dst = l == 0 ? e->bn1 : e->bn2;
        if ((rc = rl_upload(e, *mean, &dst[0])) || (rc = rl_upload(e, invstd, &dst[1])) || (rc = rl_upload(e, *w, &dst[2])) ||
            (rc = rl_upload(e, *b, &dst[3])))
            return rc;
    }
    for (int l = 0; l < 2; ++l) {
        const int in = l == 0 ? RL_H : 2 * RL_H;
        std::vector<float> w_ih((size_t)2 * RL_G4 * in), bias((size_t)2 * RL_G4), w3t((size_t)2 * RL_H * 3 * RL_H),
            wo((size_t)2 * RL_H * RL_H);
        for (int d = 0; d < 2; ++d) {
            const std::string sfx = "_l" + std::to_string(l) + (d ? "_reverse" : "");
            RL_NEED(wih, "lstm.weight_ih" + sfx, RL_G4 * in)
            RL_NEED(whh, "lstm.weight_hh" + sfx, RL_G4 * RL_H)
            RL_NEED(bih, "lstm.bias_ih" + sfx, RL_G4)
            RL_NEED(bhh, "lstm.bias_hh" + sfx, RL_G4)
            std::copy(wih->begin(), wih->end(), w_ih.begin() + (size_t)d * RL_G4 * in);
            for (int r = 0; r < RL_G4; ++r) bias[(size_t)d * RL_G4 + r] = (*bih)[r] + (*bhh)[r];
            for (int gate = 0; gate < 3; ++gate)
                for (int jj = 0; jj < RL_H; ++jj)
                    for (int k = 0; k < RL_H; ++k)
                        w3t[((size_t)d * RL_H + k) * 3 * RL_H + gate * RL_H + jj] = (*whh)[((size_t)gate * RL_H + jj) * RL_H + k];
            for (int jj = 0; jj < RL_H; ++jj)
                for (int k = 0; k < RL_H; ++k) wo[((size_t)d * RL_H + jj) * RL_H + k] = (*whh)[((size_t)3 * RL_H + jj) * RL_H + k];
        }
        if ((rc = rl_upload(e, w_ih, &e->lstm[l].w_ih)) || (rc = rl_upload(e, bias, &e->lstm[l].bias)) ||
            (rc = rl_upload(e, w3t, &e->lstm[l].w3t)) || (rc = rl_upload(e, wo, &e->lstm[l].wo)))
            return rc;
        // tensor-core operands: hi plane row-major (torch's [4H][H] as it is), lo plane as K-major tiles per gate
        std::vector<__half> hi((size_t)2 * RL_G4 * RL_H), lo_t((size_t)2 * RL_G4 * RL_H), lo_rm((size_t)2 * RL_G4 * RL_H);
        for (int d = 0; d < 2; ++d) {
            const std::string sfx = "_l" + std::to_string(l) + (d ? "_reverse" : "");
            const std::vector<float> &whh = e->host["lstm.weight_hh" + sfx];
            for (int r = 0; r < RL_G4; ++r)
                for (int k = 0; k < RL_H; ++k) {
                    const float v = whh[(size_t)r * RL_H + k];
                    const __half h16 = __float2half_rn(v);
                    hi[((size_t)d * RL_G4 + r) * RL_H + k] = h16;
                    const int g = r / RL_H, jj = r % RL_H;
                    const __half l16 = __float2half_rn(v - __half2float(h16));
                    lo_t[(size_t)d * RL_G4 * RL_H + (((size_t)g * (RL_H / 8) + k / 8) * RL_H + jj) * 8 + (k % 8)] = l16;
                    lo_rm[((size_t)d * RL_G4 + r) * RL_H + k] = l16;
                }
        }
        void *p1 = nullptr, *p2 = nullptr, *p3 = nullptr;
        MDK_CUDA(cudaMalloc(&p3, lo_rm.size() * sizeof(__half)));
        e->allocs.push_back(p3);
        MDK_CUDA(cudaMemcpy(p3, lo_rm.data(), lo_rm.size() * sizeof(__half), cudaMemcpyHostToDevice));
        e->lstm[l].w_lo_rm = static_cast<__half *>(p3);
        MDK_CUDA(cudaMalloc(&p1, hi.size() * sizeof(__half)));
        e->allocs.push_back(p1);
        MDK_CUDA(cudaMalloc(&p2, lo_t.size() * sizeof(__half)));
        e->allocs.push_back(p2);
        MDK_CUDA(cudaMemcpy(p1, hi.data(), hi.size() * sizeof(__half), cudaMemcpyHostToDevice));
        MDK_CUDA(cudaMemcpy(p2, lo_t.data(), lo_t.size() * sizeof(__half), cudaMemcpyHostToDevice));
        e->lstm[l].w_hi = static_cast<__half *>(p1);
        e->lstm[l].w_lo = static_cast<uint8_t *>(p2);
    }
#undef RL_NEED
    e->prepared = true;
    return MDK_OK;
}

}  // namespace

extern "C" {

int mdk_rl_create(int device, int32_t lstm_size, int32_t cnn_size, int32_t use_dwells, int32_t num_classes,
                  mdk_rl_engine **out) {
    MDK_REQUIRE(out, MDK_ERR_ARG, "rl_create: out is NULL");
    *out = nullptr;
    MDK_REQUIRE(lstm_size == RL_H && cnn_size == RL_C, MDK_ERR_UNSUPPORTED, "rl_create: lstm_size = cnn_size = 128 only");
    MDK_REQUIRE(num_classes == NCLS, MDK_ERR_UNSUPPORTED, "rl_create: 5 classes only");
    MDK_CUDA(cudaSetDevice(device));
    mdk_rl_engine *e = new (std::nothrow) mdk_rl_engine();
    MDK_REQUIRE(e, MDK_ERR_NOMEM, "rl_create: out of host memory");
    e->device = device;
    e->use_dwells = use_dwells ? 1 : 0;
    {
        const char *v = getenv("MDK_RL_CONV");      // "fp32": CUDA-core convolution (validation)
        if (v && v[0] == 'f') { e->conv_tc = 0; e->lstm_tc = 0; }
    }
    cudaError_t err = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
    if (err != cudaSuccess) { delete e; return cuda_fail(err, "cudaStreamCreate", __FILE__, __LINE__); }
    *out = e;
    return MDK_OK;
}

int mdk_rl_destroy(mdk_rl_engine *e) {
    if (!e) return MDK_OK;
    cudaSetDevice(e->device);
    if (e->stream) { cudaStreamSynchronize(e->stream); cudaStreamDestroy(e->stream); }
    for (void *p : e->allocs) cudaFree(p);
    if (e->scratch) cudaFree(e->scratch);
    delete e;
    cudaGetLastError();
    return MDK_OK;
}

int mdk_rl_load(mdk_rl_engine *e, const char *name, const float *data, int64_t n) {
    MDK_REQUIRE(e && name && (data || n == 0) && n >= 0, MDK_ERR_ARG, "rl_load: bad arguments");
    MDK_REQUIRE(!e->prepared, MDK_ERR_STATE, "rl_load: the model has already run; create a new engine to change weights");
    e->host[name] = std::vector<float>(data, data + n);
    return MDK_OK;
}

int mdk_rl_set_conv(mdk_rl_engine *e, int tensor_cores) {
    MDK_REQUIRE(e, MDK_ERR_ARG, "rl_set_conv: engine is NULL");
    e->conv_tc = (tensor_cores & 1) ? 1 : 0;
    e->lstm_tc = (tensor_cores & 2) ? 1 : 0;
    return MDK_OK;
}

int mdk_rl_forward(mdk_rl_engine *e, const int8_t *x_host, int64_t B, int64_t P, int64_t D, int64_t F, float *probs_host) {
    MDK_REQUIRE(e && x_host && probs_host, MDK_ERR_ARG, "rl_forward: NULL argument");
    MDK_REQUIRE(B >= 1 && P >= 1 && D >= 1, MDK_ERR_ARG, "rl_forward: need B, P, D >= 1");
    MDK_REQUIRE(F == (e->use_dwells ? 5 : 4) || (!e->use_dwells && F >= 4), MDK_ERR_ARG,
                "rl_forward: feature vector length does not match the model (4, or 5 with dwells)");
    // grid limits (y, z <= 65 535; x < 2^31): B is gridDim.z of the convolution and y of the pooling, the read groups
    // gridDim.y (<= 16 384), B * D gridDim.x of the mask and fp32 k = 1 convolution kernels; positions are in x (or
    // strided over in y)
    MDK_REQUIRE(D <= 65535 && B <= 65535 && B * D <= 0x7fffffff, MDK_ERR_ARG, "rl_forward: B, D <= 65535, B * D < 2^31");
    MDK_CUDA(cudaSetDevice(e->device));
    int rc = rl_prepare(e);
    if (rc) return rc;
    cudaStream_t s = e->stream;
    const int dgroup = 4;
    const int n_groups = (int)((D + dgroup - 1) / dgroup);
    const int64_t BP = B * P;
    size_t off = 0;
    auto take = [&off](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t o_x = take((size_t)BP * D * F), o_mask = take((size_t)B * D), o_y1 = take(e->conv_tc ? 256 : (size_t)B * D * P * RL_C * 4),
                 o_part = take((size_t)B * n_groups * P * RL_C * 4), o_z = take((size_t)BP * RL_H * 4),
                 o_gi = take((size_t)BP * 2 * RL_G4 * 4), o_h0 = take((size_t)BP * 2 * RL_H * 4),
                 o_h1 = take((size_t)BP * 2 * RL_H * 4), o_probs = take((size_t)BP * NCLS * 4);
    if (off > e->scratch_bytes) {
        if (e->scratch) cudaFree(e->scratch);
        e->scratch = nullptr;
        e->scratch_bytes = 0;
        MDK_CUDA(cudaMalloc(&e->scratch, off + off / 8));
        e->scratch_bytes = off + off / 8;
    }
    uint8_t *buf = e->scratch;
    int8_t *d_x = (int8_t *)(buf + o_x);
    uint8_t *d_mask = buf + o_mask;
    float *d_y1 = (float *)(buf + o_y1), *d_part = (float *)(buf + o_part), *d_z = (float *)(buf + o_z),
          *d_gi = (float *)(buf + o_gi), *d_h0 = (float *)(buf + o_h0), *d_h1 = (float *)(buf + o_h1),
          *d_probs = (float *)(buf + o_probs);
    MDK_CUDA(cudaMemcpyAsync(d_x, x_host, (size_t)BP * D * F, cudaMemcpyHostToDevice, s));
    rl_mask_kernel<<<(unsigned)(B * D), 256, 0, s>>>(d_x, P, (int)D, (int)F, d_mask);
    RlConv1 c1{e->emb_base, e->emb_strand, e->c1_w, e->c1_b, e->bn1[0], e->bn1[1], e->bn1[2], e->bn1[3]};
    RlConv17 c17{e->c17_wt, e->c17_b, e->bn2[0], e->bn2[1], e->bn2[2], e->bn2[3]};
    if (e->conv_tc) {
        MDK_CUDA(cudaFuncSetAttribute(rl_conv17_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CT_SMEM));
        rl_conv17_tc_kernel<<<dim3((unsigned)((P + CT_NPOS - 1) / CT_NPOS), (unsigned)n_groups, (unsigned)B), 256, CT_SMEM, s>>>(
            d_x, d_mask, c1, c17, e->c17_tc, P, (int)D, (int)F, e->use_dwells, dgroup, d_part);
    } else {
        rl_embed_conv1_kernel<<<dim3((unsigned)(B * D), (unsigned)std::min<int64_t>((P + 31) / 32, 65535)), RL_C, 0, s>>>(
            d_x, d_mask, c1, P, (int)D, (int)F, e->use_dwells, d_y1);
        MDK_CUDA(cudaFuncSetAttribute(rl_conv17_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, RL_CONV_SMEM));
        rl_conv17_pool_kernel<<<dim3((unsigned)((P + RL_PT - 1) / RL_PT), (unsigned)n_groups, (unsigned)B), 256, RL_CONV_SMEM, s>>>(
            d_y1, d_mask, c17, P, (int)D, dgroup, d_part);
    }
    rl_pool_linear_kernel<<<dim3((unsigned)((P + RL_PLT - 1) / RL_PLT), (unsigned)B), RL_H, 0, s>>>(d_part, d_mask, e->pool_w, e->pool_b, P, (int)D,
                                                                          n_groups, d_z);
    MDK_CUDA(cudaFuncSetAttribute(rl_lstm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, RL_LSTM_SMEM));
    const float *layer_in = d_z;
    float *layer_out[2] = {d_h0, d_h1};
    for (int l = 0; l < 2; ++l) {
        const int in = l == 0 ? RL_H : 2 * RL_H;
        rl_gemm_kernel<<<dim3((unsigned)((BP + 127) / 128), 2 * RL_G4 / 128), 256, 0, s>>>(layer_in, e->lstm[l].w_ih, e->lstm[l].bias,
                                                                                       d_gi, BP, in, 2 * RL_G4);
        if (e->lstm_tc) {
            MDK_CUDA(cudaFuncSetAttribute(rl_lstm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LT_SMEM));
            rl_lstm_tc_kernel<<<dim3((unsigned)((B + LT_N - 1) / LT_N), 2), LT_THREADS, LT_SMEM, s>>>(d_gi, e->lstm[l].w_hi, e->lstm[l].w_lo_rm,
                                                                                            e->lstm[l].w_lo, layer_out[l], B, P);
        } else {
            rl_lstm_kernel<<<dim3((unsigned)((B + RL_NB - 1) / RL_NB), 2), 256, RL_LSTM_SMEM, s>>>(d_gi, e->lstm[l].w3t, e->lstm[l].wo,
                                                                                                layer_out[l], B, P);
        }
        layer_in = layer_out[l];
    }
    MDK_CUDA(cudaGetLastError());
    MDK_CUDA(launch_head(d_h1, e->lin_w, e->lin_b, B, P, 0, d_probs, nullptr, nullptr, s));
    MDK_CUDA(cudaMemcpyAsync(probs_host, d_probs, (size_t)BP * NCLS * 4, cudaMemcpyDeviceToHost, s));
    MDK_CUDA(cudaStreamSynchronize(s));
    return MDK_OK;
}

}  // extern "C"
