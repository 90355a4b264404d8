// Memory-bound pieces of the unit encoder and the target-unit attention head (policy.py:99-136,144-153).
//
// The 128x128 unit-embedding GEMMs run on the tensor cores (gemm_tf32x3.cu); everything around them is
// bandwidth work on ~20 KB/token of activations and is written here so that each tensor crosses HBM once:
//
//   env_fwd / env_bwd   relu(env W_e^T + b_e), 3 -> 128, written into / read from columns [0,128) of the concatenated
//                       [N, 896] pre-rnn input row (no torch.cat), policy.py:55,97
//   unit_basic_fwd      relu(units W_b^T + b_b)            [R,12] -> [R,128]     (K = 12: not a tensor-core shape),
//                       optionally with its ReLU sign bits for the data-gradient kernel
//   unit_basic reduce   fixed-order sum of the dW_b / db_b partials of the fused data-gradient kernel (gemm_tf32x3.cu)
//   target_unit_q_fwd   logits[n,u] = <att[n] W_g, basic[n,u]> + <att[n], b_g>: the head WITHOUT the [N,40,128] embedding
//   target_unit_q_bwd   s_g[n] = sum_u dlogits[n,u] basic_g[n,u] (-> d_att and the head's share of dW_g as token-level GEMMs)
//   target_unit_fwd/bwd the dense form on a materialised embedding (policy.py:152-153), for callers that keep one
// The max-pool over a group's units lives in the embedding GEMM's epilogue (dc_gemm_unit_max) and its backward routing is
// generated inside the weight- / data-gradient kernels (dc_unit_wgrad_routed, dc_unit_dgrad_fused), all in gemm_tf32x3.cu.
//
// Thread mapping everywhere: one warp per row of 128 channels, lane l owns channels 4l..4l+3 -> every global access
// is a fully coalesced 512-byte row segment (16 bytes per lane).
#include "dc_common.cuh"

namespace {

constexpr int kC = 128;          // embedding width (policy.py:56-63)
constexpr int kIn = 12;          // unit feature count (policy.py:56)
constexpr int kWarps = 8;
constexpr int kThreadsE = kWarps * 32;
constexpr int kMaxUnits = 40;

// ---- relu(units W_b^T + b_b) -------------------------------------------------------------------
// mask (optional): the ReLU sign bits for the data-gradient kernel, uint32 [ceil(R/32)][128] with bit i of word [b][j] =
// basic[32b + i][j] > 0 (bits of rows >= R are 0).  A warp iteration owns 32 rows starting at a multiple of 32 and lane l owns
// channels 4l..4l+3, so a lane collects one bit per row in four registers and stores one 16-byte word per iteration (512 coalesced
// bytes per warp).  The bit is taken from the value written to `basic`, so the backward sees exactly the forward's mask.
__global__ void __launch_bounds__(kThreadsE) unit_basic_fwd_kernel(const float *__restrict__ units,
                                                                   const float *__restrict__ w_b,
                                                                   const float *__restrict__ b_b,
                                                                   float *__restrict__ basic, uint32_t *__restrict__ mask,
                                                                   int64_t R) {
    __shared__ float s_u[kWarps][32][kIn];                        // 32 rows of raw features per warp per iteration
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // weights as channel PAIRS for the packed fp32x2 FMA (FFMA2): w2[p][k] = (W_b[4l+2p][k], W_b[4l+2p+1][k])
    float2 w2[2][kIn], b2[2];
#pragma unroll
    for (int p = 0; p < 2; ++p) {
        b2[p] = make_float2(b_b[lane * 4 + 2 * p], b_b[lane * 4 + 2 * p + 1]);
#pragma unroll
        for (int k = 0; k < kIn; ++k) w2[p][k] = make_float2(w_b[(lane * 4 + 2 * p) * kIn + k], w_b[(lane * 4 + 2 * p + 1) * kIn + k]);
    }
    const int64_t rows_per_iter = (int64_t)gridDim.x * kWarps * 32;
    for (int64_t base = ((int64_t)blockIdx.x * kWarps + warp) * 32; base < R; base += rows_per_iter) {
        const int nrows = (int)min((int64_t)32, R - base);
        // stage 32 x 12 contiguous floats (coalesced), then every lane reads each row as a broadcast
        float *su = &s_u[warp][0][0];
        for (int i = lane; i < nrows * kIn; i += 32) su[i] = units[base * kIn + i];
        __syncwarp();
        uint4 bits = make_uint4(0u, 0u, 0u, 0u);
        for (int r = 0; r < nrows; ++r) {
            float2 a0 = b2[0], a1 = b2[1];
#pragma unroll
            for (int k = 0; k < kIn; ++k) {
                const float u = s_u[warp][r][k];
                const float2 uu = make_float2(u, u);
                a0 = __ffma2_rn(uu, w2[0][k], a0);
                a1 = __ffma2_rn(uu, w2[1][k], a1);
            }
            const float4 o = make_float4(fmaxf(a0.x, 0.f), fmaxf(a0.y, 0.f), fmaxf(a1.x, 0.f), fmaxf(a1.y, 0.f));
            *reinterpret_cast<float4 *>(basic + (base + r) * kC + lane * 4) = o;
            bits.x |= (uint32_t)(o.x > 0.f) << r; bits.y |= (uint32_t)(o.y > 0.f) << r;
            bits.z |= (uint32_t)(o.z > 0.f) << r; bits.w |= (uint32_t)(o.w > 0.f) << r;
        }
        if (mask != nullptr) *reinterpret_cast<uint4 *>(mask + (base >> 5) * kC + lane * 4) = bits;
        __syncwarp();
    }
}

// ---- dW_b, db_b: fixed-order sum of the [128][13] partials of dc_unit_dgrad_fused (12 weight-gradient columns + the bias gradient)
__global__ void unit_basic_bwd_reduce_kernel(const float *__restrict__ partial, int nblocks, float *__restrict__ dw_b,
                                             float *__restrict__ db_b, int accumulate) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;          // over 128 x 13
    if (i >= kC * (kIn + 1)) return;
    float s = 0.f;
    for (int b = 0; b < nblocks; ++b) s += partial[(size_t)b * kC * (kIn + 1) + i];
    const int o = i / (kIn + 1), k = i % (kIn + 1);
    float *dst = k < kIn ? dw_b + o * kIn + k : db_b + o;
    *dst = accumulate ? *dst + s : s;
}

// ---- environment encoder: relu(env W_e^T + b_e), 3 -> 128 (policy.py:55,97) ---------------------------------------
// Written straight into columns [0,128) of the concatenated pre-rnn input row (row pitch ld), next to the group maxima
// that dc_gemm_unit_max puts in columns [128,896): the reference's torch.cat (policy.py:129-136) never materialises.
constexpr int kEnvIn = 3;
__global__ void __launch_bounds__(kThreadsE) env_fwd_kernel(const float *__restrict__ env, const float *__restrict__ w_e,
                                                            const float *__restrict__ b_e, float *__restrict__ out, int ld,
                                                            int64_t N) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float w[4][kEnvIn], b[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        b[c] = b_e[lane * 4 + c];
#pragma unroll
        for (int k = 0; k < kEnvIn; ++k) w[c][k] = w_e[(lane * 4 + c) * kEnvIn + k];
    }
    const int64_t rows_per_iter = (int64_t)gridDim.x * kWarps * 32;
    for (int64_t base = ((int64_t)blockIdx.x * kWarps + warp) * 32; base < N; base += rows_per_iter) {
        const int nrows = (int)min((int64_t)32, N - base);
        float e[kEnvIn];                                           // lane r holds row base+r, rows are broadcast by shuffle
#pragma unroll
        for (int k = 0; k < kEnvIn; ++k) e[k] = lane < nrows ? env[(base + lane) * kEnvIn + k] : 0.f;
        for (int r = 0; r < nrows; ++r) {
            float a[4] = {b[0], b[1], b[2], b[3]};
#pragma unroll
            for (int k = 0; k < kEnvIn; ++k) {
                const float u = __shfl_sync(0xffffffffu, e[k], r);
#pragma unroll
                for (int c = 0; c < 4; ++c) a[c] = fmaf(u, w[c][k], a[c]);
            }
            *reinterpret_cast<float4 *>(out + (base + r) * ld + lane * 4) =
                make_float4(fmaxf(a[0], 0.f), fmaxf(a[1], 0.f), fmaxf(a[2], 0.f), fmaxf(a[3], 0.f));
        }
    }
}

// dW_e, db_e from d_out, the ReLU mask (out > 0) and env: partial[block][128][4] (3 weight columns + bias), then reduced.
__global__ void __launch_bounds__(kThreadsE) env_bwd_kernel(const float *__restrict__ d_out, const float *__restrict__ out, int ld,
                                                            const float *__restrict__ env, int64_t N,
                                                            float *__restrict__ partial) {
    __shared__ float s_red[kC][kEnvIn + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float acc[4][kEnvIn + 1];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int k = 0; k <= kEnvIn; ++k) acc[c][k] = 0.f;
    const int64_t rows_per_iter = (int64_t)gridDim.x * kWarps * 32;
    for (int64_t base = ((int64_t)blockIdx.x * kWarps + warp) * 32; base < N; base += rows_per_iter) {
        const int nrows = (int)min((int64_t)32, N - base);
        float e[kEnvIn];
#pragma unroll
        for (int k = 0; k < kEnvIn; ++k) e[k] = lane < nrows ? env[(base + lane) * kEnvIn + k] : 0.f;
        for (int r0 = 0; r0 < nrows; r0 += 8) {                    // 8 rows per trip: 16 independent 16-byte loads per lane
            float4 g4[8], y4[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int r = min(r0 + j, nrows - 1);
                g4[j] = __ldg(reinterpret_cast<const float4 *>(d_out + (base + r) * ld) + lane);
                y4[j] = __ldg(reinterpret_cast<const float4 *>(out + (base + r) * ld) + lane);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const bool live = r0 + j < nrows;                  // uniform across the warp
                const float g[4] = {live && y4[j].x > 0.f ? g4[j].x : 0.f, live && y4[j].y > 0.f ? g4[j].y : 0.f,
                                    live && y4[j].z > 0.f ? g4[j].z : 0.f, live && y4[j].w > 0.f ? g4[j].w : 0.f};
#pragma unroll
                for (int k = 0; k < kEnvIn; ++k) {
                    const float u = __shfl_sync(0xffffffffu, e[k], min(r0 + j, 31));
#pragma unroll
                    for (int c = 0; c < 4; ++c) acc[c][k] = fmaf(g[c], u, acc[c][k]);
                }
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[c][kEnvIn] += g[c];
            }
        }
    }
    for (int w = 0; w < kWarps; ++w) {                             // fixed fold order: deterministic
        if (warp == w) {
#pragma unroll
            for (int c = 0; c < 4; ++c)
#pragma unroll
                for (int k = 0; k <= kEnvIn; ++k) {
                    float *dst = &s_red[lane * 4 + c][k];
                    *dst = (w == 0 ? 0.f : *dst) + acc[c][k];
                }
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < kC * (kEnvIn + 1); i += kThreadsE)
        partial[(size_t)blockIdx.x * kC * (kEnvIn + 1) + i] = (&s_red[0][0])[i];
}

// 32 outputs x 8 block-groups per CTA: group y sums blocks y, y+8, ...; the groups are then added in order.
__global__ void __launch_bounds__(256) env_bwd_reduce_kernel(const float *__restrict__ partial, int nblocks, float *__restrict__ dw_e,
                                                             float *__restrict__ db_e) {
    __shared__ float sh[8][32];
    const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + x;                             // over 128 x 4
    float s = 0.f;
    if (i < kC * (kEnvIn + 1))
        for (int b = y; b < nblocks; b += 8) s += partial[(size_t)b * kC * (kEnvIn + 1) + i];
    sh[y][x] = s;
    __syncthreads();
    if (y == 0 && i < kC * (kEnvIn + 1)) {
        float t = 0.f;
#pragma unroll
        for (int r = 0; r < 8; ++r) t += sh[r][x];
        const int o = i / (kEnvIn + 1), k = i % (kEnvIn + 1);
        if (k < kEnvIn) dw_e[o * kEnvIn + k] = t; else db_e[o] = t;
    }
}

// ---- target-unit attention head ---------------------------------------------------------------------
__global__ void __launch_bounds__(kThreadsE) target_unit_fwd_kernel(const float *__restrict__ att,
                                                                    const float *__restrict__ ue,
                                                                    float *__restrict__ logits, int64_t N) {
    const int lane = threadIdx.x & 31;
    const int64_t n = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (n >= N) return;
    const float4 a = __ldg(reinterpret_cast<const float4 *>(att + n * kC) + lane);
    const float4 *row = reinterpret_cast<const float4 *>(ue + n * kMaxUnits * kC) + lane;
    float mine = 0.f;                                             // lane u keeps logit u (u < 32), lanes 0..7 also u+32
    float mine_hi = 0.f;
#pragma unroll 8
    for (int u = 0; u < kMaxUnits; ++u) {
        const float4 v = __ldg(row + u * (kC / 4));
        float d = v.x * a.x + v.y * a.y + v.z * a.z + v.w * a.w;
        d = dc_warp_sum(d);
        if (u < 32) { if (lane == u) mine = d; } else { if (lane == u - 32) mine_hi = d; }
    }
    logits[n * kMaxUnits + lane] = mine;
    if (lane < kMaxUnits - 32) logits[n * kMaxUnits + 32 + lane] = mine_hi;
}

__global__ void __launch_bounds__(kThreadsE) target_unit_bwd_kernel(const float *__restrict__ dlogits,
                                                                    const float *__restrict__ att,
                                                                    const float *__restrict__ ue,
                                                                    float *__restrict__ d_att, float *__restrict__ d_ue,
                                                                    int64_t N) {
    const int lane = threadIdx.x & 31;
    const int64_t n = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (n >= N) return;
    const float g_lo = dlogits[n * kMaxUnits + lane];
    const float g_hi = lane < kMaxUnits - 32 ? dlogits[n * kMaxUnits + 32 + lane] : 0.f;
    const bool any = __any_sync(0xffffffffu, g_lo != 0.f || g_hi != 0.f);
    float4 *drow = d_ue ? reinterpret_cast<float4 *>(d_ue + n * kMaxUnits * kC) + lane : nullptr;   // NULL: d_att only
    float4 da = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!any) {                                                   // head unused on this token: exact zeros, no reads
        if (drow) {
#pragma unroll 8
            for (int u = 0; u < kMaxUnits; ++u) drow[u * (kC / 4)] = da;
        }
    } else {
        const float4 a = __ldg(reinterpret_cast<const float4 *>(att + n * kC) + lane);
        const float4 *row = reinterpret_cast<const float4 *>(ue + n * kMaxUnits * kC) + lane;
#pragma unroll 8
        for (int u = 0; u < kMaxUnits; ++u) {
            const float g = __shfl_sync(0xffffffffu, u < 32 ? g_lo : g_hi, u & 31);
            const float4 v = __ldg(row + u * (kC / 4));
            da.x = fmaf(g, v.x, da.x); da.y = fmaf(g, v.y, da.y); da.z = fmaf(g, v.z, da.z); da.w = fmaf(g, v.w, da.w);
            if (drow) drow[u * (kC / 4)] = make_float4(g * a.x, g * a.y, g * a.z, g * a.w);
        }
    }
    *(reinterpret_cast<float4 *>(d_att + n * kC) + lane) = da;
}

int grid_rows(int64_t rows_per_block_iter_unused) { (void)rows_per_block_iter_unused; return 4 * dc_sm_count(); }


// ---- target-unit head without the unit embedding ------------------------------------------------------------------------
// logits[n,u] = <att[n], W_g basic[n,u] + b_g> = <att[n] W_g, basic[n,u]> + <att[n], b_g> (policy.py:144-153; algebra pinned in
// tests/test_oracle.py): with q[n, g*128 + j] = (att W_g)[n, j] and q[n, 768 + g] = <att[n], b_g> from ONE small GEMM over tokens,
// the head reads the stored `basic` rows and the [N, 40, 128] embedding is never materialised.
struct BasicPtrs { const float *p[6]; };
__constant__ int kGroupUnits[6] = {1, 5, 16, 16, 1, 1};
__constant__ int kGroupOffset[6] = {0, 1, 6, 22, 38, 39};

__global__ void __launch_bounds__(kThreadsE) target_unit_q_fwd_kernel(const float *__restrict__ q, int ld_q, BasicPtrs basics,
                                                                      float *__restrict__ logits, int64_t N) {
    const int lane = threadIdx.x & 31;
    const int64_t n = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (n >= N) return;
    const float *qrow = q + n * ld_q;
    float mine = 0.f, mine_hi = 0.f;                              // lane u keeps logit u (u < 32), lanes 0..7 also u+32
#pragma unroll
    for (int g = 0; g < 6; ++g) {
        const float4 a = __ldg(reinterpret_cast<const float4 *>(qrow + g * kC) + lane);
        const float c = __ldg(qrow + 6 * kC + g);
        const int nu = kGroupUnits[g], off = kGroupOffset[g];
        const float4 *row = reinterpret_cast<const float4 *>(basics.p[g] + n * nu * kC) + lane;
        for (int u = 0; u < nu; ++u) {
            const float4 v = __ldg(row + u * (kC / 4));
            float d = v.x * a.x + v.y * a.y + v.z * a.z + v.w * a.w;
            d = dc_warp_sum(d) + c;
            const int o = off + u;
            if (o < 32) { if (lane == o) mine = d; } else { if (lane == o - 32) mine_hi = d; }
        }
    }
    logits[n * kMaxUnits + lane] = mine;
    if (lane < kMaxUnits - 32) logits[n * kMaxUnits + 32 + lane] = mine_hi;
}

// s[n, g*128 + j] = sum_u dlogits[n, off_g + u] basic_g[n,u,j],  s[n, 768 + g] = sum_u dlogits[n, off_g + u]  (zeros elsewhere):
// d_att = s [W_0 | ... | W_5 | b_0..b_5]^T is then one GEMM over tokens.  Tokens that did not use the head write zeros, read nothing.
__global__ void __launch_bounds__(kThreadsE) target_unit_q_bwd_kernel(const float *__restrict__ dlogits, BasicPtrs basics,
                                                                      float *__restrict__ s, int ld_s, int64_t N) {
    const int lane = threadIdx.x & 31;
    const int64_t n = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
    if (n >= N) return;
    const float g_lo = dlogits[n * kMaxUnits + lane];
    const float g_hi = lane < kMaxUnits - 32 ? dlogits[n * kMaxUnits + 32 + lane] : 0.f;
    const bool any = __any_sync(0xffffffffu, g_lo != 0.f || g_hi != 0.f);
    float4 *srow = reinterpret_cast<float4 *>(s + n * ld_s) + lane;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!any) {
#pragma unroll
        for (int g = 0; g < 7; ++g) srow[g * (kC / 4)] = zero;
        return;
    }
    float sig[6];
#pragma unroll
    for (int g = 0; g < 6; ++g) {
        const int nu = kGroupUnits[g], off = kGroupOffset[g];
        const float4 *row = reinterpret_cast<const float4 *>(basics.p[g] + n * nu * kC) + lane;
        float4 acc = zero;
        float sg = 0.f;
        for (int u = 0; u < nu; ++u) {
            const int o = off + u;
            const float gv = __shfl_sync(0xffffffffu, o < 32 ? g_lo : g_hi, o & 31);
            const float4 v = __ldg(row + u * (kC / 4));
            acc.x = fmaf(gv, v.x, acc.x); acc.y = fmaf(gv, v.y, acc.y); acc.z = fmaf(gv, v.z, acc.z); acc.w = fmaf(gv, v.w, acc.w);
            sg += gv;
        }
        srow[g * (kC / 4)] = acc;
        sig[g] = sg;
    }
    float4 tail = zero;                                            // columns 768..895: the six sums, then zeros
    if (lane == 0) tail = make_float4(sig[0], sig[1], sig[2], sig[3]);
    if (lane == 1) tail = make_float4(sig[4], sig[5], 0.f, 0.f);
    srow[6 * (kC / 4)] = tail;
}

}  // namespace

extern "C" int dc_unit_basic_fwd(const float *units, const float *w_b, const float *b_b, float *basic, int64_t R,
                                 dc_stream_t stream) {
    DC_REQUIRE(units && w_b && b_b && basic && R > 0, DC_EINVAL, "dc_unit_basic_fwd: bad arguments");
    DC_REQUIRE(((uintptr_t)basic & 15) == 0, DC_EINVAL, "dc_unit_basic_fwd: output must be 16-byte aligned");
    unit_basic_fwd_kernel<<<grid_rows(0), kThreadsE, 0, dc_cu_stream(stream)>>>(units, w_b, b_b, basic, nullptr, R);
    DC_LAUNCH_OK();
    return DC_OK;
}

extern "C" int dc_unit_basic_fwd_mask(const float *units, const float *w_b, const float *b_b, float *basic, uint32_t *mask,
                                      int64_t R, dc_stream_t stream) {
    DC_REQUIRE(units && w_b && b_b && basic && mask && R > 0, DC_EINVAL, "dc_unit_basic_fwd_mask: bad arguments");
    DC_REQUIRE(((uintptr_t)basic & 15) == 0 && ((uintptr_t)mask & 15) == 0, DC_EINVAL,
               "dc_unit_basic_fwd_mask: basic and mask must be 16-byte aligned");
    unit_basic_fwd_kernel<<<grid_rows(0), kThreadsE, 0, dc_cu_stream(stream)>>>(units, w_b, b_b, basic, mask, R);
    DC_LAUNCH_OK();
    return DC_OK;
}

extern "C" size_t dc_unit_basic_bwd_workspace_bytes(void) { return (size_t)4 * 1024 * kC * (kIn + 1) * sizeof(float); }

int dc_unit_basic_reduce(const float *partial, int nblocks, float *dw_b, float *db_b, int accumulate, cudaStream_t st) {
    unit_basic_bwd_reduce_kernel<<<(kC * (kIn + 1) + 255) / 256, 256, 0, st>>>(partial, nblocks, dw_b, db_b, accumulate);
    DC_LAUNCH_OK();
    return DC_OK;
}

extern "C" int dc_env_fwd(const float *env, const float *w_e, const float *b_e, float *out, int ld_out, int64_t N,
                          dc_stream_t stream) {
    DC_REQUIRE(env && w_e && b_e && out && N > 0 && ld_out >= kC && ld_out % 4 == 0 && ((uintptr_t)out & 15) == 0, DC_EINVAL,
               "dc_env_fwd: bad arguments");
    env_fwd_kernel<<<grid_rows(0), kThreadsE, 0, dc_cu_stream(stream)>>>(env, w_e, b_e, out, ld_out, N);
    DC_LAUNCH_OK();
    return DC_OK;
}

extern "C" size_t dc_env_bwd_workspace_bytes(void) { return (size_t)1024 * kC * (kEnvIn + 1) * sizeof(float); }

extern "C" int dc_env_bwd(const float *d_out, const float *out, int ld, const float *env, float *dw_e, float *db_e, int64_t N,
                          void *workspace, dc_stream_t stream) {
    DC_REQUIRE(d_out && out && env && dw_e && db_e && workspace && N > 0 && ld >= kC && ld % 4 == 0, DC_EINVAL,
               "dc_env_bwd: bad arguments");
    DC_REQUIRE((((uintptr_t)d_out | (uintptr_t)out) & 15) == 0, DC_EINVAL, "dc_env_bwd: inputs must be 16-byte aligned");
    cudaStream_t st = dc_cu_stream(stream);
    float *partial = reinterpret_cast<float *>(workspace);
    const int blocks = 2 * dc_sm_count();                          // <= 1024 (workspace bound)
    env_bwd_kernel<<<blocks, kThreadsE, 0, st>>>(d_out, out, ld, env, N, partial);
    DC_LAUNCH_OK();
    env_bwd_reduce_kernel<<<(kC * (kEnvIn + 1) + 31) / 32, 256, 0, st>>>(partial, blocks, dw_e, db_e);
    DC_LAUNCH_OK();
    return DC_OK;
}

extern "C" int dc_target_unit_fwd(const float *att, const float *ue, float *logits, int64_t N, dc_stream_t stream) {
    DC_REQUIRE(att && ue && logits && N > 0, DC_EINVAL, "dc_target_unit_fwd: bad arguments");
    DC_REQUIRE((((uintptr_t)att | (uintptr_t)ue) & 15) == 0, DC_EINVAL, "dc_target_unit_fwd: alignment");
    target_unit_fwd_kernel<<<(unsigned)((N + kWarps - 1) / kWarps), kThreadsE, 0, dc_cu_stream(stream)>>>(att, ue, logits, N);
    DC_LAUNCH_OK();
    return DC_OK;
}

extern "C" int dc_target_unit_q_fwd(const float *q, int ld_q, const float *const basics[6], float *logits, int64_t N,
                                    dc_stream_t stream) {
    DC_REQUIRE(q && basics && logits && N > 0 && ld_q >= 7 * kC && ld_q % 4 == 0, DC_EINVAL, "dc_target_unit_q_fwd: bad arguments");
    BasicPtrs bp;
    for (int g = 0; g < 6; ++g) {
        DC_REQUIRE(basics[g] && ((uintptr_t)basics[g] & 15) == 0, DC_EINVAL, "dc_target_unit_q_fwd: basic[%d] null / unaligned", g);
        bp.p[g] = basics[g];
    }
    DC_REQUIRE(((uintptr_t)q & 15) == 0, DC_EINVAL, "dc_target_unit_q_fwd: alignment");
    target_unit_q_fwd_kernel<<<(unsigned)((N + kWarps - 1) / kWarps), kThreadsE, 0, dc_cu_stream(stream)>>>(q, ld_q, bp, logits, N);
    DC_LAUNCH_OK();
    return DC_OK;
}

extern "C" int dc_target_unit_q_bwd(const float *dlogits, const float *const basics[6], float *s, int ld_s, int64_t N,
                                    dc_stream_t stream) {
    DC_REQUIRE(dlogits && basics && s && N > 0 && ld_s >= 7 * kC && ld_s % 4 == 0, DC_EINVAL, "dc_target_unit_q_bwd: bad arguments");
    BasicPtrs bp;
    for (int g = 0; g < 6; ++g) {
        DC_REQUIRE(basics[g] && ((uintptr_t)basics[g] & 15) == 0, DC_EINVAL, "dc_target_unit_q_bwd: basic[%d] null / unaligned", g);
        bp.p[g] = basics[g];
    }
    DC_REQUIRE(((uintptr_t)s & 15) == 0, DC_EINVAL, "dc_target_unit_q_bwd: alignment");
    target_unit_q_bwd_kernel<<<(unsigned)((N + kWarps - 1) / kWarps), kThreadsE, 0, dc_cu_stream(stream)>>>(dlogits, bp, s, ld_s, N);
    DC_LAUNCH_OK();
    return DC_OK;
}

extern "C" int dc_target_unit_bwd(const float *dlogits, const float *att, const float *ue, float *d_att, float *d_ue,
                                  int64_t N, dc_stream_t stream) {
    DC_REQUIRE(dlogits && att && ue && d_att && N > 0, DC_EINVAL, "dc_target_unit_bwd: bad arguments");
    DC_REQUIRE((((uintptr_t)att | (uintptr_t)ue | (uintptr_t)d_att | (uintptr_t)d_ue) & 15) == 0, DC_EINVAL,
               "dc_target_unit_bwd: alignment");
    target_unit_bwd_kernel<<<(unsigned)((N + kWarps - 1) / kWarps), kThreadsE, 0, dc_cu_stream(stream)>>>(dlogits, att, ue,
                                                                                                         d_att, d_ue, N);
    DC_LAUNCH_OK();
    return DC_OK;
}

