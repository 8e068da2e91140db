// U-Net glue kernels around the convolutions (all HBM-bound, channels-last):
//   * pg_conv_simt      exact-fp32 CUDA-core convolution (small channel counts, GPU-side check)
//   * pg_channel_stats  per-(clip, channel) {n, mean, M2} of a conv output (SIMT path; the
//                       tensor-core kernel produces the same records in its epilogue)
//   * pg_bn_finalize    combine partial records (Chan) -> per-channel scale/shift of the
//                       train-mode batch norm of model.py:81,83 (batch or per-clip statistics)
//   * pg_bn_act         y*scale+shift, ReLU / LeakyReLU(0.2) (model.py:80,82), written as the
//                       next layer's operand(s): fp32 or bf16 hi/lo planes, at a channel offset
//                       (this is how the skip concat of model.py:113 is materialised)
//   * pg_pack_weight    torch Conv/ConvT weight layouts (SURVEY 8a9) -> [tap][C_out][C_in] planes
//   * pg_transpose      [B][R][S] -> [B][S][R] (reference [B,C,T] layout <-> channels-last)
#include "common.cuh"
#include "conv_plan.h"

namespace pg {

// ---------------------------------------------------------------------------- SIMT conv
constexpr int kSimtPos = 4;

__global__ void __launch_bounds__(256)
conv_simt_kernel(const __grid_constant__ ConvPlan pl, const float* __restrict__ x, int in_rows, int in_ld,
                 const float* __restrict__ w, float* __restrict__ y) {
    const int co = blockIdx.x * blockDim.x + threadIdx.x;
    const int m0 = (blockIdx.y * blockDim.y + threadIdx.y) * kSimtPos;
    const int b = blockIdx.z / pl.OS, phase = blockIdx.z % pl.OS;
    const int l_phase = (pl.L_out - phase + pl.OS - 1) / pl.OS;
    if (co >= pl.C_out || m0 >= l_phase) return;
    float acc[kSimtPos];
#pragma unroll
    for (int i = 0; i < kSimtPos; ++i) acc[i] = 0.f;
    const float* xb = x + (size_t)b * in_rows * in_ld;
    for (int t = 0; t < pl.n_taps[phase]; ++t) {
        const ConvTap tp = pl.taps[phase][t];
        const float* wp = w + (size_t)tp.w_idx * pl.C_in * pl.C_out + co;
        const float* xr[kSimtPos];
        bool ok[kSimtPos];
#pragma unroll
        for (int i = 0; i < kSimtPos; ++i) {
            int row = (m0 + i + tp.d) * pl.IS + tp.parity;
            ok[i] = row >= 0 && row < pl.L_in && (m0 + i) < l_phase;
            xr[i] = xb + (size_t)(ok[i] ? row : 0) * in_ld;
        }
        for (int ci = 0; ci < pl.C_in; ++ci) {
            const float wv = __ldg(wp + (size_t)ci * pl.C_out);
#pragma unroll
            for (int i = 0; i < kSimtPos; ++i)
                if (ok[i]) acc[i] = fmaf(__ldg(xr[i] + ci), wv, acc[i]);
        }
    }
#pragma unroll
    for (int i = 0; i < kSimtPos; ++i) {
        if (m0 + i < l_phase) {
            int row = (m0 + i) * pl.OS + phase;
            y[((size_t)b * pl.out_rows + row) * pl.out_ld + co] = acc[i];
        }
    }
}

// ------------------------------------------------------------------------- channel stats
__global__ void channel_stats_kernel(const float* __restrict__ y, int L, int C, int rows, int ld, float4* __restrict__ stats) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (c >= C) return;
    const float* p = y + (size_t)b * rows * ld + c;
    float s = 0.f;
    for (int l = 0; l < L; ++l) s += p[(size_t)l * ld];
    const float mean = s / (float)L;
    float m2 = 0.f;
    for (int l = 0; l < L; ++l) { float d = p[(size_t)l * ld] - mean; m2 += d * d; }
    stats[(size_t)b * C + c] = make_float4((float)L, mean, m2, 0.f);
}

// --------------------------------------------------------------------------- BN finalize
// Pooled statistics of the records {n_i, mean_i, M2_i} in double, two passes: mean = sum n_i mean_i / N, then
// M2 = sum (M2_i + n_i (mean_i - mean)^2) -- Chan's combination without a division inside the loop.  (The first version merged
// the records one by one with two dependent fp64 divisions per record: 37 us per launch for the 64-128 records of a training
// batch, 0.22 ms per training step in six launches.)  The loads of a pass are independent, so they are issued in batches of 8.
__global__ void bn_finalize_kernel(const float4* __restrict__ stats, int B, int P, int C, int per_clip,
                                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                   float2* __restrict__ scale_shift, float2* __restrict__ mean_var) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int g = blockIdx.y;
    if (c >= C) return;
    const int b0 = per_clip ? g : 0, b1 = per_clip ? g + 1 : B;
    const float4* rec = stats + (size_t)b0 * P * C + c;
    const int R = (b1 - b0) * P;                            // records of channel c, C apart
    double n = 0.0, s = 0.0;
#pragma unroll 8
    for (int r = 0; r < R; ++r) {
        const float4 q = __ldg(rec + (size_t)r * C);
        if (q.x > 0.f) { n += (double)q.x; s += (double)q.x * (double)q.y; }
    }
    const double mean = n > 0.0 ? s / n : 0.0;
    double m2 = 0.0;
#pragma unroll 8
    for (int r = 0; r < R; ++r) {
        const float4 q = __ldg(rec + (size_t)r * C);
        if (q.x > 0.f) { const double d = (double)q.y - mean; m2 += (double)q.z + (double)q.x * d * d; }
    }
    const double var = n > 0.0 ? m2 / n : 0.0;
    const double sc = (gamma ? (double)gamma[c] : 1.0) / sqrt(var + (double)eps);
    const double sh = (beta ? (double)beta[c] : 0.0) - mean * sc;
    scale_shift[(size_t)g * C + c] = make_float2((float)sc, (float)sh);
    if (mean_var) mean_var[(size_t)g * C + c] = make_float2((float)mean, (float)var);
}

// ------------------------------------------------------------------------------- BN + act
// A thread owns a fixed group of four channels -- its (scale, shift) pairs are read once and live in registers (the first
// version re-read 32 B of them from L1/L2 for every 16 B of payload) -- and walks rows; four rows are loaded before any is
// stored so that 64 B per thread are in flight.
// RAGGED: clip b holds valid rows [0, L_b) only (clip_rows[b]); rows [L_b, L) of every destination are written as zeros
// and y is not read there.
template <bool RAGGED>
__global__ void __launch_bounds__(256)
bn_act_kernel(const float* __restrict__ y, int L, int C, int rows, int ld, const float2* __restrict__ scale_shift,
              int per_clip, ActDst d0, ActDst d1, const int* __restrict__ clip_rows) {
    const int c4 = C >> 2;
    const int b = blockIdx.y;
    const int L_b = RAGGED ? min(__ldg(clip_rows + b), L) : L;
    const int tpr = c4 < 256 ? c4 : 256;                    // threads per row (C >= 64 on this path, a multiple of 64)
    const int rpb = 256 / tpr;                              // rows per CTA pass
    const int q0 = threadIdx.x % tpr, r = threadIdx.x / tpr;
    const float2* ss = scale_shift ? scale_shift + (size_t)(per_clip ? b : 0) * C : nullptr;
    bool bad0 = false, bad1 = false;
    if (r < rpb) {
        for (int q = q0; q < c4; q += tpr) {                // one pass unless C > 1024
            const int c = q * 4;
            float4 s01 = make_float4(1.f, 0.f, 1.f, 0.f), s23 = s01;
            if (ss) {
                s01 = __ldg(reinterpret_cast<const float4*>(ss + c));
                s23 = __ldg(reinterpret_cast<const float4*>(ss + c + 2));
            }
            const float* yb = y + (size_t)b * rows * ld + c;
            const int step = gridDim.x * rpb;
            for (int l0 = blockIdx.x * rpb + r; l0 < L; l0 += 4 * step) {
                float4 v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int l = l0 + u * step;
                    if (l < L_b) v[u] = __ldcs(reinterpret_cast<const float4*>(yb + (size_t)l * ld));   // read once: evict first
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int l = l0 + u * step;
                    if (l >= L) break;
                    float4 w = v[u];
                    w.x = fmaf(w.x, s01.x, s01.y); w.y = fmaf(w.y, s01.z, s01.w);
                    w.z = fmaf(w.z, s23.x, s23.y); w.w = fmaf(w.w, s23.z, s23.w);
                    if (RAGGED && l >= L_b) w = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (d0.dtype) bad0 |= store_act4(d0, b, l, c, w);
                    if (d1.dtype) bad1 |= store_act4(d1, b, l, c, w);
                }
            }
        }
    }
    if (bad0 && d0.range_flag) atomicOr(d0.range_flag, 1);
    if (bad1 && d1.range_flag) atomicOr(d1.range_flag, 1);
}

// momentum update of the running buffers from the batch statistics (train-mode nn.BatchNorm side effect)
__global__ void bn_running_update_kernel(const float2* __restrict__ mean_var, float* __restrict__ running_mean,
                                         float* __restrict__ running_var, int C, float momentum, float unbias) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float2 mv = mean_var[c];
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mv.x;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (mv.y * unbias);
}

// eval-mode norm (nn.BatchNorm with running statistics): scale = gamma / sqrt(running_var + eps), shift = beta - mean*scale
__global__ void bn_from_running_kernel(const float* __restrict__ mean, const float* __restrict__ var, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, float eps, int C, int G, float2* __restrict__ scale_shift,
                                       float2* __restrict__ mean_var) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float sc = (gamma ? gamma[c] : 1.f) * rsqrtf(var[c] + eps);
    const float sh = (beta ? beta[c] : 0.f) - mean[c] * sc;
    for (int g = 0; g < G; ++g) {
        scale_shift[(size_t)g * C + c] = make_float2(sc, sh);
        if (mean_var) mean_var[(size_t)g * C + c] = make_float2(mean[c], var[c]);
    }
}

// --------------------------------------------------------------------------- weight pack
__global__ void pack_weight_kernel(const float* __restrict__ w, int transposed, int C_in, int C_out, int k,
                                   uint16_t* __restrict__ hi, uint16_t* __restrict__ lo, float* __restrict__ simt, int fmt) {
    const size_t total = (size_t)k * C_out * C_in;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int ci = (int)(i % C_in);
        const int co = (int)((i / C_in) % C_out);
        const int t = (int)(i / ((size_t)C_in * C_out));
        // Conv1d weight [C_out][C_in][k]; ConvTranspose1d weight [C_in][C_out][k]
        const float v = transposed ? w[((size_t)ci * C_out + co) * k + t] : w[((size_t)co * C_in + ci) * k + t];
        if (hi) {
            uint16_t h, l;
            split16(v, fmt, h, l);
            hi[i] = h;
            if (lo) lo[i] = l;
        }
        if (simt) simt[((size_t)t * C_in + ci) * C_out + co] = v;
    }
}

// ------------------------------------------------------------------------------ cast/split
__global__ void __launch_bounds__(256)
cast_split_kernel(const float* __restrict__ src, size_t n4, uint16_t* __restrict__ hi, uint16_t* __restrict__ lo, int fmt, int* __restrict__ range_flag) {
    bool bad = false;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        const float4 v = reinterpret_cast<const float4*>(src)[i];
        if (fmt == PG_FMT_F16) bad |= !f16_fits(v.x) || !f16_fits(v.y) || !f16_fits(v.z) || !f16_fits(v.w);
        __align__(8) uint16_t h[4], l[4];
        split16(v.x, fmt, h[0], l[0]); split16(v.y, fmt, h[1], l[1]); split16(v.z, fmt, h[2], l[2]); split16(v.w, fmt, h[3], l[3]);
        reinterpret_cast<uint2*>(hi)[i] = *reinterpret_cast<uint2*>(h);
        if (lo) reinterpret_cast<uint2*>(lo)[i] = *reinterpret_cast<uint2*>(l);
    }
    if (bad && range_flag) atomicOr(range_flag, 1);
}

// ----------------------------------------------------------------------------- transpose
__global__ void transpose_kernel(const float* __restrict__ src, int R, int S, long long src_batch_stride,
                                 float* __restrict__ dst, uint16_t* __restrict__ hi, uint16_t* __restrict__ lo,
                                 long long dst_batch_stride, int dst_ld, int fmt, int* __restrict__ range_flag) {
    __shared__ float tile[32][33];
    bool bad = false;
    const int b = blockIdx.z;
    const int s0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const float* sp = src + (size_t)b * src_batch_stride;
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        int r = r0 + j, s = s0 + threadIdx.x;
        tile[j][threadIdx.x] = (r < R && s < S) ? sp[(size_t)r * S + s] : 0.f;
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        int s = s0 + j, r = r0 + threadIdx.x;
        if (s < S && r < R) {
            const float v = tile[threadIdx.x][j];
            const size_t o = (size_t)b * dst_batch_stride + (size_t)s * dst_ld + r;
            if (dst) dst[o] = v;
            if (hi) {
                uint16_t h, l;
                split16(v, fmt, h, l);
                if (fmt == PG_FMT_F16) bad |= !f16_fits(v);
                hi[o] = h;
                if (lo) lo[o] = l;
            }
        }
    }
    if (bad && range_flag) atomicOr(range_flag, 1);
}

}  // namespace pg

using namespace pg;

extern "C" int pg_conv_simt(const pg_conv_desc* d, const float* x, const float* w_simt, float* y, pg_stream stream) {
    PG_REQUIRE(d && x && w_simt && y, "pg_conv_simt: null pointer");
    ConvPlan pl;
    pg_conv_desc dd = *d;
    dd.taps_per_group = 1;
    int rc = conv_plan_build(&dd, &pl);
    if (rc != PG_OK) return rc;
    const int bx = pl.C_out >= 64 ? 64 : 32;
    dim3 block(bx, 256 / bx);
    const int l_max = (pl.L_out + pl.OS - 1) / pl.OS;
    dim3 grid((pl.C_out + bx - 1) / bx, (l_max + block.y * kSimtPos - 1) / (block.y * kSimtPos), pl.B * pl.OS);
    PG_REQUIRE(grid.z <= 65535 && grid.y <= 65535, "pg_conv_simt: grid too large");
    conv_simt_kernel<<<grid, block, 0, reinterpret_cast<cudaStream_t>(stream)>>>(pl, x, d->in_rows, d->in_ld, w_simt, y);
    return check_launch("conv_simt_kernel");
}

extern "C" int pg_channel_stats(const float* y, int B, int L, int C, int rows, int ld, float* stats, pg_stream stream) {
    PG_REQUIRE(y && stats && B > 0 && L > 0 && C > 0 && B <= 65535, "pg_channel_stats: bad arguments");
    dim3 grid((C + 127) / 128, B);
    channel_stats_kernel<<<grid, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(y, L, C, rows, ld, reinterpret_cast<float4*>(stats));
    return check_launch("channel_stats_kernel");
}

extern "C" int pg_bn_finalize(const float* stats, int B, int P, int C, int per_clip, const float* gamma, const float* beta,
                              float eps, float* scale_shift, float* mean_var, pg_stream stream) {
    PG_REQUIRE(stats && scale_shift && B > 0 && P > 0 && C > 0 && B <= 65535, "pg_bn_finalize: bad arguments");
    dim3 grid((C + 127) / 128, per_clip ? B : 1);
    bn_finalize_kernel<<<grid, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const float4*>(stats), B, P, C, per_clip, gamma, beta, eps,
        reinterpret_cast<float2*>(scale_shift), reinterpret_cast<float2*>(mean_var));
    return check_launch("bn_finalize_kernel");
}

static int bn_act_launch(const float* y, int B, int L, int C, int rows, int ld, const float* scale_shift, int per_clip,
                         const pg_act_dst* dst0, const pg_act_dst* dst1, const int* clip_rows, pg_stream stream) {
    PG_REQUIRE(y && B > 0 && L > 0 && C > 0 && B <= 65535, "pg_bn_act: bad arguments");
    PG_REQUIRE(C % 4 == 0 && ld % 4 == 0, "pg_bn_act: channel count and pitch must be multiples of 4");
    ActDst d0, d1;
    int rc;
    if ((rc = to_act_dst(dst0, C, &d0, "pg_bn_act", "dst0")) != PG_OK) return rc;
    if ((rc = to_act_dst(dst1, C, &d1, "pg_bn_act", "dst1")) != PG_OK) return rc;
    // ~16 CTAs per SM in total: enough to fill the machine, few enough that a thread's (scale, shift) registers pay off
    const int c4 = C / 4, rpb = 256 / (c4 < 256 ? c4 : 256);
    int gx = (L + rpb - 1) / rpb;
    const int want = (148 * 16 + B - 1) / B;
    if (gx > want) gx = want;
    if (gx < 1) gx = 1;
    (clip_rows ? bn_act_kernel<true> : bn_act_kernel<false>)<<<dim3(gx, B), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        y, L, C, rows, ld, reinterpret_cast<const float2*>(scale_shift), per_clip, d0, d1, clip_rows);
    return check_launch("bn_act_kernel");
}

extern "C" int pg_bn_act(const float* y, int B, int L, int C, int rows, int ld, const float* scale_shift, int per_clip,
                         const pg_act_dst* dst0, const pg_act_dst* dst1, pg_stream stream) {
    return bn_act_launch(y, B, L, C, rows, ld, scale_shift, per_clip, dst0, dst1, nullptr, stream);
}

extern "C" int pg_bn_act_ragged(const float* y, int B, int L, int C, int rows, int ld, const float* scale_shift, int per_clip,
                                const pg_act_dst* dst0, const pg_act_dst* dst1, const int* clip_rows, pg_stream stream) {
    PG_REQUIRE(clip_rows, "pg_bn_act_ragged: null per-clip row table");
    return bn_act_launch(y, B, L, C, rows, ld, scale_shift, per_clip, dst0, dst1, clip_rows, stream);
}

extern "C" int pg_pack_weight(const float* w, int kind, int C_in, int C_out, int k, uint16_t* w_hi, uint16_t* w_lo,
                              float* w_simt, int fmt, pg_stream stream) {
    PG_REQUIRE(w && (w_hi || w_simt) && C_in > 0 && C_out > 0 && k > 0, "pg_pack_weight: bad arguments");
    PG_REQUIRE(fmt == PG_FMT_BF16 || fmt == PG_FMT_F16, "pg_pack_weight: bad operand format %d", fmt);
    const size_t total = (size_t)k * C_out * C_in;
    int gx = (int)((total + 255) / 256); if (gx > 148 * 16) gx = 148 * 16;
    pack_weight_kernel<<<gx, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        w, kind == PG_CONV_TRANSPOSE, C_in, C_out, k, w_hi, w_lo, w_simt, fmt);
    return check_launch("pack_weight_kernel");
}

extern "C" int pg_bn_running_update(const float* mean_var, float* running_mean, float* running_var, int C, float momentum,
                                    float unbias, pg_stream stream) {
    PG_REQUIRE(mean_var && running_mean && running_var && C > 0, "pg_bn_running_update: bad arguments");
    bn_running_update_kernel<<<(C + 255) / 256, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const float2*>(mean_var), running_mean, running_var, C, momentum, unbias);
    return check_launch("bn_running_update_kernel");
}

extern "C" int pg_bn_from_running(const float* running_mean, const float* running_var, const float* gamma, const float* beta,
                                  float eps, int C, int G, float* scale_shift, float* mean_var, pg_stream stream) {
    PG_REQUIRE(running_mean && running_var && scale_shift && C > 0 && G > 0, "pg_bn_from_running: bad arguments");
    bn_from_running_kernel<<<(C + 127) / 128, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        running_mean, running_var, gamma, beta, eps, C, G, reinterpret_cast<float2*>(scale_shift), reinterpret_cast<float2*>(mean_var));
    return check_launch("bn_from_running_kernel");
}

extern "C" int pg_cast_split(const float* src, int64_t n, uint16_t* hi, uint16_t* lo, int fmt, int* range_flag, pg_stream stream) {
    PG_REQUIRE(src && hi && n > 0 && n % 4 == 0, "pg_cast_split: bad arguments (n must be a multiple of 4)");
    PG_REQUIRE(fmt == PG_FMT_BF16 || fmt == PG_FMT_F16, "pg_cast_split: bad operand format %d", fmt);
    const size_t n4 = (size_t)n / 4;
    int gx = (int)((n4 + 255) / 256); if (gx > 148 * 32) gx = 148 * 32;
    cast_split_kernel<<<gx, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, n4, hi, lo, fmt, range_flag);
    return check_launch("cast_split_kernel");
}

extern "C" int pg_transpose(const float* src, int B, int R, int S, int64_t src_batch_stride, float* dst, uint16_t* dst_hi,
                            uint16_t* dst_lo, int64_t dst_batch_stride, int dst_ld, int fmt, int* range_flag, pg_stream stream) {
    PG_REQUIRE(src && (dst || dst_hi) && B > 0 && R > 0 && S > 0 && B <= 65535 && dst_ld >= R, "pg_transpose: bad arguments");
    dim3 grid((S + 31) / 32, (R + 31) / 32, B);
    transpose_kernel<<<grid, dim3(32, 8), 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        src, R, S, src_batch_stride, dst, dst_hi, dst_lo, dst_batch_stride, dst_ld, fmt, range_flag);
    return check_launch("transpose_kernel");
}
