// STFT front end and ISTFT back end (hand-written, sm_100a).
//
// Reference path replaced:
//   * librosa.stft call + DC-row drop + re/im split   preproc_mdb.py:84-97 (call at :93)
//   * abs / log1p / angle                             data.py:39-47
//   * expm1(mag) * exp(j*phase)                       demo.py:39, train.py:83
//   * zero DC row + librosa.istft + peak normalise    utils.py:34-42
//
// Both kernels keep everything between the HBM read and the HBM write on chip (frame transforms:
// stft_core.cuh, checked on the host by fft_selftest2.cpp):
//   STFT : a frame is owned by n_fft/32 threads (one warp at n_fft 1024): windowed samples straight from
//          global memory (float2, coalesced; the 75 % overlap between frames is served by L1/L2; reflect
//          padding resolved on the edge frames only) -> n_fft/2-point complex Stockham FFT in a private
//          shared buffer, passes separated by __syncwarp -> Hermitian post-processing (fused with the last
//          radix-2 pass at n_fft 1024) -> log1p|X| (and atan2 only when the phase plane is requested)
//          -> fp32 frame-major [B][T][C] + the 16-bit hi/lo operand planes the first convolution consumes.
//          A CTA (8 warps) loops over 32+ frames so the twiddle/window tables are built once per CTA.
//   ISTFT: a CTA walks a run of consecutive frames of one clip, 256/TG frames per iteration into a
//          two-generation ring of windowed frames in shared memory; after each iteration it emits the
//          output hop-blocks whose four covering frames are complete (GATHER overlap-add, window-sum-square
//          normalisation, float4 stores).  Only 3 halo frames are recomputed per ~90-frame run (the first
//          version recomputed 3 per 13).  No atomics on the output; the per-clip peak (utils.py:42) is one
//          atomicMax per warp on a scalar.
// hop must be n_fft/4 (true for every configuration of the reference and of BASELINE.json).
#include "common.cuh"
#include "stft_core.cuh"

namespace pg {
using namespace pgfft;

constexpr int kStftThreads = 256;

template <int NC> struct FrameCfg {
    static constexpr int TG = NC / 16;                      // threads per frame
    static constexpr int FC = kStftThreads / TG;            // frames in flight per CTA
    static constexpr int NFFT = 2 * NC;
    static constexpr int HOP = NFFT / 4;
    static constexpr int PL = padded_len2(NC);              // float2 elements of one frame buffer
    static constexpr size_t smem_stft() { return sizeof(float2) * (Radix<NC, false>::TOTAL + NC + (size_t)FC * PL); }
    static constexpr int RING = FC + 3;                     // windowed frames kept on chip: this iteration's + 3 of the last
    static constexpr size_t smem_istft() { return sizeof(float2) * (Radix<NC, true>::TOTAL + NC + (size_t)RING * PL + NC /*scale/shift table*/) + sizeof(float) * HOP; }
};

// the threads of one frame: lanes of a warp (TG <= 32) or two warps on a named barrier (TG = 64)
template <int TG> struct FrameSync {
    int slot;
    __device__ __forceinline__ void operator()() const {
        if (TG <= 32) __syncwarp();
        else asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "r"(TG) : "memory");
    }
};

// log1p|X| with two special-function instructions and no selects: sqrt.approx(0) = 0 needs no guard, and 1 + |X| >= 1 is
// never subnormal, so lg2.approx needs none of the scaling __logf wraps around it (2 ulp each; the parity bound is 1e-4).
__device__ __forceinline__ float fast_log1p_mag(float re, float im) {
    const float m2 = fmaf(re, re, im * im);
    float mag, l2;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(mag) : "f"(m2));
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2) : "f"(1.0f + mag));
    return l2 * 0.693147180559945f;
}

// ------------------------------------------------------------------------------------ STFT
// FAST = 0: every output selected at run time.  FAST = 1 / 2: the inference path (log-magnitude fp32 plane +
// bf16 / fp16 hi,lo operand planes, no phase plane) with the selection compiled in.
// LAYOUT kRagged: clip b is its first n_b = clip_samples[b] samples zero-padded to N_b = (T_b - 1) * hop, T_b =
// clip_frames[b] <= T: samples >= n_b are never read, reflect padding happens at N_b, and frames >= T_b are transforms of
// zeros, so every plane holds exact zeros there.
// LAYOUT kPacked: the same clip program, clip b read from wave[o_b, o_b + n_b) of a flat buffer of n_wave samples,
// o_b = clip_offsets[b], n_b = clip_offsets[b + 1] - o_b (both clamped to [0, n_wave], n_b to [0, N]).  Whether a clip
// takes the float2 loads depends on its own offset; an interior frame of an odd-offset clip takes two unchecked scalar
// loads instead, so only edge frames pay for the reflect and bounds checks.
enum { kFixed = 0, kRagged = 1, kPacked = 2 };
template <int NC, int FAST, int LAYOUT>
__global__ void __launch_bounds__(kStftThreads, 3)          // 3 CTAs per SM (<= 85 registers): the kernel is issue/latency-bound
stft_kernel(const float* __restrict__ wave, int N, int T, const float2* __restrict__ tw_g, int mode,
            float* __restrict__ out_a, float* __restrict__ out_b,
            uint16_t* __restrict__ op_hi, uint16_t* __restrict__ op_lo,
            long long op_batch_stride, int op_fmt, int frames_per_cta, const float* __restrict__ proj_mag,
            float std_mean, float std_inv, const int* __restrict__ clip_samples, const int* __restrict__ clip_frames,
            const long long* __restrict__ clip_offsets, long long n_wave) {
    using Cfg = FrameCfg<NC>;
    using R = Radix<NC, false>;
    extern __shared__ float2 smem2[];
    cpx* tabs = reinterpret_cast<cpx*>(smem2);              // compact twiddle tables
    cpx* win = tabs + R::TOTAL;                             // (w[2m], w[2m+1]) / 2, periodic Hann
    cpx* bufs = win + NC;                                   // FC frame buffers

    const int tid = threadIdx.x;
    const cpx* twc = reinterpret_cast<const cpx*>(tw_g);
    for (int e = tid; e < R::TOTAL; e += kStftThreads) tabs[e] = table_entry<NC, false>(twc, e);
    for (int m = tid; m < NC; m += kStftThreads)            // Hann(n) = 0.5 - 0.5 cos(2 pi n / n_fft); the 1/2 of the
        win[m] = {0.25f - 0.25f * tw_g[2 * m].x, 0.25f - 0.25f * tw_g[2 * m + 1].x};   // post-processing folded in
    __syncthreads();

    constexpr bool RAGGED = LAYOUT != kFixed;               // per-clip frame counts (ragged and packed)
    const int b = blockIdx.y;
    // packed: the clip's offset o_b is re-read from shared memory at every frame; held in registers across the frame
    // program it pushes the n_fft 2048 / 1024 variants past the 80 registers of 3 CTAs per SM
    __shared__ long long clip_base;
    int n_b = N;
    if (LAYOUT == kPacked) {
        const long long o_b = min(max(__ldg(clip_offsets + b), 0ll), n_wave);
        const long long e_b = min(max(__ldg(clip_offsets + b + 1), o_b), n_wave);
        n_b = (int)min(e_b - o_b, (long long)N);            // samples read from the clip
        if (tid == 0) clip_base = o_b;
        __syncthreads();
    } else if (LAYOUT == kRagged) {
        n_b = min(__ldg(clip_samples + b), N);
    }
    const int T_b = RAGGED ? min(__ldg(clip_frames + b), T) : T;
    const int N_b = RAGGED ? (T_b - 1) * Cfg::HOP : N;      // where the reflect padding happens
    const int slot = tid / Cfg::TG, t = tid % Cfg::TG;
    cpx* s = bufs + slot * Cfg::PL;
    const FrameSync<Cfg::TG> sync{slot};
    const float* w_row = wave + (size_t)b * N;
    const bool aligned_row = (N & 1) == 0 && (reinterpret_cast<uintptr_t>(wave) & 7) == 0;   // float2 loads
    const int f_begin = blockIdx.x * frames_per_cta;

    for (int f0 = f_begin; f0 < f_begin + frames_per_cta && f0 < T; f0 += Cfg::FC) {
        const float* w = LAYOUT == kPacked ? wave + clip_base : w_row;
        const bool aligned = LAYOUT == kPacked ? (reinterpret_cast<uintptr_t>(w) & 7) == 0 : aligned_row;   // per clip
        const int frame = f0 + slot;
        const bool live = frame < T;
        // padded sample p <-> wave index p - n_fft/2, reflected at both ends (librosa center=True)
        const int p0 = frame * Cfg::HOP - NC;
        cpx v[16];
        if (live && (LAYOUT == kPacked || aligned) && p0 >= 0 && p0 + Cfg::NFFT <= n_b) {
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const int m = t + r * Cfg::TG;
                float2 xv;
                if (LAYOUT != kPacked || aligned) xv = __ldg(reinterpret_cast<const float2*>(w + p0) + m);
                else xv = make_float2(__ldg(w + p0 + 2 * m), __ldg(w + p0 + 2 * m + 1));   // interior frame, odd clip offset
                const cpx wv = win[m];
                v[r] = {xv.x * wv.x, xv.y * wv.y};
            }
        } else if (live && (!RAGGED || frame < T_b)) {
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const int m = t + r * Cfg::TG;
                int n0 = p0 + 2 * m, n1 = n0 + 1;
                if (n0 < 0) n0 = -n0;
                if (n0 >= N_b) n0 = 2 * (N_b - 1) - n0;
                if (n1 < 0) n1 = -n1;
                if (n1 >= N_b) n1 = 2 * (N_b - 1) - n1;
                const float x0 = (n0 >= 0 && n0 < n_b) ? __ldg(w + n0) : 0.f;
                const float x1 = (n1 >= 0 && n1 < n_b) ? __ldg(w + n1) : 0.f;
                const cpx wv = win[m];
                v[r] = {x0 * wv.x, x1 * wv.y};
            }
        } else {
#pragma unroll
            for (int r = 0; r < 16; ++r) v[r] = {0.f, 0.f};
        }
        fwd_phase0<NC>(s, t, v);
        sync();
        fwd_phase1<NC>(s, t, tabs, sync);
        sync();

        const size_t row = ((size_t)b * T + frame) * NC;
        const size_t orow = (size_t)b * op_batch_stride + (size_t)frame * NC;
        auto emit = [&](int bin, cpx x) {
            if (FAST) {
                const float a = fast_log1p_mag(x.x, x.y);
                uint16_t hi, lo;
                split16(a, FAST == 2 ? PG_FMT_F16 : PG_FMT_BF16, hi, lo);
                out_a[row + bin - 1] = a;
                op_hi[orow + bin - 1] = hi;
                op_lo[orow + bin - 1] = lo;
                return;
            }
            if (bin == NC) x.y = 0.f;                       // the Nyquist bin of a real signal is real
            float a, ph = 0.f;
            if (mode == PG_STFT_PROJECT) {
                // Griffin-Lim projection (utils.py:119-124): keep the phase of X, impose the magnitude proj_mag;
                // X / |X| directly instead of exp(j * angle(X)); angle(0) = 0 -> unit vector (1, 0)
                const float m2 = fmaf(x.x, x.x, x.y * x.y);
                const float inv = m2 > 0.f ? rsqrtf(m2) : 0.f;
                const float g = __ldg(proj_mag + row + bin - 1);
                a = m2 > 0.f ? g * x.x * inv : g;
                ph = g * x.y * inv;
            } else if (mode == PG_STFT_LOGMAG || mode == PG_STFT_PAIRS) {
                if (mode == PG_STFT_PAIRS) {                // global standardisation of (re, im): preproc_mdb.py:182
                    x.x = (x.x - std_mean) * std_inv;
                    x.y = (x.y - std_mean) * std_inv;
                }
                a = fast_log1p_mag(x.x, x.y);
                if (out_b) ph = atan2f(x.y, x.x);
            } else {
                a = x.x; ph = x.y;
            }
            if (out_a) out_a[row + bin - 1] = a;
            if (out_b) out_b[row + bin - 1] = ph;
            if (op_hi) {
                uint16_t hi, lo;
                split16(a, op_fmt, hi, lo);
                op_hi[orow + bin - 1] = hi;
                if (op_lo) op_lo[orow + bin - 1] = lo;
            }
        };
        if (NC == 512) {
            if (live) fwd_fused_last_512(s, t, tabs, emit);
        } else {
            fwd_phase2_unfused<NC>(s, t, tabs, sync);
            sync();
            if (live) fwd_post_generic<NC>(s, t, tabs, emit);
        }
        sync();                                             // the buffer is rewritten by the next frame
    }
}

// ----------------------------------------------------------------------------------- ISTFT
__device__ __forceinline__ cpx spec_value(float a, float p, int mode) {
    if (mode == PG_SPEC_CARTESIAN) return {a, p};
    float mag = a;
    if (mode == PG_SPEC_POLAR_LOG) mag = __expf(a) - 1.0f;    // expm1 (demo.py:39): a = log1p|X| >= 0; the absolute error 1e-7 of
                                                            // the plain form is invisible next to the bins that carry the signal
    // sin.approx / cos.approx reduce their argument themselves (multiply by 1/2pi, hardware wrap): the phase of a
    // normalised network output is a few radians, where this costs < 1e-6 absolute -- no Cody-Waite step needed
    return {mag * __cosf(p), mag * __sinf(p)};
}

// FAST: mode == PG_SPEC_POLAR_LOG with a phase plane (the inference path), selection compiled in.
// RAGGED: clip b has T_b = clip_frames[b] <= T frames and n_b = clip_samples[b] <= (T_b - 1) * hop samples: frames >= T_b
// are never read, the clip ends (window sum of squares, trim) at (T_b - 1) * hop as if it had T_b frames, peak and
// non-finite flags cover [0, (T_b - 1) * hop), and samples [n_b, (T - 1) * hop) are written as zeros.
template <int NC, bool FAST, bool RAGGED>
__global__ void __launch_bounds__(kStftThreads)
istft_kernel(const float* __restrict__ in_a, const float* __restrict__ in_b, int mode, int T,
             const float2* __restrict__ tw_g, float* __restrict__ wave,
             unsigned* __restrict__ peak_bits, int* __restrict__ nonfinite, int blocks_per_cta,
             const float2* __restrict__ b_ss, int b_ss_stride, const int* __restrict__ clip_frames,
             const int* __restrict__ clip_samples) {
    using Cfg = FrameCfg<NC>;
    using R = Radix<NC, true>;
    constexpr int FC = Cfg::FC, HOP = Cfg::HOP;
    extern __shared__ float2 smem2[];
    float* wss_full = reinterpret_cast<float*>(smem2);      // [HOP] 1 / sum of w^2 over the 4 covering frames (16-byte aligned)
    cpx* tabs = reinterpret_cast<cpx*>(wss_full + HOP);
    cpx* win = tabs + R::TOTAL;                             // synthesis Hann, (w[2m], w[2m+1])
    cpx* ring = win + NC;                                   // RING = FC + 3 windowed frames, slot = (frame - F0) mod RING
    // optional affine map of the second plane, b <- b*scale + shift per (clip, bin): the train-mode norm that ends the
    // U-Net (model.py:83,91) applied here, so the last layer's raw output is read once and never re-written
    float2* ss_tab = reinterpret_cast<float2*>(ring + (size_t)Cfg::RING * Cfg::PL);   // [NC], only when b_ss

    const int tid = threadIdx.x;
    const cpx* twc = reinterpret_cast<const cpx*>(tw_g);
    for (int e = tid; e < R::TOTAL; e += kStftThreads) tabs[e] = table_entry<NC, true>(twc, e);
    for (int m = tid; m < NC; m += kStftThreads) win[m] = {0.5f - 0.5f * tw_g[2 * m].x, 0.5f - 0.5f * tw_g[2 * m + 1].x};
    for (int i = tid; i < HOP; i += kStftThreads) {
        float acc = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) { const float wn = 0.5f - 0.5f * tw_g[q * HOP + i].x; acc += wn * wn; }
        wss_full[i] = acc > 1.17549435e-38f ? 1.0f / acc : 1.0f;   // stored as the reciprocal: the overlap-add multiplies
    }
    const int b = blockIdx.y;
    const int T_b = RAGGED ? min(__ldg(clip_frames + b), T) : T;   // table entries beyond the buffer are clamped to it
    const int n_b = RAGGED ? __ldg(clip_samples + b) : 0;
    if (b_ss) for (int m = tid; m < NC; m += kStftThreads) ss_tab[m] = __ldg(b_ss + (size_t)b * b_ss_stride + m);
    __syncthreads();

    const int J0 = blockIdx.x * blocks_per_cta;             // output hop-blocks [J0, J1) of this CTA
    const int J1 = min(J0 + blocks_per_cta, T - 1);
    const int F0 = J0 - 1;                                  // first frame needed
    const int n_iter = (J1 - J0 + 3 + FC - 1) / FC;
    const int slot = tid / Cfg::TG, t = tid % Cfg::TG;
    const FrameSync<Cfg::TG> sync{slot};
    const float scale = 0.5f / NC;
    float* wv = wave + (size_t)b * (size_t)(T - 1) * HOP;
    float pk = 0.f;
    bool bad = false;

    // the 16 (a, b) input pairs of this thread's frame are fetched one iteration ahead of their use, so the
    // global-load latency hides behind the previous frame's transform and overlap-add
    float ra[16], rb[16];
    auto is_live = [&](int frame) { return frame >= 0 && frame < T_b && frame <= J1 + 1; };
    auto fetch = [&](int frame) {
        if (!is_live(frame)) return;
        const size_t row = ((size_t)b * T + frame) * NC;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const size_t idx = row + inv_bin<NC>(t, j) - 1;
            ra[j] = __ldg(in_a + idx);
            rb[j] = (FAST || in_b) ? __ldg(in_b + idx) : 0.f;
        }
    };
    fetch(F0 + slot);

    for (int it = 0; it < n_iter; ++it) {
        const int F = F0 + it * FC;
        const int frame = F + slot;
        const bool live = is_live(frame);
        cpx* s = ring + (size_t)((frame - F0) % Cfg::RING) * Cfg::PL;
        if (live) {
            cpx x[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float pb = rb[j];
                if (b_ss) { const float2 ss = ss_tab[inv_bin<NC>(t, j) - 1]; pb = fmaf(pb, ss.x, ss.y); }
                x[j] = spec_value(ra[j], pb, FAST ? (int)PG_SPEC_POLAR_LOG : mode);
            }
            if (NC == 512) inv_fused_first_512(s, t, tabs, scale, x);
            else inv_pre_generic<NC>(s, t, tabs, scale, x);
        }
        if (it + 1 < n_iter) fetch(frame + FC);
        sync();
        inv_passes<NC>(s, t, tabs, win, sync);              // dead frames run on stale data; never read below
        __syncthreads();

        // output hop-block jb (trimmed coordinates) is covered by frames jb-1 .. jb+2; within frame
        // jb-1+q its samples sit at offset (3-q)*hop + i
        const int lo = max(J0, F - 2), hi = min(J1, F + FC - 2);
        for (int u = tid; u < (hi - lo) * (HOP / 4); u += kStftThreads) {
            const int jb = lo + u / (HOP / 4), i = (u % (HOP / 4)) * 4;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), wss;
            const bool interior = jb >= 1 && jb + 2 < T_b;
            if (interior) wss = *reinterpret_cast<const float4*>(wss_full + i);   // reciprocal of the window sum of squares
            else wss = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int fr = jb - 1 + q;
                if (fr < 0 || fr >= T_b) continue;
                const cpx* fb = ring + (size_t)((fr - F0) % Cfg::RING) * Cfg::PL;
                const int m = ((3 - q) * HOP + i) >> 1;
                const cpx z0 = fb[pad2(m)], z1 = fb[pad2(m + 1)];
                acc.x += z0.x; acc.y += z0.y; acc.z += z1.x; acc.w += z1.y;
                if (!interior) {
                    const cpx w0 = win[m], w1 = win[m + 1];
                    wss.x += w0.x * w0.x; wss.y += w0.y * w0.y; wss.z += w1.x * w1.x; wss.w += w1.y * w1.y;
                }
            }
            if (!interior) {                                // edge blocks (two per clip): divide where > tiny (librosa)
                wss.x = wss.x > 1.17549435e-38f ? 1.0f / wss.x : 1.0f; wss.y = wss.y > 1.17549435e-38f ? 1.0f / wss.y : 1.0f;
                wss.z = wss.z > 1.17549435e-38f ? 1.0f / wss.z : 1.0f; wss.w = wss.w > 1.17549435e-38f ? 1.0f / wss.w : 1.0f;
            }
            float4 y;
            y.x = acc.x * wss.x; y.y = acc.y * wss.y; y.z = acc.z * wss.z; y.w = acc.w * wss.w;
            if (RAGGED && jb >= T_b - 1) y = make_float4(0.f, 0.f, 0.f, 0.f);   // past the clip's padded end
            const float mx = fmaxf(fmaxf(fabsf(y.x), fabsf(y.y)), fmaxf(fabsf(y.z), fabsf(y.w)));
            if (!(mx <= 3.402823466e+38f) || y.x != y.x || y.y != y.y || y.z != y.z || y.w != y.w) bad = true;
            pk = fmaxf(pk, mx);
            if (RAGGED) {                                   // the zero padding of the clip is not part of its output
                const int n = jb * HOP + i;
                if (n >= n_b) y.x = 0.f;
                if (n + 1 >= n_b) y.y = 0.f;
                if (n + 2 >= n_b) y.z = 0.f;
                if (n + 3 >= n_b) y.w = 0.f;
            }
            *reinterpret_cast<float4*>(wv + (size_t)jb * HOP + i) = y;
        }
        __syncthreads();                                    // the next iteration overwrites the oldest FC frames
    }
    if (peak_bits) {
#pragma unroll
        for (int o = 16; o; o >>= 1) pk = fmaxf(pk, __shfl_xor_sync(0xffffffffu, pk, o));
        if ((tid & 31) == 0 && pk > 0.f) atomicMax(peak_bits + b, __float_as_uint(pk));
    }
    if (nonfinite && bad) atomicOr(nonfinite + b, 1);
}

__global__ void peak_normalize_kernel(float* __restrict__ wave, const unsigned* __restrict__ peak_bits, int n) {
    const int b = blockIdx.y;
    float pk = __uint_as_float(peak_bits[b]);
    if (!(pk >= 1.17549435e-38f)) return;                   // librosa.util.normalize: tiny -> unchanged
    float inv = 1.0f / pk;
    float* w = wave + (size_t)b * n;
    if ((n & 3) == 0) {
        float4* w4 = reinterpret_cast<float4*>(w);
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n / 4; i += gridDim.x * blockDim.x) {
            float4 v = w4[i];
            v.x *= inv; v.y *= inv; v.z *= inv; v.w *= inv;
            w4[i] = v;
        }
    } else {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) w[i] = w[i] * inv;
    }
}

// Packs the ISTFT's padded plane: dst[o_b + i] = src[b][i] / peak_b for i < n_b (the librosa.util.normalize rule of
// peak_normalize_kernel, so the result is bit-identical to normalising in place and slicing), a plain copy when
// peak_bits is NULL or the peak is tiny.  Offsets are clamped to [0, n_dst] and n_b to [0, src_pitch], so a bad table
// writes inside dst and reads inside row b only.  float4 stores once dst is 16-byte aligned, float4 loads too when
// src sits at the same alignment; else scalar loads.
__global__ void __launch_bounds__(256)
peak_normalize_packed_kernel(const float* __restrict__ src, long long src_pitch, const unsigned* __restrict__ peak_bits,
                             const long long* __restrict__ clip_offsets, float* __restrict__ dst, long long n_dst) {
    const int b = blockIdx.y;
    const long long o = min(max(__ldg(clip_offsets + b), 0ll), n_dst);
    const long long e = min(max(__ldg(clip_offsets + b + 1), o), n_dst);
    const long long n = min(e - o, src_pitch);
    const float pk = peak_bits ? __uint_as_float(__ldg(peak_bits + b)) : 0.f;
    const bool scale = pk >= 1.17549435e-38f;
    const float inv = scale ? 1.0f / pk : 1.0f;
    const float* s = src + (size_t)b * src_pitch;
    float* d = dst + o;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    // head: scalar up to the first 16-byte aligned dst address
    const long long head = min((long long)((16 - (reinterpret_cast<uintptr_t>(d) & 15)) & 15) / 4, n);
    for (long long i = i0; i < head; i += stride) d[i] = scale ? s[i] * inv : s[i];
    const long long n4 = (n - head) / 4;
    float4* d4 = reinterpret_cast<float4*>(d + head);
    const float* sh = s + head;
    if ((reinterpret_cast<uintptr_t>(sh) & 15) == 0) {
        const float4* s4 = reinterpret_cast<const float4*>(sh);
        for (long long i = i0; i < n4; i += stride) {
            float4 v = __ldg(s4 + i);
            if (scale) { v.x *= inv; v.y *= inv; v.z *= inv; v.w *= inv; }
            d4[i] = v;
        }
    } else {
        for (long long i = i0; i < n4; i += stride) {
            float4 v = make_float4(__ldg(sh + 4 * i), __ldg(sh + 4 * i + 1), __ldg(sh + 4 * i + 2), __ldg(sh + 4 * i + 3));
            if (scale) { v.x *= inv; v.y *= inv; v.z *= inv; v.w *= inv; }
            d4[i] = v;
        }
    }
    for (long long i = head + 4 * n4 + i0; i < n; i += stride) d[i] = scale ? s[i] * inv : s[i];
}

// Long-form stitching (BASELINE.json config 4): windows of `win` samples every `step` samples (step >= win/2, so at
// most two overlap) are cross-faded with a periodic-Hann ramp over the ov = win - step shared samples (rising half on
// the later window, falling half on the earlier one: the two gains sum to one).  Window i sits at slot
// (i % world) * per_rank + i / world of `windows` -- the layout an all-gather of round-robin-dealt windows produces
// (world = 1: plain order).  One pass, gather form: no atomics on the output; the global peak is one atomicMax per warp.
__global__ void __launch_bounds__(256)
stitch_kernel(const float* __restrict__ windows, int n_windows, int win, int step, int world, int per_rank,
              float* __restrict__ out, long long n_out, unsigned* __restrict__ peak_bits) {
    const int ov = win - step;
    const float inv_ov = ov > 0 ? 1.0f / (float)ov : 0.f;
    float pk = 0.f;
    for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < n_out; n += (long long)gridDim.x * blockDim.x) {
        long long i1 = n / step; if (i1 > n_windows - 1) i1 = n_windows - 1;
        float acc = 0.f;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const long long i = i1 - q;
            if (i < 0) continue;
            const long long o = n - i * step;
            if (o >= win) continue;
            float g = 1.f;
            if (i > 0 && o < ov) g = 0.5f - 0.5f * cospif((float)o * inv_ov);                               // rising half
            else if (i < n_windows - 1 && o >= win - ov) g = 0.5f + 0.5f * cospif((float)(o - (win - ov)) * inv_ov);   // falling half
            const size_t slot = (size_t)(i % world) * per_rank + (size_t)(i / world);
            acc = fmaf(__ldg(windows + slot * win + o), g, acc);
        }
        out[n] = acc;
        pk = fmaxf(pk, fabsf(acc));
    }
    if (peak_bits) {
#pragma unroll
        for (int o = 16; o; o >>= 1) pk = fmaxf(pk, __shfl_xor_sync(0xffffffffu, pk, o));
        if ((threadIdx.x & 31) == 0 && pk > 0.f) atomicMax(peak_bits, __float_as_uint(pk));
    }
}

template <int NC, int LAYOUT>
static auto stft_variant(bool fast, int fmt) {
    return !fast ? stft_kernel<NC, 0, LAYOUT> : fmt == PG_FMT_F16 ? stft_kernel<NC, 2, LAYOUT> : stft_kernel<NC, 1, LAYOUT>;
}

template <int NC>
static int launch_stft(const float* wave, int B, int N, int T, const float* tw, int mode, float* a, float* bq,
                       uint16_t* hi, uint16_t* lo, long long bs, int fmt, cudaStream_t st, const float* proj_mag = nullptr,
                       float std_mean = 0.f, float std_inv = 1.f, const int* clip_samples = nullptr, const int* clip_frames = nullptr,
                       const long long* clip_offsets = nullptr, long long n_wave = 0) {
    using Cfg = FrameCfg<NC>;
    const bool fast = mode == PG_STFT_LOGMAG && a && !bq && hi && lo;
    auto k = clip_offsets ? stft_variant<NC, kPacked>(fast, fmt)
           : clip_samples ? stft_variant<NC, kRagged>(fast, fmt) : stft_variant<NC, kFixed>(fast, fmt);
    const size_t sm = Cfg::smem_stft();
    static bool configured_dev[kMaxDevices] = {};
    bool& configured = configured_dev[current_device_slot()];
    if (!configured) {
        for (int f = 0; f < 3; ++f)
            for (auto kv : {stft_variant<NC, kFixed>(f > 0, f == 2 ? PG_FMT_F16 : PG_FMT_BF16),
                            stft_variant<NC, kRagged>(f > 0, f == 2 ? PG_FMT_F16 : PG_FMT_BF16),
                            stft_variant<NC, kPacked>(f > 0, f == 2 ? PG_FMT_F16 : PG_FMT_BF16)})
                cudaFuncSetAttribute(kv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        configured = true;
    }
    const int frames_per_cta = Cfg::FC * 4;                 // tables are built once per 4 passes over the frame slots
    dim3 grid((T + frames_per_cta - 1) / frames_per_cta, B);
    k<<<grid, kStftThreads, sm, st>>>(wave, N, T, reinterpret_cast<const float2*>(tw), mode, a, bq, hi, lo, bs, fmt, frames_per_cta, proj_mag,
                                      std_mean, std_inv, clip_samples, clip_frames, clip_offsets, n_wave);
    return check_launch("stft_kernel");
}

template <int NC>
static int launch_istft(const float* a, const float* bq, int mode, int B, int T, const float* tw, float* wave,
                        float* peak, int* nonfinite, cudaStream_t st, const float* b_ss, int b_ss_stride,
                        const int* clip_frames = nullptr, const int* clip_samples = nullptr) {
    using Cfg = FrameCfg<NC>;
    const bool fast = mode == PG_SPEC_POLAR_LOG && bq;
    auto k = clip_frames ? (fast ? istft_kernel<NC, true, true> : istft_kernel<NC, false, true>)
                         : (fast ? istft_kernel<NC, true, false> : istft_kernel<NC, false, false>);
    const size_t sm = Cfg::smem_istft();
    static bool configured_dev[kMaxDevices] = {};
    bool& configured = configured_dev[current_device_slot()];
    if (!configured) {
        for (auto kv : {istft_kernel<NC, true, false>, istft_kernel<NC, false, false>, istft_kernel<NC, true, true>, istft_kernel<NC, false, true>})
            cudaFuncSetAttribute(kv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        configured = true;
    }
    // a run of 11 iterations: 11*FC - 3 output blocks per CTA, 3 halo frames recomputed per run
    const int blocks_per_cta = 11 * Cfg::FC - 3;
    dim3 grid((T - 1 + blocks_per_cta - 1) / blocks_per_cta, B);
    k<<<grid, kStftThreads, sm, st>>>(a, bq, mode, T, reinterpret_cast<const float2*>(tw), wave,
                                     reinterpret_cast<unsigned*>(peak), nonfinite, blocks_per_cta,
                                     reinterpret_cast<const float2*>(b_ss), b_ss_stride, clip_frames, clip_samples);
    return check_launch("istft_kernel");
}

}  // namespace pg

extern "C" int pg_stft_num_frames(int n_samples, int hop) { return hop > 0 ? 1 + n_samples / hop : 0; }

static int stft_entry(const float* wave, int B, int N, int n_fft, int hop, const float* twiddle, int mode,
                      float* out_a, float* out_b, uint16_t* op_hi, uint16_t* op_lo,
                      int64_t op_batch_stride, int op_fmt, const int* cs, const int* cf, pg_stream stream,
                      const int64_t* co = nullptr, int64_t n_wave = 0) {
    PG_REQUIRE(wave && twiddle && B > 0 && N > 0, "pg_stft: null pointer or empty batch");
    PG_REQUIRE(hop * 4 == n_fft, "pg_stft: hop must be n_fft/4 (got n_fft=%d hop=%d)", n_fft, hop);
    PG_REQUIRE(N > n_fft / 2, "pg_stft: reflect padding needs more than n_fft/2 samples (N=%d)", N);
    PG_REQUIRE(mode == PG_STFT_LOGMAG || mode == PG_STFT_REIM, "pg_stft: bad mode %d", mode);
    PG_REQUIRE(B <= 65535, "pg_stft: batch too large for one launch");
    const int T = 1 + N / hop;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    switch (n_fft) {
        case 256:  return pg::launch_stft<128>(wave, B, N, T, twiddle, mode, out_a, out_b, op_hi, op_lo, op_batch_stride, op_fmt, st, nullptr, 0.f, 1.f, cs, cf,
                                                 reinterpret_cast<const long long*>(co), n_wave);
        case 512:  return pg::launch_stft<256>(wave, B, N, T, twiddle, mode, out_a, out_b, op_hi, op_lo, op_batch_stride, op_fmt, st, nullptr, 0.f, 1.f, cs, cf,
                                                 reinterpret_cast<const long long*>(co), n_wave);
        case 1024: return pg::launch_stft<512>(wave, B, N, T, twiddle, mode, out_a, out_b, op_hi, op_lo, op_batch_stride, op_fmt, st, nullptr, 0.f, 1.f, cs, cf,
                                                 reinterpret_cast<const long long*>(co), n_wave);
        case 2048: return pg::launch_stft<1024>(wave, B, N, T, twiddle, mode, out_a, out_b, op_hi, op_lo, op_batch_stride, op_fmt, st, nullptr, 0.f, 1.f, cs, cf,
                                                 reinterpret_cast<const long long*>(co), n_wave);
    }
    pg::set_error("pg_stft: n_fft must be 256, 512, 1024 or 2048 (got %d)", n_fft);
    return PG_ERR_UNSUPPORTED;
}

extern "C" int pg_stft(const float* wave, int B, int N, int n_fft, int hop, const float* twiddle, int mode,
                       float* out_a, float* out_b, uint16_t* op_hi, uint16_t* op_lo,
                       int64_t op_batch_stride, int op_fmt, pg_stream stream) {
    return stft_entry(wave, B, N, n_fft, hop, twiddle, mode, out_a, out_b, op_hi, op_lo, op_batch_stride, op_fmt, nullptr, nullptr, stream);
}

extern "C" int pg_stft_ragged(const float* wave, int B, int N, int n_fft, int hop, const float* twiddle, int mode,
                              float* out_a, float* out_b, uint16_t* op_hi, uint16_t* op_lo,
                              int64_t op_batch_stride, int op_fmt, const int* clip_samples, const int* clip_frames, pg_stream stream) {
    PG_REQUIRE(clip_samples && clip_frames, "pg_stft_ragged: null per-clip table");
    if (mode != PG_STFT_LOGMAG) {
        pg::set_error("pg_stft_ragged: only PG_STFT_LOGMAG takes per-clip lengths (got mode %d)", mode);
        return PG_ERR_UNSUPPORTED;
    }
    return stft_entry(wave, B, N, n_fft, hop, twiddle, mode, out_a, out_b, op_hi, op_lo, op_batch_stride, op_fmt, clip_samples, clip_frames, stream);
}

extern "C" int pg_stft_packed(const float* wave, int64_t n_wave, const int64_t* clip_offsets, int B, int T, int n_fft, int hop,
                              const float* twiddle, int mode, float* out_a, float* out_b, uint16_t* op_hi, uint16_t* op_lo,
                              int64_t op_batch_stride, int op_fmt, const int* clip_frames, pg_stream stream) {
    PG_REQUIRE(clip_offsets && clip_frames && n_wave > 0, "pg_stft_packed: null per-clip table or empty buffer");
    PG_REQUIRE(T >= 2 && hop > 0 && (int64_t)(T - 1) * hop <= INT32_MAX, "pg_stft_packed: bad frame count T=%d", T);
    if (mode != PG_STFT_LOGMAG) {
        pg::set_error("pg_stft_packed: only PG_STFT_LOGMAG takes packed clips (got mode %d)", mode);
        return PG_ERR_UNSUPPORTED;
    }
    return stft_entry(wave, B, (T - 1) * hop, n_fft, hop, twiddle, mode, out_a, out_b, op_hi, op_lo, op_batch_stride, op_fmt,
                      nullptr, clip_frames, stream, clip_offsets, n_wave);
}

extern "C" int pg_stft_project(const float* wave, int B, int N, int n_fft, int hop, const float* twiddle, const float* mag,
                               float* out_re, float* out_im, pg_stream stream) {
    PG_REQUIRE(wave && twiddle && mag && out_re && out_im && B > 0 && N > 0, "pg_stft_project: null pointer or empty batch");
    PG_REQUIRE(hop * 4 == n_fft, "pg_stft_project: hop must be n_fft/4 (got n_fft=%d hop=%d)", n_fft, hop);
    PG_REQUIRE(N > n_fft / 2, "pg_stft_project: reflect padding needs more than n_fft/2 samples (N=%d)", N);
    PG_REQUIRE(B <= 65535, "pg_stft_project: batch too large for one launch");
    const int T = 1 + N / hop;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    switch (n_fft) {
        case 256:  return pg::launch_stft<128>(wave, B, N, T, twiddle, PG_STFT_PROJECT, out_re, out_im, nullptr, nullptr, 0, 0, st, mag);
        case 512:  return pg::launch_stft<256>(wave, B, N, T, twiddle, PG_STFT_PROJECT, out_re, out_im, nullptr, nullptr, 0, 0, st, mag);
        case 1024: return pg::launch_stft<512>(wave, B, N, T, twiddle, PG_STFT_PROJECT, out_re, out_im, nullptr, nullptr, 0, 0, st, mag);
        case 2048: return pg::launch_stft<1024>(wave, B, N, T, twiddle, PG_STFT_PROJECT, out_re, out_im, nullptr, nullptr, 0, 0, st, mag);
    }
    pg::set_error("pg_stft_project: n_fft must be 256, 512, 1024 or 2048 (got %d)", n_fft);
    return PG_ERR_UNSUPPORTED;
}

extern "C" int pg_stft_pairs(const float* wave, int B, int N, int n_fft, int hop, const float* twiddle, float mean, float std,
                             float* out_logmag, float* out_phase, pg_stream stream) {
    PG_REQUIRE(wave && twiddle && out_logmag && out_phase && B > 0 && N > 0, "pg_stft_pairs: null pointer or empty batch");
    PG_REQUIRE(hop * 4 == n_fft, "pg_stft_pairs: hop must be n_fft/4 (got n_fft=%d hop=%d)", n_fft, hop);
    PG_REQUIRE(N > n_fft / 2, "pg_stft_pairs: reflect padding needs more than n_fft/2 samples (N=%d)", N);
    PG_REQUIRE(std > 0.f && B <= 65535, "pg_stft_pairs: std must be positive and B <= 65535");
    const int T = 1 + N / hop;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const float inv = 1.0f / std;
    switch (n_fft) {
        case 256:  return pg::launch_stft<128>(wave, B, N, T, twiddle, PG_STFT_PAIRS, out_logmag, out_phase, nullptr, nullptr, 0, 0, st, nullptr, mean, inv);
        case 512:  return pg::launch_stft<256>(wave, B, N, T, twiddle, PG_STFT_PAIRS, out_logmag, out_phase, nullptr, nullptr, 0, 0, st, nullptr, mean, inv);
        case 1024: return pg::launch_stft<512>(wave, B, N, T, twiddle, PG_STFT_PAIRS, out_logmag, out_phase, nullptr, nullptr, 0, 0, st, nullptr, mean, inv);
        case 2048: return pg::launch_stft<1024>(wave, B, N, T, twiddle, PG_STFT_PAIRS, out_logmag, out_phase, nullptr, nullptr, 0, 0, st, nullptr, mean, inv);
    }
    pg::set_error("pg_stft_pairs: n_fft must be 256, 512, 1024 or 2048 (got %d)", n_fft);
    return PG_ERR_UNSUPPORTED;
}

static int istft_entry(const float* in_a, const float* in_b, int mode, int B, int T, int n_fft, int hop,
                       const float* twiddle, float* wave, float* peak, int* nonfinite,
                       const float* b_scale_shift, int b_ss_per_clip, const int* cf, const int* cs, pg_stream stream) {
    PG_REQUIRE(in_a && twiddle && wave && B > 0 && T > 1, "pg_istft: null pointer or empty input");
    PG_REQUIRE(hop * 4 == n_fft, "pg_istft: hop must be n_fft/4 (got n_fft=%d hop=%d)", n_fft, hop);
    PG_REQUIRE(mode >= PG_SPEC_POLAR_LOG && mode <= PG_SPEC_POLAR_MAG, "pg_istft: bad mode %d", mode);
    PG_REQUIRE(in_b || mode != PG_SPEC_CARTESIAN, "pg_istft: second plane missing");   // polar modes: NULL phase = zero phase
    PG_REQUIRE(B <= 65535, "pg_istft: batch too large for one launch");
    PG_REQUIRE(!b_scale_shift || in_b, "pg_istft: scale/shift given without a second plane");
    const int ss_stride = b_ss_per_clip ? n_fft / 2 : 0;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (peak) cudaMemsetAsync(peak, 0, sizeof(float) * B, st);
    if (nonfinite) cudaMemsetAsync(nonfinite, 0, sizeof(int) * B, st);
    switch (n_fft) {
        case 256:  return pg::launch_istft<128>(in_a, in_b, mode, B, T, twiddle, wave, peak, nonfinite, st, b_scale_shift, ss_stride, cf, cs);
        case 512:  return pg::launch_istft<256>(in_a, in_b, mode, B, T, twiddle, wave, peak, nonfinite, st, b_scale_shift, ss_stride, cf, cs);
        case 1024: return pg::launch_istft<512>(in_a, in_b, mode, B, T, twiddle, wave, peak, nonfinite, st, b_scale_shift, ss_stride, cf, cs);
        case 2048: return pg::launch_istft<1024>(in_a, in_b, mode, B, T, twiddle, wave, peak, nonfinite, st, b_scale_shift, ss_stride, cf, cs);
    }
    pg::set_error("pg_istft: n_fft must be 256, 512, 1024 or 2048 (got %d)", n_fft);
    return PG_ERR_UNSUPPORTED;
}

extern "C" int pg_istft(const float* in_a, const float* in_b, int mode, int B, int T, int n_fft, int hop,
                        const float* twiddle, float* wave, float* peak, int* nonfinite,
                        const float* b_scale_shift, int b_ss_per_clip, pg_stream stream) {
    return istft_entry(in_a, in_b, mode, B, T, n_fft, hop, twiddle, wave, peak, nonfinite, b_scale_shift, b_ss_per_clip, nullptr, nullptr, stream);
}

extern "C" int pg_istft_ragged(const float* in_a, const float* in_b, int mode, int B, int T, int n_fft, int hop,
                               const float* twiddle, float* wave, float* peak, int* nonfinite,
                               const float* b_scale_shift, int b_ss_per_clip, const int* clip_frames, const int* clip_samples,
                               pg_stream stream) {
    PG_REQUIRE(clip_frames && clip_samples, "pg_istft_ragged: null per-clip table");
    return istft_entry(in_a, in_b, mode, B, T, n_fft, hop, twiddle, wave, peak, nonfinite, b_scale_shift, b_ss_per_clip, clip_frames, clip_samples, stream);
}

extern "C" int pg_peak_normalize(float* wave, const float* peak, int B, int N, pg_stream stream) {
    PG_REQUIRE(wave && peak && B > 0 && N > 0 && B <= 65535, "pg_peak_normalize: bad arguments");
    dim3 grid((N + 1023) / 1024 < 64 ? (N + 1023) / 1024 : 64, B);
    pg::peak_normalize_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        wave, reinterpret_cast<const unsigned*>(peak), N);
    return pg::check_launch("peak_normalize_kernel");
}

extern "C" int pg_peak_normalize_packed(const float* src, int B, int64_t src_pitch, const float* peak,
                                        const int64_t* clip_offsets, float* dst, int64_t n_dst, pg_stream stream) {
    PG_REQUIRE(src && clip_offsets && dst && B > 0 && B <= 65535 && src_pitch > 0 && n_dst >= 0,
               "pg_peak_normalize_packed: bad arguments");
    const int64_t per = (src_pitch + 1023) / 1024;
    dim3 grid(per < 64 ? (unsigned)per : 64u, B);
    pg::peak_normalize_packed_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        src, src_pitch, reinterpret_cast<const unsigned*>(peak), reinterpret_cast<const long long*>(clip_offsets), dst, n_dst);
    return pg::check_launch("peak_normalize_packed_kernel");
}

extern "C" int pg_stitch(const float* windows, int n_windows, int win, int step, int world, int per_rank, float* out,
                         int64_t n_out, float* peak, pg_stream stream) {
    PG_REQUIRE(windows && out && n_windows > 0 && win > 0 && n_out > 0, "pg_stitch: bad arguments");
    PG_REQUIRE(step > 0 && step <= win && 2 * step >= win, "pg_stitch: step must lie in [win/2, win] (got win=%d step=%d)", win, step);
    PG_REQUIRE(world >= 1 && per_rank >= (n_windows + world - 1) / world, "pg_stitch: per_rank too small for %d windows on %d ranks", n_windows, world);
    PG_REQUIRE(n_out <= (int64_t)win + (int64_t)(n_windows - 1) * step, "pg_stitch: n_out exceeds the span of the windows");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (peak) cudaMemsetAsync(peak, 0, sizeof(float), st);
    long long blocks = (n_out + 255) / 256; if (blocks > 148 * 16) blocks = 148 * 16;
    pg::stitch_kernel<<<(int)blocks, 256, 0, st>>>(windows, n_windows, win, step, world, per_rank, out, n_out, reinterpret_cast<unsigned*>(peak));
    return pg::check_launch("stitch_kernel");
}
