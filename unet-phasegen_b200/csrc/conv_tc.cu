// Implicit-GEMM Conv1d / ConvTranspose1d on the 5th-gen tensor cores (tcgen05 + TMEM + TMA).
//
// Reference path replaced: the eight nn.Conv1d / nn.ConvTranspose1d calls of
// /root/reference/model.py:77-78,88-89,94-95,101-102 (library cuDNN/oneDNN kernels there).
//
// Formulation.  Activations are channels-last bf16 [B][rows][C] stored as two planes
// (hi, lo; x = hi + lo to 2^-16), weights are packed [tap][C_out][C_in] as two planes too.
// One CTA tile is  D[128 output channels][N output positions of one clip and one output
// phase], accumulated in TMEM (fp32) over K = (tap, 64-channel chunk):
//     D += Whi*Xhi + Whi*Xlo + Wlo*Xhi          (n_terms = 3, "fp32-class": rel. error ~2^-16)
//     D += Whi*Xhi                              (n_terms = 1, plain bf16)
// Operands reach shared memory by TMA with 128-byte swizzle, K-major:
//   A (weights)    : box {64 ci, 128 co, 1 tap}
//   B (activations): box {64 ci, 1 parity, R rows, 1 clip}.  The zero padding of the
//     convolution is TMA's out-of-bounds zero fill (row coordinate < 0 or >= extent), the
//     stride-2 convolutions read the even/odd row view of the same buffer (parity dim), and a
//     stride-2 transposed convolution is two interleaved output phases, each a stride-1
//     correlation over the taps of matching parity.
//   "Strip" reuse: consecutive taps read the same rows shifted by one, so one activation strip
//   of N + shift rows is loaded per (chunk, tap group) and every tap of the group issues its
//   MMAs from a descriptor whose start address is advanced by shift*128 B inside the swizzle
//   pattern.  taps_per_group = 1 disables the trick (one strip per tap).
// Warp roles (192 threads): warp 0 TMA producer, warp 1 MMA issuer (+TMEM alloc), warps 2-5
// epilogue: TMEM -> registers -> one of three forms (PG_EPI_*, include/phasegen.h):
//   RAW       per-channel partial batch-norm statistics (count, mean, M2; two passes over TMEM so the
//             variance is centred) and the raw fp32 output, channels-last;
//   ACT       activation(s) (model.py:80,82) and the consumers' 16-bit hi/lo operand planes, written at a
//             channel offset (the skip concat of model.py:113) -- layers without norm;
//   NORM_ACT  train-mode norm with the clip's own statistics first (three passes over TMEM), for tiles that
//             hold every output position of a clip ("whole-clip" tiles: all output phases x position tiles
//             side by side in the accumulator, see ConvPlan::whole_clip).
// Stores go through a per-warp shared-memory tile so that they leave as 128-bit stores.
// Persistent: grid = min(#tiles, #SMs); the tile order keeps co-resident CTAs on the same
// weight slab (L2 reuse).  Two TMEM accumulators (2 x 256 columns) overlap epilogue and MMA.
//
// CTA pairs (PAIR = true, the default whenever C_out is a multiple of 256).  In the single-CTA form
// every MMA reads its 128 x 16 weight tile AND its N x 16 activation tile from shared memory, and the
// measured tensor-pipe time per MMA is ~32 + N/2 cycles instead of N/2 (profiles/r01_conv_tc_ncu_full_v1.csv:
// 72 % at N = 176): the operand reads are what paces the pipe.  A cluster of two CTAs on one TPC issues
// cta_group::2 MMAs with M = 256 instead: CTA r owns output channels [256 t + 128 r, +128) (its own
// weight tile, its own TMEM lanes) and supplies positions [r N/2, (r+1) N/2) of the activation strip,
// so the activation bytes each SM reads per MMA halve.  Only the even CTA issues MMAs; both CTAs run a
// TMA producer (bytes are counted on the even CTA's "full" barriers, cta_group::2 TMA), the "empty" and
// "accumulator full" barriers are signalled in both CTAs by multicast commits, and the epilogue warps of
// both CTAs release the accumulator on the even CTA's barrier.
#include "tc_ptx.cuh"
#include "conv_plan.h"

namespace pg {

// ------------------------------------------------------------------------------------ kernel
struct ConvTcParams {
    ConvPlan plan;                  // tap tables, tile geometry (conv_plan.h)
    float* y;                       // [B][out_rows][out_ld] raw conv output (fp32)
    float4* stats;                  // [B][P][C_out] {n, mean, M2, 0}, P = OS * n_ntiles; may be null
    int n_a_slots;                  // A ring depth
    int b_slot_bytes;               // bytes of one plane of a B strip (R * 128)
    int n_terms;                    // 3 = hi*hi + hi*lo + lo*hi, 2 = Whi*(Xhi + Xlo), 1 = hi*hi
    int f16;                        // operand planes are fp16 (else bf16)
    int base_offset_mode;           // descriptor base-offset handling for shifted strips
    int a_mn;                       // weight planes are [k][C_in][C_out]: A is fed MN-major (data-gradient mode)
    // fused epilogue (model.py:80-83,113): PG_EPI_RAW stores y (+ statistics records); PG_EPI_ACT applies the activation(s)
    // and writes the consumers' operand planes; PG_EPI_NORM_ACT first normalises with the clip's own statistics
    // (train-mode norm of a batch-1 call), which are complete inside the tile (plan.whole_clip or a one-part layer)
    int epi_mode;
    const float* gamma; const float* beta; float eps;
    ActDst dst0, dst1;
    float2* ss_out;                 // NORM_ACT: optional [B][C_out] (scale, shift) record of what was applied
    const int* clip_rows;           // ragged batch (RAGGED = true): valid output rows L_b <= L_out of each clip
};
// plan.pair = 1: tiles are 256 output channels wide and owned by a CTA pair; plan.strip_rows is then the
// HALF strip each CTA loads (n_tile/2 + largest shift rows).

constexpr int kThreads = 192;
constexpr int kATileBytes = 128 * 128;        // one plane: 128 co x 64 ci bf16
constexpr int kMaxASlots = 8;

struct TileCoord { int co_tile, phase, b0, nt; };

// Tile order: clips are taken in L2-sized groups; inside a group all tiles of one weight slab
// (128 output channels x one output phase) are adjacent, so co-resident CTAs share the slab and
// the group's activations are read from HBM once and re-used from L2 by every slab.
__device__ __forceinline__ int n_bundles(const ConvPlan& p) { return (p.B + p.nb - 1) / p.nb; }
__device__ __forceinline__ int n_co_slabs(const ConvPlan& p) { return p.pair ? p.n_cotiles / 2 : p.n_cotiles; }
// whole-clip tiles carry every phase and position tile of their clips: the phase / position-tile coordinates collapse
__device__ __forceinline__ int tile_OS(const ConvPlan& p) { return p.whole_clip ? 1 : p.OS; }
__device__ __forceinline__ int tile_NT(const ConvPlan& p) { return p.whole_clip ? 1 : p.n_ntiles; }
__device__ __forceinline__ int total_tiles(const ConvPlan& p) { return n_co_slabs(p) * tile_OS(p) * n_bundles(p) * tile_NT(p); }
__device__ __forceinline__ TileCoord decode_tile(const ConvPlan& p, int tile) {
    TileCoord c;
    const int OSx = tile_OS(p), NTx = tile_NT(p);
    const int nbg = n_bundles(p), G = p.clip_group, n_slabs = n_co_slabs(p) * OSx;
    const int tiles_full = n_slabs * G * NTx;
    const int g = tile / tiles_full, r = tile % tiles_full;
    int Gg = nbg - g * G; if (Gg > G) Gg = G;
    const int per_slab = Gg * NTx;
    const int slab = r / per_slab, r2 = r % per_slab;
    c.co_tile = slab / OSx; c.phase = slab % OSx;
    c.b0 = (g * G + r2 / NTx) * p.nb; c.nt = r2 % NTx;
    return c;
}

// RAGGED: clip b's output is valid in rows [0, L_b) only (prm.clip_rows).  Statistics count those rows; the fused
// epilogues write zeros into rows [L_b, L_out) of their destinations, so a later layer reads zeros there, as TMA's
// out-of-bounds fill supplies them to the same clip run alone.
template <bool PAIR, bool RAGGED>
__global__ void __launch_bounds__(kThreads, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
               const __grid_constant__ CUtensorMap map_x_hi, const __grid_constant__ CUtensorMap map_x_lo,
               const __grid_constant__ ConvTcParams prm) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const ConvPlan& pl = prm.plan;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int nA = prm.n_a_slots;
    const int bPlane = prm.b_slot_bytes;
    const int a_planes = prm.n_terms == 3 ? 2 : 1;            // weight planes per slot: hi (+ lo)
    const int b_planes = prm.n_terms >= 2 ? 2 : 1;            // activation planes per slot: hi (+ lo)
    uint8_t* a_base = smem;                                   // nA x {hi 16 KB (, lo 16 KB)}
    uint8_t* b_base = a_base + (size_t)nA * a_planes * kATileBytes;  // 2 x {hi bPlane (, lo bPlane)}
    uint64_t* bars = reinterpret_cast<uint64_t*>(b_base + 2 * (size_t)b_planes * bPlane);
    uint64_t* fullA = bars;                   // [kMaxASlots]
    uint64_t* emptyA = bars + kMaxASlots;     // [kMaxASlots]
    uint64_t* fullB = bars + 2 * kMaxASlots;  // [2]
    uint64_t* emptyB = fullB + 2;             // [2]
    uint64_t* accFull = emptyB + 2;           // [2]
    uint64_t* accEmpty = accFull + 2;         // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accEmpty + 2);
    uint32_t* epi_tiles = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(bars) + 256);   // 4 warps x [16 rows][32 ch] words

    // warp index through a shuffle: provably warp-uniform, so the role branches below are uniform branches and
    // the single-thread instructions' operands can live in uniform registers
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int n_tiles = total_tiles(pl);
    const bool w_lo = prm.n_terms == 3, x_lo = prm.n_terms >= 2;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&map_w_hi); tma_prefetch_desc(&map_x_hi);
        if (w_lo) tma_prefetch_desc(&map_w_lo);
        if (x_lo) tma_prefetch_desc(&map_x_lo);
        for (int i = 0; i < nA; ++i) { mbar_init(fullA + i, 1); mbar_init(emptyA + i, 1); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(fullB + i, 1); mbar_init(emptyB + i, 1);
            mbar_init(accFull + i, 1); mbar_init(accEmpty + i, PAIR ? 8 : 4);
        }
        fence_barrier_init();
    }
    if (warp == 1) { if (PAIR) tmem_alloc_pair(tmem_slot, 512); else tmem_alloc(tmem_slot, 512); }
    tc_fence_before();
    if (PAIR) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
    const int rank = PAIR ? (int)cluster_ctarank() : 0;           // 0 = leader (issues the MMAs)
    const int tile0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int tile_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int half_n = pl.n_tile >> 1;                            // PAIR, not merged: positions each CTA supplies per clip
    const int nb_grp = pl.nb / pl.mgroups;                        // clips per MMA (merged) / per tile (mgroups = 1)
    const int nb_cta = (PAIR && pl.merged) ? nb_grp >> 1 : nb_grp;   // clips of one group whose strips this CTA loads
    const int t_phases = pl.whole_clip ? pl.OS : 1;               // phases / position tiles ("parts") held by one tile
    const int t_nts = pl.whole_clip ? pl.n_ntiles : 1;
    const int n_sub = pl.merged ? pl.mgroups : t_nts;             // activation boxes per strip slot

    if (warp == 0) {
        // ===================================================================== TMA producer
        // Warp-uniform like the MMA warp (every lane runs the loop, one elected lane issues): the TMA operands
        // live in uniform registers instead of going through an R2UR waterfall per UTMALDG, and the ring
        // indices are counters (no runtime division).  With one or two products per MAC a weight tile is
        // consumed in 640-770 tensor cycles, so the producer's per-tap cost is on the critical path.
        {
            uint32_t b_it = 0;
            int a_slot = 0; uint32_t a_ph = 0;
            const uint32_t grp_bytes = (uint32_t)nb_cta * pl.strip_rows * 128u;   // one merged group's strips in this CTA
            const uint32_t a_bytes = a_planes * kATileBytes;
            const uint32_t b_bytes = b_planes * (uint32_t)bPlane;
            for (int tile = tile0; tile < n_tiles; tile += tile_step) {
                TileCoord tc = decode_tile(pl, tile);
                if (PAIR) tc.co_tile = tc.co_tile * 2 + rank;
                const int m0 = tc.nt * pl.n_tile + ((PAIR && !pl.merged) ? rank * half_n : 0);
                const int clip0 = tc.b0 + ((PAIR && pl.merged) ? rank * nb_cta : 0);   // + g * nb_grp per merged group
                for (int ch = 0; ch < pl.n_chunks; ++ch) {
                  for (int ph = tc.phase; ph < tc.phase + t_phases; ++ph) {
                    const int ng = pl.n_groups[ph];
                    for (int g = 0; g < ng; ++g) {
                        const ConvGroup grp = pl.groups[ph][g];
                        {
                            const int s = b_it & 1; const uint32_t bph = (b_it >> 1) & 1;
                            mbar_wait(emptyB + s, bph ^ 1);
                            uint8_t* dst = b_base + (size_t)s * b_planes * bPlane;
                            if (elect_one()) {
                                if (PAIR) { if (rank == 0) mbar_expect_tx(fullB + s, 2 * b_bytes); }   // both CTAs' halves
                                else mbar_expect_tx(fullB + s, b_bytes);
                                // one box per merged group (its clips are contiguous) / per position tile of a whole-clip tile
                                for (int sub = 0; sub < n_sub; ++sub) {
                                    uint8_t* dg = dst + (size_t)sub * grp_bytes;
                                    const int cg = clip0 + (pl.merged ? sub * nb_grp : 0);
                                    const int r0 = m0 + (pl.merged ? 0 : sub * pl.n_tile) + grp.row0;
                                    if (PAIR) {
                                        tma_load_4d_pair(dg, &map_x_hi, fullB + s, ch * 64, grp.parity, r0, cg);
                                        if (x_lo) tma_load_4d_pair(dg + bPlane, &map_x_lo, fullB + s, ch * 64, grp.parity, r0, cg);
                                    } else {
                                        tma_load_4d(dg, &map_x_hi, fullB + s, ch * 64, grp.parity, r0, cg);
                                        if (x_lo) tma_load_4d(dg + bPlane, &map_x_lo, fullB + s, ch * 64, grp.parity, r0, cg);
                                    }
                                }
                            }
                            __syncwarp();
                            ++b_it;
                        }
                        for (int j = 0; j < grp.n_taps; ++j) {
                            const int w_idx = pl.taps[ph][grp.first_tap + j].w_idx;
                            const int s = a_slot; const uint32_t aph = a_ph;
                            mbar_wait(emptyA + s, aph ^ 1);
                            uint8_t* dst = a_base + (size_t)s * a_planes * kATileBytes;
                            if (elect_one()) {
                                if (!PAIR) mbar_expect_tx(fullA + s, a_bytes);
                                else if (rank == 0) mbar_expect_tx(fullA + s, 2 * a_bytes);
                                auto load_w = [&](uint8_t* d, const CUtensorMap* m, int c0, int c1) {
                                    if (PAIR) tma_load_3d_pair(d, m, fullA + s, c0, c1, w_idx);
                                    else tma_load_3d(d, m, fullA + s, c0, c1, w_idx);
                                };
                                if (prm.a_mn) {     // two {64 co, 64 ci-rows} boxes: MN-major atom stacks, 8 KB apart
                                    for (int h = 0; h < 2; ++h) {
                                        load_w(dst + h * 8192, &map_w_hi, tc.co_tile * 128 + h * 64, ch * 64);
                                        if (w_lo) load_w(dst + kATileBytes + h * 8192, &map_w_lo, tc.co_tile * 128 + h * 64, ch * 64);
                                    }
                                } else {
                                    load_w(dst, &map_w_hi, ch * 64, tc.co_tile * 128);
                                    if (w_lo) load_w(dst + kATileBytes, &map_w_lo, ch * 64, tc.co_tile * 128);
                                }
                            }
                            __syncwarp();
                            if (++a_slot == nA) { a_slot = 0; a_ph ^= 1; }
                        }
                    }
                  }
                }
            }
        }
    } else if (warp == 1) {
        // ======================================================================= MMA issuer
        // The whole warp runs this loop with warp-uniform control flow; only the tcgen05 instructions
        // themselves are issued by one elected lane (always the same one, so tcgen05.commit tracks them).
        if (rank == 0) {
            uint32_t b_it = 0, t_it = 0;
            int a_slot = 0; uint32_t a_ph = 0;
            // operand format field: 1 = bf16, 0 = fp16 (bits [7,10) for A, [10,13) for B)
            const int n_mma = pl.merged ? nb_grp * pl.strip_rows : pl.n_tile;
            // merged: one MMA covers every clip of a group (column step n_mma); else position tiles (outer) x clips (inner),
            // strips laid out [position tile][clip], clip c's parts at columns c * (n_tile * parts per clip)
            const int n_outer = pl.merged ? 1 : t_nts, n_inner = pl.merged ? pl.mgroups : pl.nb;
            const uint32_t dcol_step = pl.merged ? (uint32_t)n_mma : (uint32_t)(pl.n_tile * t_phases * t_nts);
            const uint32_t idesc = (make_idesc_bf16(n_mma, PAIR ? 256 : 128) & ~(prm.f16 ? ((7u << 7) | (7u << 10)) : 0u)) |
                                   (prm.a_mn ? (1u << 15) : 0u);
            const bool a_mn = prm.a_mn != 0;
            // descriptors travel as their low 32-bit words (tc_ptx.cuh): the issue loop only adds to start addresses
            auto mma = [&](uint32_t d, uint32_t da, uint32_t db, uint32_t acc_flag) {
                if (elect_one()) { if (PAIR) umma_words_pair(d, da, db, idesc, acc_flag); else umma_words(d, da, db, idesc, acc_flag); }
            };
            const uint32_t a_step = a_mn ? (2048u >> 4) : (32u >> 4);   // +16 K elements: 2 atoms down (MN-major) / 32 B along (K-major)
            auto commit = [&](uint64_t* bar) {
                if (elect_one()) { if (PAIR) umma_commit_pair(bar); else umma_commit(bar); }
                __syncwarp();
            };
            for (int tile = tile0; tile < n_tiles; tile += tile_step, ++t_it) {
                TileCoord tc = decode_tile(pl, tile);
                const int acc = pl.acc_stages == 2 ? (t_it & 1) : 0;
                const uint32_t acc_ph = pl.acc_stages == 2 ? ((t_it >> 1) & 1) : (t_it & 1);
                mbar_wait_sleep(accEmpty + acc, acc_ph ^ 1, 200);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * 256;
                const uint32_t strip_bytes = (uint32_t)pl.strip_rows * 128u;
                // merged: MMA c covers the nb_grp clips of group c (columns c*n_mma ...); else one MMA per (position tile,
                // clip) of the tile, part (phase, nt) of clip c at column ((c*t_phases + phase)*t_nts + nt)*n_tile
                const uint32_t clip_step = (pl.merged ? (uint32_t)nb_cta * strip_bytes : strip_bytes) >> 4;   // descriptor units
                for (int ch = 0; ch < pl.n_chunks; ++ch) {
                  for (int ph = tc.phase; ph < tc.phase + t_phases; ++ph) {
                    const int ng = pl.n_groups[ph];
                    const uint32_t dcol_ph = d_tmem + (uint32_t)((ph - tc.phase) * t_nts * pl.n_tile);
                    for (int g = 0; g < ng; ++g) {
                        const ConvGroup grp = pl.groups[ph][g];
                        const int bs = b_it & 1; const uint32_t bph = (b_it >> 1) & 1;
                        mbar_wait(fullB + bs, bph);
                        tc_fence_after();
                        const uint32_t b_hi = smem_u32(b_base + (size_t)bs * b_planes * bPlane);
                        const uint32_t b_lo = b_hi + bPlane;
                        for (int j = 0; j < grp.n_taps; ++j) {
                            const ConvTap tp = pl.taps[ph][grp.first_tap + j];
                            const int as = a_slot; const uint32_t aph = a_ph;
                            mbar_wait(fullA + as, aph);
                            tc_fence_after();
                            const uint32_t a_hi = smem_u32(a_base + (size_t)as * a_planes * kATileBytes);
                            const uint32_t a_lo = a_hi + kATileBytes;
                            const uint32_t sh = (uint32_t)tp.shift * 128u;
                            const uint32_t acc_first = (ch | g | j) ? 1u : 0u;   // first MMA into this phase's columns overwrites
                            // one MMA group per (position tile, clip) of the bundle -- merged: per clip group.  Offsets advance by
                            // additions only: this loop is the issue path of the tensor pipe (one MMA per ~88 tensor cycles
                            // with two products per MAC), a runtime division per group starved it (measured: -31 %).
                            const uint32_t aw_hi = a_mn ? desc_lo_sw128_mn(a_hi, 8192) : desc_lo_sw128(a_hi);
                            const uint32_t aw_lo = a_mn ? desc_lo_sw128_mn(a_lo, 8192) : desc_lo_sw128(a_lo);
                            uint32_t bw_hi = desc_lo_sw128(b_hi + sh), bw_lo = desc_lo_sw128(b_lo + sh);
                            for (int o = 0; o < n_outer; ++o) {
                                uint32_t dcol = dcol_ph + (uint32_t)o * (uint32_t)pl.n_tile;
                                for (int c = 0; c < n_inner; ++c, bw_hi += clip_step, bw_lo += clip_step, dcol += dcol_step) {
                                    if (w_lo) {
#pragma unroll
                                        for (uint32_t kk = 0; kk < 4; ++kk) {   // 4 x (K = 16) per 64-channel chunk
                                            mma(dcol, aw_lo + kk * a_step, bw_hi + kk * 2, kk == 0 ? acc_first : 1u);
                                            mma(dcol, aw_hi + kk * a_step, bw_lo + kk * 2, 1);
                                            mma(dcol, aw_hi + kk * a_step, bw_hi + kk * 2, 1);
                                        }
                                    } else if (x_lo) {
#pragma unroll
                                        for (uint32_t kk = 0; kk < 4; ++kk) {
                                            mma(dcol, aw_hi + kk * a_step, bw_lo + kk * 2, kk == 0 ? acc_first : 1u);
                                            mma(dcol, aw_hi + kk * a_step, bw_hi + kk * 2, 1);
                                        }
                                    } else {
#pragma unroll
                                        for (uint32_t kk = 0; kk < 4; ++kk) mma(dcol, aw_hi + kk * a_step, bw_hi + kk * 2, kk == 0 ? acc_first : 1u);
                                    }
                                }
                            }
                            commit(emptyA + as);
                            if (++a_slot == nA) { a_slot = 0; a_ph ^= 1; }
                        }
                        commit(emptyB + bs);
                        ++b_it;
                    }
                  }
                }
                commit(accFull + acc);
            }
        }
    } else {
        // ========================================================================= epilogue
        // A thread owns one output channel (TMEM lane) and reads 16 consecutive positions per tcgen05.ld.  Storing them
        // directly is one 2- or 4-byte store per element (64-128 B per warp instruction): measured, the global-store
        // instruction rate -- not bytes -- then bounds the epilogue (+16 % on d1 with two fp16 destinations).  So every
        // 16 x 32 chunk goes through a private shared-memory tile [16 rows][32 channels] of 32-bit words (conflict-free
        // both ways) and leaves as 128-bit stores of 8 (16-bit planes) or 4 (fp32) consecutive channels of one row.
        const int q = warp & 3;                               // TMEM lane quarter this warp may read
        uint32_t* tile = epi_tiles + q * 512;
        uint32_t t_it = 0;
        const int n_parts = t_phases * t_nts;
        const int col_pitch = pl.merged ? pl.strip_rows : pl.n_tile * n_parts;   // accumulator columns per clip
        bool bad_range = false;
        // fp32 rows: v[i] = value of row (row0 + i*OS) of this thread's channel, i < nv
        auto store_f32 = [&](float* base, size_t off0, size_t row_pitch, const float* v, int nv) {
#pragma unroll
            for (int i = 0; i < 16; ++i) tile[i * 32 + lane] = __float_as_uint(v[i]);
            __syncwarp();
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int idx = lane + 32 * t, r = idx >> 3, part = idx & 7;
                if (r < nv) {
                    const uint4 w = *reinterpret_cast<const uint4*>(tile + r * 32 + part * 4);
                    *reinterpret_cast<uint4*>(base + off0 + (size_t)r * row_pitch + part * 4) = w;
                }
            }
            __syncwarp();
        };
        // activation + hi/lo split into a consumer's operand planes (hi | lo << 16 per word in the tile)
        auto store_split = [&](const ActDst& d, size_t off0, size_t row_pitch, const float* v, int nv) {
            const int fmt = fmt_of_dtype(d.dtype);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float a = leaky(v[i], d.slope);
                uint16_t h, l;
                split16(a, fmt, h, l);
                if (fmt == PG_FMT_F16 && i < nv) bad_range |= !f16_fits(a);
                tile[i * 32 + lane] = (uint32_t)h | ((uint32_t)l << 16);
            }
            __syncwarp();
            const bool two = d.dtype == PG_DT_BF16_SPLIT || d.dtype == PG_DT_F16_SPLIT;
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                const int idx = lane + 32 * t, r = idx >> 2, part = idx & 3;
                if (r < nv) {
                    const uint4 w0 = *reinterpret_cast<const uint4*>(tile + r * 32 + part * 8);
                    const uint4 w1 = *reinterpret_cast<const uint4*>(tile + r * 32 + part * 8 + 4);
                    uint4 hv, lv;
                    hv.x = __byte_perm(w0.x, w0.y, 0x5410); hv.y = __byte_perm(w0.z, w0.w, 0x5410);
                    hv.z = __byte_perm(w1.x, w1.y, 0x5410); hv.w = __byte_perm(w1.z, w1.w, 0x5410);
                    lv.x = __byte_perm(w0.x, w0.y, 0x7632); lv.y = __byte_perm(w0.z, w0.w, 0x7632);
                    lv.z = __byte_perm(w1.x, w1.y, 0x7632); lv.w = __byte_perm(w1.z, w1.w, 0x7632);
                    const size_t o = off0 + (size_t)r * row_pitch + part * 8;
                    *reinterpret_cast<uint4*>(static_cast<uint16_t*>(d.hi) + o) = hv;
                    if (two) *reinterpret_cast<uint4*>(static_cast<uint16_t*>(d.lo) + o) = lv;
                }
            }
            __syncwarp();
        };
        for (int tile_i = tile0; tile_i < n_tiles; tile_i += tile_step, ++t_it) {
            TileCoord tc = decode_tile(pl, tile_i);
            if (PAIR) tc.co_tile = tc.co_tile * 2 + rank;
            const int acc = pl.acc_stages == 2 ? (t_it & 1) : 0;
            const uint32_t acc_ph = pl.acc_stages == 2 ? ((t_it >> 1) & 1) : (t_it & 1);
            mbar_wait_sleep(accFull + acc, acc_ph, 1000);
            tc_fence_after();
            const int co_base = tc.co_tile * 128 + q * 32;
            const int co = co_base + lane;
            // part p = (phase, position tile) of the tile: its columns among the first L output rows, and the output row
            // of its column 0
            auto part_geom = [&](int p, int L, int& phase, int& m0, int& n_valid) {
                phase = tc.phase + p / t_nts;
                m0 = (tc.nt + p % t_nts) * pl.n_tile;
                const int l_phase = (L - phase + pl.OS - 1) / pl.OS;          // positions of this phase
                n_valid = l_phase - m0; if (n_valid > pl.n_tile) n_valid = pl.n_tile; if (n_valid < 0) n_valid = 0;
            };
            for (int c = 0; c < pl.nb; ++c) {
                const int b = tc.b0 + c;
                if (b >= pl.B) break;
                const int L_b = RAGGED ? min(__ldg(prm.clip_rows + b), pl.L_out) : pl.L_out;   // rows holding the clip's own output
                const uint32_t tclip = tmem_base + acc * 256 + c * col_pitch + ((uint32_t)(q * 32) << 16);
                if (prm.epi_mode == PG_EPI_RAW) {
                    for (int p = 0; p < n_parts; ++p) {
                        int phase, m0, n_valid;
                        part_geom(p, L_b, phase, m0, n_valid);
                        const uint32_t taddr = tclip + p * pl.n_tile;
                        // pass 1: mean over the valid columns
                        float sum = 0.f;
                        for (int c0 = 0; c0 < n_valid; c0 += 16) {
                            float v[16];
                            tmem_ld16(taddr + c0, v);
#pragma unroll
                            for (int i = 0; i < 16; ++i) if (c0 + i < n_valid) sum += v[i];
                        }
                        const float mean = n_valid > 0 ? sum / (float)n_valid : 0.f;
                        // pass 2: centred second moment + store
                        float m2 = 0.f;
                        const size_t row_pitch = (size_t)pl.OS * pl.out_ld;
                        for (int c0 = 0; c0 < n_valid; c0 += 16) {
                            float v[16];
                            tmem_ld16(taddr + c0, v);
#pragma unroll
                            for (int i = 0; i < 16; ++i) if (c0 + i < n_valid) { const float d = v[i] - mean; m2 += d * d; }
                            const size_t off0 = ((size_t)b * pl.out_rows + (size_t)(m0 + c0) * pl.OS + phase) * pl.out_ld + co_base;
                            store_f32(prm.y, off0, row_pitch, v, n_valid - c0);
                        }
                        if (prm.stats) {
                            const int P = pl.OS * pl.n_ntiles;
                            const int pi = phase * pl.n_ntiles + m0 / pl.n_tile;
                            prm.stats[((size_t)b * P + pi) * pl.C_out + co] = make_float4((float)n_valid, mean, m2, 0.f);
                        }
                    }
                } else {
                    // fused norm (per-clip statistics, complete inside this tile) + activation(s) + operand-plane store
                    float sc = 1.f, sh = 0.f;
                    if (prm.epi_mode == PG_EPI_NORM_ACT) {
                        float sum = 0.f; int n_tot = 0;
                        for (int p = 0; p < n_parts; ++p) {
                            int phase, m0, n_valid;
                            part_geom(p, L_b, phase, m0, n_valid);
                            n_tot += n_valid;
                            for (int c0 = 0; c0 < n_valid; c0 += 16) {
                                float v[16];
                                tmem_ld16(tclip + p * pl.n_tile + c0, v);
#pragma unroll
                                for (int i = 0; i < 16; ++i) if (c0 + i < n_valid) sum += v[i];
                            }
                        }
                        const float mean = n_tot > 0 ? sum / (float)n_tot : 0.f;
                        float m2 = 0.f;
                        for (int p = 0; p < n_parts; ++p) {
                            int phase, m0, n_valid;
                            part_geom(p, L_b, phase, m0, n_valid);
                            for (int c0 = 0; c0 < n_valid; c0 += 16) {
                                float v[16];
                                tmem_ld16(tclip + p * pl.n_tile + c0, v);
#pragma unroll
                                for (int i = 0; i < 16; ++i) if (c0 + i < n_valid) { const float d = v[i] - mean; m2 += d * d; }
                            }
                        }
                        const float var = n_tot > 0 ? m2 / (float)n_tot : 0.f;
                        sc = (prm.gamma ? __ldg(prm.gamma + co) : 1.f) * rsqrtf(var + prm.eps);
                        sh = (prm.beta ? __ldg(prm.beta + co) : 0.f) - mean * sc;
                        if (prm.ss_out) prm.ss_out[(size_t)b * pl.C_out + co] = make_float2(sc, sh);
                    }
                    for (int p = 0; p < n_parts; ++p) {
                        int phase, m0, n_valid, n_own = 0;
                        part_geom(p, pl.L_out, phase, m0, n_valid);
                        if (RAGGED) { int ph_, m0_; part_geom(p, L_b, ph_, m0_, n_own); }
                        for (int c0 = 0; c0 < n_valid; c0 += 16) {
                            float v[16];
                            tmem_ld16(tclip + p * pl.n_tile + c0, v);
#pragma unroll
                            for (int i = 0; i < 16; ++i) v[i] = fmaf(v[i], sc, sh);
                            if (RAGGED) {                               // rows [L_b, L_out): zeros (act(0) = 0)
#pragma unroll
                                for (int i = 0; i < 16; ++i) if (c0 + i >= n_own) v[i] = 0.f;
                            }
                            const size_t row0 = (size_t)(m0 + c0) * pl.OS + phase;
#pragma unroll
                            for (int k = 0; k < 2; ++k) {
                                const ActDst& d = k ? prm.dst1 : prm.dst0;
                                if (!d.dtype) continue;
                                const size_t off0 = (size_t)b * d.batch_stride + row0 * d.ld + d.ch_off + co_base;
                                if (d.dtype == PG_DT_F32) {
                                    float a[16];
#pragma unroll
                                    for (int i = 0; i < 16; ++i) a[i] = leaky(v[i], d.slope);
                                    store_f32(static_cast<float*>(d.hi), off0, (size_t)pl.OS * d.ld, a, n_valid - c0);
                                } else {
                                    store_split(d, off0, (size_t)pl.OS * d.ld, v, n_valid - c0);
                                }
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) { if (PAIR) mbar_arrive_leader(accEmpty + acc); else mbar_arrive(accEmpty + acc); }
        }
        if (bad_range) {
            if (prm.dst0.range_flag) atomicOr(prm.dst0.range_flag, 1);
            else if (prm.dst1.range_flag) atomicOr(prm.dst1.range_flag, 1);
        }
    }
    tc_fence_before();
    if (PAIR) cluster_sync_all(); else __syncthreads();      // the peer's shared memory and barriers stay valid until both are done
    if (warp == 1) { tc_fence_after(); if (PAIR) tmem_dealloc_pair(tmem_base, 512); else tmem_dealloc(tmem_base, 512); }
}

// ------------------------------------------------------------------------------------- host
static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

int encode_bf16_map(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                       const uint32_t* box, const char* what) {
    EncodeTiledFn enc = get_encode();
    if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return PG_ERR_CUDA; }
    cuuint64_t d[5], s[5]; cuuint32_t bx[5], es[5];
    for (int i = 0; i < rank; ++i) { d[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) s[i] = strides_bytes[i];
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(base), d, s, bx, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(%s) failed with CUresult %d", what, (int)r); return PG_ERR_CUDA; }
    return PG_OK;
}

// per device (a process may drive several GPUs)
void device_limits(int* sm_count, int* max_smem) {
    static int sm_dev[kMaxDevices] = {}, smem_dev[kMaxDevices] = {};
    const int slot = current_device_slot();
    if (!sm_dev[slot]) {
        int dev = 0; cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sm_dev[slot], cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&smem_dev[slot], cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    }
    *sm_count = sm_dev[slot]; *max_smem = smem_dev[slot];
}

}  // namespace pg

// Can the tensor-core kernel run `mode` as its fused epilogue for this layer?  PG_EPI_NORM_ACT needs every output position
// of a clip inside one tile (<= 512 accumulator columns).  Returns 1 / 0, or a negative error code.
extern "C" int pg_conv_epilogue_supported(const pg_conv_desc* d, int mode) {
    using namespace pg;
    PG_REQUIRE(d, "pg_conv_epilogue_supported: null descriptor");
    if (mode == PG_EPI_RAW) return 1;
    if (mode != PG_EPI_ACT && mode != PG_EPI_NORM_ACT) return 0;
    if (d->precision == PG_PREC_FP32_SIMT || d->C_in % 64 || d->C_out % 128) return 0;
    if (mode == PG_EPI_ACT) return 1;
    pg_conv_desc dd = *d;
    dd.tc_whole_clip = 1;
    ConvPlan pl;
    if (conv_plan_build(&dd, &pl) != PG_OK) return 0;
    return (pl.whole_clip || (pl.OS == 1 && pl.n_ntiles == 1)) ? 1 : 0;
}

static int conv_tc_launch(const pg_conv_desc* d, const uint16_t* x_hi, const uint16_t* x_lo, const uint16_t* w_hi,
                          const uint16_t* w_lo, float* y, float* stats, const pg_conv_epilogue* epi, const int* out_rows,
                          pg_stream stream) {
    using namespace pg;
    const int epi_mode = epi ? epi->mode : PG_EPI_RAW;
    PG_REQUIRE(d && x_hi && w_hi && (y || epi_mode != PG_EPI_RAW), "pg_conv_tc: null pointer");
    PG_REQUIRE(epi_mode == PG_EPI_RAW || epi_mode == PG_EPI_ACT || epi_mode == PG_EPI_NORM_ACT, "pg_conv_tc: bad epilogue mode %d", epi_mode);
    PG_REQUIRE(d->precision >= PG_PREC_BF16X3 && d->precision <= PG_PREC_F16, "pg_conv_tc: precision must be BF16X3, BF16, F16X3, F16X2 or F16");
    const int n_terms = (d->precision == PG_PREC_BF16X3 || d->precision == PG_PREC_F16X3) ? 3 : d->precision == PG_PREC_F16X2 ? 2 : 1;
    const bool three = n_terms == 3;
    PG_REQUIRE(n_terms < 3 || w_lo, "pg_conv_tc: weight lo plane required for the three-product precisions");
    PG_REQUIRE(n_terms < 2 || x_lo, "pg_conv_tc: activation lo plane required for this precision");
    PG_REQUIRE(d->C_in % 64 == 0 && d->C_out % 128 == 0, "pg_conv_tc: needs C_in %% 64 == 0 and C_out %% 128 == 0 (got %d, %d)", d->C_in, d->C_out);
    PG_REQUIRE(d->in_ld % 8 == 0, "pg_conv_tc: input row pitch must be a multiple of 8 elements");
    PG_REQUIRE(d->tc_base_offset_mode == 0, "pg_conv_tc: descriptor base-offset mode 0 is the only supported one (the UMMA swizzle is a "
               "function of the absolute shared-memory address: profiles/r01_tc_probe.log)");
    ConvTcParams prm;
    pg_conv_desc d_local = *d;
    if (const char* e = getenv("PG_TC_PAIR")) d_local.tc_cta_pair = atoi(e);   // A/B hook: 1 = single CTAs, 2 = require pairs
    d_local.tc_whole_clip = epi_mode == PG_EPI_NORM_ACT ? 1 : 0;              // the plan follows the epilogue
    d = &d_local;
    int rc = conv_plan_build(d, &prm.plan);
    if (rc != PG_OK) return rc;
    const ConvPlan& pl = prm.plan;
    prm.epi_mode = epi_mode; prm.gamma = nullptr; prm.beta = nullptr; prm.eps = 1e-5f; prm.ss_out = nullptr;
    prm.clip_rows = out_rows;
    const bool ragged = out_rows != nullptr;
    if ((rc = to_act_dst(nullptr, 0, &prm.dst0, "pg_conv_tc", "dst0")) != PG_OK) return rc;
    prm.dst1 = prm.dst0;
    if (epi_mode != PG_EPI_RAW) {
        PG_REQUIRE(epi_mode != PG_EPI_NORM_ACT || pl.whole_clip || (pl.OS == 1 && pl.n_ntiles == 1),
                   "pg_conv_tc: the fused per-clip norm needs a whole clip per tile (L_out %d does not fit 512 accumulator columns)", pl.L_out);
        if ((rc = to_act_dst(&epi->dst0, d->C_out, &prm.dst0, "pg_conv_tc", "dst0")) != PG_OK) return rc;
        if ((rc = to_act_dst(&epi->dst1, d->C_out, &prm.dst1, "pg_conv_tc", "dst1")) != PG_OK) return rc;
        PG_REQUIRE(prm.dst0.dtype || prm.dst1.dtype, "pg_conv_tc: fused epilogue without a destination");
        for (const ActDst* a : {&prm.dst0, &prm.dst1})        // 128-bit stores of 8 (16-bit) / 4 (fp32) consecutive channels
            PG_REQUIRE(!a->dtype || (a->ld % 8 == 0 && a->ch_off % 8 == 0 && a->batch_stride % 8 == 0 && (reinterpret_cast<uintptr_t>(a->hi) & 15) == 0 &&
                                      (reinterpret_cast<uintptr_t>(a->lo) & 15) == 0),
                       "pg_conv_tc: fused-epilogue destinations need 16-byte aligned planes and ld, ch_off, batch_stride multiples of 8");
        prm.gamma = epi->gamma; prm.beta = epi->beta; prm.eps = epi->eps; prm.ss_out = reinterpret_cast<float2*>(epi->scale_shift);
    } else {
        PG_REQUIRE(d->out_ld % 4 == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0, "pg_conv_tc: y must be 16-byte aligned with out_ld a multiple of 4");
    }
    int g_sm_count, g_max_smem;
    device_limits(&g_sm_count, &g_max_smem);
    prm.y = y; prm.stats = reinterpret_cast<float4*>(stats);
    prm.n_terms = n_terms;
    prm.f16 = (d->precision == PG_PREC_F16X3 || d->precision == PG_PREC_F16X2 || d->precision == PG_PREC_F16) ? 1 : 0;
    prm.base_offset_mode = d->tc_base_offset_mode;
    prm.a_mn = d->weights_mn_major ? 1 : 0;
    const int nb_grp = pl.nb / pl.mgroups;
    const int nb_cta = (pl.pair && pl.merged) ? nb_grp / 2 : nb_grp;
    prm.b_slot_bytes = (pl.merged ? pl.mgroups : (pl.whole_clip ? pl.n_ntiles : 1)) * nb_cta * pl.strip_rows * 128;
    const int a_planes = n_terms == 3 ? 2 : 1, b_planes = n_terms >= 2 ? 2 : 1;
    // merged tiles read up to 15 rows past the last strip (junk columns only): 2 KB of slack keeps that inside the allocation
    const int fixed = 2 * b_planes * prm.b_slot_bytes + 1024 /*alignment slack*/ + 256 /*barriers*/ + 8192 /*epilogue staging tiles*/ +
                      (pl.merged ? 2048 : 0);
    int nA = (g_max_smem - fixed) / (a_planes * kATileBytes);
    if (nA > kMaxASlots) nA = kMaxASlots;
    PG_REQUIRE(nA >= 2, "pg_conv_tc: strip of %d rows leaves no room for the weight ring", pl.strip_rows);
    prm.n_a_slots = nA;
    const size_t smem_bytes = (size_t)fixed + (size_t)nA * a_planes * kATileBytes;

    CUtensorMap mw_hi, mw_lo, mx_hi, mx_lo;
    {
        // weights [tap][C_out][C_in] bf16
        // normal: [tap][C_out][C_in] (K = C_in contiguous); MN-major mode: [tap][C_in][C_out] (M = C_out contiguous)
        const uint64_t inner = prm.a_mn ? d->C_out : d->C_in, outer = prm.a_mn ? d->C_in : d->C_out;
        uint64_t dims[3] = {inner, outer, (uint64_t)d->k};
        uint64_t str[2] = {inner * 2, inner * outer * 2};
        uint32_t box[3] = {64, prm.a_mn ? 64u : 128u, 1};
        if ((rc = encode_bf16_map(&mw_hi, w_hi, 3, dims, str, box, "w_hi")) != PG_OK) return rc;
        if ((rc = encode_bf16_map(&mw_lo, three ? w_lo : w_hi, 3, dims, str, box, "w_lo")) != PG_OK) return rc;
    }
    {
        // activations [B][in_rows][in_ld] viewed as {channel, parity, row / IS, clip}
        const int IS = pl.IS;
        uint64_t dims[4] = {(uint64_t)d->C_in, (uint64_t)IS, (uint64_t)((d->L_in + IS - 1) / IS), (uint64_t)d->B};
        uint64_t str[3] = {(uint64_t)d->in_ld * 2, (uint64_t)d->in_ld * 2 * IS, (uint64_t)d->in_rows * d->in_ld * 2};
        uint32_t box[4] = {64, 1, (uint32_t)pl.strip_rows, (uint32_t)nb_cta};
        PG_REQUIRE(d->in_rows >= ((d->L_in + IS - 1) / IS) * IS, "pg_conv_tc: in_rows %d too small for L_in %d at stride %d", d->in_rows, d->L_in, IS);
        if ((rc = encode_bf16_map(&mx_hi, x_hi, 4, dims, str, box, "x_hi")) != PG_OK) return rc;
        if ((rc = encode_bf16_map(&mx_lo, n_terms >= 2 ? x_lo : x_hi, 4, dims, str, box, "x_lo")) != PG_OK) return rc;
    }
    const bool pair = pl.pair != 0;
    auto kernel = pair ? (ragged ? conv_tc_kernel<true, true> : conv_tc_kernel<true, false>)
                       : (ragged ? conv_tc_kernel<false, true> : conv_tc_kernel<false, false>);
    {
        static size_t configured_dev[kMaxDevices][4] = {};
        const int variant = 2 * pair + ragged;
        size_t* configured = configured_dev[current_device_slot()];
        if (smem_bytes > configured[variant]) {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
            if (e != cudaSuccess) { set_error("conv_tc: cannot opt in to %zu bytes of shared memory: %s", smem_bytes, cudaGetErrorString(e)); return PG_ERR_CUDA; }
            configured[variant] = smem_bytes;
        }
    }
    {
        // clips per L2-resident group: keep ~64 MB of activations hot while every weight slab passes over them
        const int nbg = (pl.B + pl.nb - 1) / pl.nb;
        const double bundle_bytes = (double)pl.nb * d->in_rows * d->in_ld * (n_terms >= 2 ? 4.0 : 2.0);
        int G = (int)(64.0e6 / bundle_bytes);
        if (const char* e = getenv("PG_TC_CLIP_GROUP")) G = atoi(e);   // test hook: force small groups
        if (G < 1) G = 1;
        if (G > nbg) G = nbg;
        prm.plan.clip_group = G;
    }
    const int n_tiles = (pair ? pl.n_cotiles / 2 : pl.n_cotiles) * ((pl.B + pl.nb - 1) / pl.nb) * (pl.whole_clip ? 1 : pl.OS * pl.n_ntiles);
    int units = pair ? g_sm_count / 2 : g_sm_count;           // persistent CTAs (or CTA pairs: one per TPC)
    if (const char* e = getenv("PG_TC_MAX_CTAS")) {           // experiment hook: leave SMs free (e.g. for NCCL)
        const int cap = atoi(e);
        if (cap > 0 && units > (pair ? cap / 2 : cap)) units = pair ? cap / 2 : cap;
    }
    if (d->tc_max_ctas > 0 && units > (pair ? (d->tc_max_ctas + 1) / 2 : d->tc_max_ctas)) units = pair ? (d->tc_max_ctas + 1) / 2 : d->tc_max_ctas;
    if (units > n_tiles) units = n_tiles;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(pair ? 2 * units : units);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = reinterpret_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = pair ? 2 : 1; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaError_t le = cudaLaunchKernelEx(&cfg, kernel, mw_hi, mw_lo, mx_hi, mx_lo, prm);
    if (le != cudaSuccess) { set_error("conv_tc_kernel launch failed: %s", cudaGetErrorString(le)); return PG_ERR_CUDA; }
    return check_launch("conv_tc_kernel");
}

extern "C" int pg_conv_tc(const pg_conv_desc* d, const uint16_t* x_hi, const uint16_t* x_lo, const uint16_t* w_hi,
                          const uint16_t* w_lo, float* y, float* stats, const pg_conv_epilogue* epi, pg_stream stream) {
    return conv_tc_launch(d, x_hi, x_lo, w_hi, w_lo, y, stats, epi, nullptr, stream);
}

extern "C" int pg_conv_tc_ragged(const pg_conv_desc* d, const uint16_t* x_hi, const uint16_t* x_lo, const uint16_t* w_hi,
                                 const uint16_t* w_lo, float* y, float* stats, const pg_conv_epilogue* epi, const int* out_rows,
                                 pg_stream stream) {
    PG_REQUIRE(out_rows, "pg_conv_tc_ragged: null per-clip row table");
    return conv_tc_launch(d, x_hi, x_lo, w_hi, w_lo, y, stats, epi, out_rows, stream);
}
