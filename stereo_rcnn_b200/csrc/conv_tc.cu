// conv_tc.cu -- implicit-GEMM convolution on tcgen05 tensor cores (sm_100a only).
//
// The dense contractions of the Stereo R-CNN forward -- every 1x1 / 3x3 convolution of the
// ResNet-101 trunk, FPN, RPN, the 25088->2048 box-head FC, the keypoint-head convs and the
// 2x2 deconv (as four 1x1s) -- run through this one kernel:
//
//   D[M = output pixels, N = Cout] = sum over taps (r,s) and Cin chunks of
//        A[(pixel shifted by tap), Cin chunk] * W[Cout, tap, Cin chunk]^T
//
//   * operands are fp16 in HBM by default (in_dtype 1: NHWC activations, [Cout][kh][kw][Cin] weights, both rounded
//     to nearest once by their producer) and feed `tcgen05.mma.kind::f16`; the fp32 / `kind::tf32` mode (in_dtype 0,
//     the tensor core reads the top 19 bits) is kept for comparison.  Accumulation is fp32 in TMEM either way; the
//     exact-fp32 SIMT kernel (conv_simt.cu) is the yardstick.
//   * TMA moves every operand tile: weights through a 2-D map, activations through a 2-D map (1x1: pixels are rows
//     of a flat [M, Cin] matrix) or a 4-D [C, W, H, N] map (3x3: an 8x16 pixel patch per tile; the tap shift is a
//     coordinate offset and the hardware zero-fills the padding halo, so im2col never exists in memory).  128-byte
//     swizzle, 1024-byte aligned stages, one 128-byte row (64 fp16 / 32 fp32 = one K-step) per pixel per stage.
//   * warp-specialised persistent CTAs (one per SM): warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane)
//     + TMEM allocator, warps 2..9 = epilogue (two warps per TMEM lane quarter, each taking half of the tile's
//     columns).  Three mbarrier pipelines: smem full/empty (4 stages of 48 KB for 256-wide tiles, 6 of 32 KB for
//     128-wide ones -- the main loop is bound by bytes in flight, so nearly all shared memory is operand stages),
//     TMEM full/empty (two accumulator stages: the epilogue of tile i overlaps the main loop of tile i+1).
//   * fused epilogue out of TMEM (`tcgen05.ld.32x32b.x32`): folded frozen-BN scale/shift or bias, residual add
//     (rows prefetched into registers across tile boundaries and into L2 with cp.async.bulk.prefetch two tiles
//     ahead), FPN bilinear (align_corners) upsample-add, ReLU, fp32 and/or fp16 ("twin") stores with arbitrary
//     n/h/w strides and channel offset (RPN L|R concat, deconv scatter).  See the epilogue's own comment block.
//   * programmatic dependent launch: the prologue (barrier init, TMEM alloc, descriptor prefetch) overlaps the
//     previous kernel's tail; dependents are released after the CTA's last MMAs.
//   * optional per-CTA phase trace (sb_conv_trace) for tools/conv_trace.py.
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace {

constexpr int TW = 16, TH = 8;  // spatial patch of a 3x3 tile (TW*TH == BLOCK_M)
// epilogue warps per CTA: 8 (one big CTA per SM) or 4 ("small" variant: two CTAs per SM for layers with few tiles)
constexpr int kMaxCout = 2048;   // scale/shift staged in shared memory

// ------------------------------------------------------------------ kernel
constexpr size_t epi_smem(int ew) { return (size_t)ew * (32 * 8 * 16); }

struct TcParams {
    sb_conv_desc d;
    int patch;            // 0: flat [M,Cin] rows (1x1), 1: 8x16 spatial patches (3x3 / pad 1)
    int tiles_w, tiles_h; // patch mode
    int num_m_tiles, num_n_tiles;
    int kblocks_per_tap;  // Cin / 32
    int num_k_blocks;     // taps * kblocks_per_tap
    long long M;
    int pdl_late;         // fire griddepcontrol.launch_dependents after the last tile's MMAs instead of at entry
    int cg2_direct;       // CTA pairs: the peer's TMA loads signal the LEADER's full barrier directly (no forwarding warp)
    unsigned long long* trace;   // optional per-CTA phase timestamps (sb_conv_trace), 16 words per CTA
};

__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t) :: "memory");
    return t;
}
constexpr int kTraceWords = 16, kTraceCtas = 304;

// CG2 (CTA pairs, `tcgen05.mma.cta_group::2`): the two CTAs of a 2-cluster compute two vertically adjacent 128-row
// tiles against the SAME 256-wide weight tile; each CTA loads its own A tile and HALF of the weight tile (128 rows),
// the leader (cluster rank 0) issues M = 256 MMAs that read both CTAs' shared memory and write each CTA's own TMEM.
// Per SM and K-step that is 32 KB of operands for 512 MMA cycles (62 B/clk) instead of 48 KB (94 B/clk, above the
// ~80 B/clk an SM ingests from L2): the 256-wide 3x3 convs become MMA-bound.  Barrier protocol on top of the
// single-CTA one: the peer's warp 1 forwards "my stage is full" to the leader (remote mbarrier arrive), the leader's
// commits are multicast to both CTAs' empty / tfull barriers, the peer's epilogue warps release the accumulator
// stage on the leader's tempty barrier; cluster barriers fence set-up and tear-down.
template <int BLOCK_N, int kStages, bool HAS_RES, bool HAS_UP, bool IN16, int EW, bool CG2 = false>
__global__ void __launch_bounds__(64 + 32 * EW, EW == 4 ? 2 : 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
               const TcParams p) {
    static_assert(!CG2 || (BLOCK_N == 256 && IN16 && !HAS_RES && !HAS_UP && EW == 8), "CTA-pair variant");
    constexpr uint32_t kABytes = BLOCK_M * kRowBytes, kBBytes = (CG2 ? BLOCK_N / 2 : BLOCK_N) * kRowBytes;
    constexpr int BLOCK_K = IN16 ? 64 : 32;     // elements per K-step
    constexpr uint32_t kStageBytes = kABytes + kBBytes;
    constexpr uint32_t kTmemCols = (2 * BLOCK_N <= 32) ? 32 : (2 * BLOCK_N <= 64) ? 64 : (2 * BLOCK_N <= 128) ? 128
                                   : (2 * BLOCK_N <= 256) ? 256 : 512;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
    uint64_t* empty = full + kStages;
    uint64_t* tfull = empty + kStages;
    uint64_t* tempty = tfull + 2;
    uint64_t* pfull = tempty + 2;              // CG2, leader: "the peer's stage is full" (remote arrivals)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pfull + (CG2 ? kStages : 0));
    float4* epi_stage = reinterpret_cast<float4*>(smem + kStages * kStageBytes + 256);   // [EW warps][32 rows][8 float4]
    static_assert(((CG2 ? 3 : 2) * kStages + 4) * 8 + 16 <= 256, "barrier block");

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const sb_conv_desc& d = p.d;
    const uint32_t crank = CG2 ? cluster_ctarank() : 0u;      // 0 = leader
    unsigned long long* tr = p.trace ? p.trace + (size_t)blockIdx.x * kTraceWords : nullptr;
    if (tr && threadIdx.x == 0) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        tr[0] = gtimer(); tr[8] = clock64(); tr[6] = smid;
    }

    if (warp == 0 && elect_one()) {
        prefetch_tmap(&map_a);
        prefetch_tmap(&map_b);
    }
    if (warp == 1) {
        if (elect_one()) {
            for (int i = 0; i < kStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
            for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], CG2 ? 2 * EW : EW); }
            if (CG2) for (int i = 0; i < kStages; ++i) mbar_init(&pfull[i], 1);
            fence_barrier_init();
        }
        __syncwarp();
        if (CG2) {      // one warp of EACH CTA of the pair takes part in the pair-wide allocation
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                         "r"(kTmemCols));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                         "r"(kTmemCols));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
        }
    }
    tc_fence_before();
    if (CG2) cluster_sync_all();     // barriers of BOTH CTAs are initialised before any remote arrive / multicast commit
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor prefetch,
    // scale/shift staging -- weights only) overlapped the previous kernel's tail.  Let the next kernel start
    // its own prologue as soon as our CTAs retire, then wait for the producers of our activations.
    if (!p.pdl_late) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (tr && threadIdx.x == 0) { tr[1] = gtimer(); tr[9] = clock64(); }

    // CG2: a "tile" of the loops below is a PAIR of row tiles (2q, 2q+1) x one 256-wide column tile, one pair per
    // cluster; this CTA owns row tile 2q + crank (past the end for an odd count: loads zero-fill, stores are masked)
    const int num_tiles = CG2 ? ((p.num_m_tiles + 1) >> 1) * p.num_n_tiles : p.num_m_tiles * p.num_n_tiles;
    const int tile0 = CG2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int tstep = CG2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    auto row_tile = [&](int tile) { const int q = tile / p.num_n_tiles; return CG2 ? 2 * q + (int)crank : q; };

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (elect_one()) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = tile0; tile < num_tiles; tile += tstep) {
                const int mt = row_tile(tile), nt = tile % p.num_n_tiles;
                int n_img = 0, h0 = 0, w0 = 0;
                if (p.patch) {
                    const int tw = mt % p.tiles_w;
                    const int t2 = mt / p.tiles_w;
                    h0 = (t2 % p.tiles_h) * TH;
                    n_img = t2 / p.tiles_h;
                    w0 = tw * TW;
                }
                for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                    const int tap = kb / p.kblocks_per_tap;
                    const int c0 = (kb - tap * p.kblocks_per_tap) * BLOCK_K;
                    mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * kStageBytes;
                    uint8_t* sb = sa + kABytes;
                    if (CG2 && p.cg2_direct) {
                        // all four loads of the pair complete on the LEADER's barrier (patch mode only)
                        const uint32_t lbar = mapa_rank(smem_u32(&full[stage]), 0);
                        if (crank == 0) mbar_expect_tx(&full[stage], 2 * kStageBytes);
                        const int r = tap / d.kw, s = tap - r * d.kw;
                        tma_load_4d_pair(&map_a, lbar, sa, c0, w0 + s - d.pad, h0 + r - d.pad, n_img);
                        tma_load_2d_pair(&map_b, lbar, sb, tap * d.Cin + c0, nt * BLOCK_N + (int)crank * (BLOCK_N / 2));
                        if (++stage == kStages) { stage = 0; phase ^= 1; }
                        continue;
                    }
                    mbar_expect_tx(&full[stage], kStageBytes);
                    if (p.patch) {
                        const int r = tap / d.kw, s = tap - r * d.kw;
                        tma_load_4d(&map_a, &full[stage], sa, c0, w0 + s - d.pad, h0 + r - d.pad, n_img);
                    } else {
                        tma_load_2d(&map_a, &full[stage], sa, c0, mt * BLOCK_M);
                    }
                    // CG2: this CTA's half (128 rows) of the pair's 256-row weight tile
                    tma_load_2d(&map_b, &full[stage], sb, tap * d.Cin + c0, nt * BLOCK_N + (CG2 ? (int)crank * (BLOCK_N / 2) : 0));
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1 && CG2 && crank != 0) {
        // ===================== peer CTA: forward "stage full" to the leader =====================
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = tile0; tile < num_tiles && !p.cg2_direct; tile += tstep) {
            for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                mbar_wait(&full[stage], phase);                       // my A tile and my half of the weights have landed
                if (lane == 0) mbar_arrive_remote(mapa_rank(smem_u32(&pfull[stage]), 0));
                __syncwarp();
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
        }
        if (p.pdl_late) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        if (tr && lane == 0) { tr[3] = gtimer(); tr[11] = clock64(); }
    } else if (warp == 1) {
        // ===================== MMA issuer (CG2: leader CTA only) =====================
        constexpr uint32_t idesc = CG2 ? make_idesc_2cta(BLOCK_N, IN16) : make_idesc(BLOCK_N, IN16);
        int stage = 0;
        uint32_t phase = 0;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int tile = tile0; tile < num_tiles; tile += tstep) {
            if (CG2) mbar_wait_cluster(&tempty[acc], acc_phase ^ 1);    // released by the epilogues of BOTH CTAs
            else mbar_wait(&tempty[acc], acc_phase ^ 1);
            tc_fence_after();
            const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
            for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                if (CG2 && p.cg2_direct) mbar_wait_cluster(&full[stage], phase);    // completed by both CTAs' loads
                else mbar_wait(&full[stage], phase);
                if (CG2 && !p.cg2_direct) mbar_wait_cluster(&pfull[stage], phase);
                tc_fence_after();
                if (tr && lane == 0 && kb == 0 && tile == tile0) { tr[2] = gtimer(); tr[10] = clock64(); }
                if (elect_one()) {
                    const uint32_t sa = smem_u32(smem + stage * kStageBytes);
                    const uint64_t da = make_smem_desc(sa), db = make_smem_desc(sa + kABytes);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        // advance 32 bytes (8 tf32) inside the 128-byte swizzle row: +2 in 16-byte units
                        if (CG2) umma_f16_2cta(tmem_d, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) != 0);
                        else if (IN16) umma_f16(tmem_d, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) != 0);
                        else umma_tf32(tmem_d, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) != 0);
                    }
                    if (CG2) {
                        umma_commit_2cta(&empty[stage]);                  // frees the slot in BOTH CTAs
                        if (kb == p.num_k_blocks - 1) umma_commit_2cta(&tfull[acc]);
                    } else {
                        umma_commit(&empty[stage]);                       // frees the smem slot when the MMAs retire
                        if (kb == p.num_k_blocks - 1) umma_commit(&tfull[acc]);  // accumulator complete
                    }
                }
                __syncwarp();
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (p.pdl_late) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        if (tr && lane == 0) { tr[3] = gtimer(); tr[11] = clock64(); }
    } else {
        // ===================== epilogue (warps 2..9) =====================
        // warp w may only touch TMEM lanes 32*(w%4)..+31; two warps share each lane quarter and split the
        // tile's columns in halves.  Per 32-column chunk: TMEM -> registers (one accumulator row per thread)
        // -> XOR-swizzled per-warp staging tile in shared memory -> read back transposed, so that every global
        // access of the warp covers four full 128-byte rows and each lane owns four fixed channels: scale /
        // shift are two register float4 per chunk.  The epilogue is latency / issue bound, so row addressing
        // is hoisted to once per tile (exchanged through the idle staging tile: shared memory is spent on
        // operand stages, the main loop being bound by bytes in flight), the residual rows are prefetched two
        // chunks ahead -- across tile boundaries -- and the bilinear taps of the FPN upsample-add are issued
        // four rows at a time before they are consumed.
        const int q = warp & 3;
        const int ew = warp - 2;
        // EW / 4 warps share each TMEM lane quarter and split the tile's columns between them.  EW = 16 is the
        // variant for epilogue-bound convs (few K-steps per tile): four warps per scheduler hide each other's
        // latencies, at 112 registers per thread -- so it reads the residual where it is used (L2 hits, thanks to
        // the bulk prefetch) instead of through the 64-register prefetch ring.
        constexpr int kParts = EW / 4;
        const int half = ew >> 2;          // which column part this warp owns (0 for EW = 4)
        constexpr int kColsPerWarp = BLOCK_N / kParts >= 32 ? BLOCK_N / kParts : 32;
        constexpr bool kResRing = HAS_RES && EW <= 8;
        constexpr int kChunks = kColsPerWarp / 32;
        const int col_begin = half * kColsPerWarp;
        const bool has_cols = col_begin < BLOCK_N;
        const uint32_t stg = smem_u32(epi_stage + ew * (32 * 8));      // this warp's 4 KB staging tile (shared-space address)
        int acc = 0;
        uint32_t acc_phase = 0;
        float rh = 0.f, rw = 0.f;
        if (HAS_UP) {
            rh = d.Ho > 1 ? __fdiv_rn((float)(d.UH - 1), (float)(d.Ho - 1)) : 0.f;
            rw = d.Wo > 1 ? __fdiv_rn((float)(d.UW - 1), (float)(d.Wo - 1)) : 0.f;
        }
        const int rsub = lane >> 3, c4 = lane & 7;
        const bool relu = d.relu != 0;
        const int out_mode = d.out_mode;
        const bool res_biased = d.res_biased != 0;
        // residual rows (HAS_RES implies a 1x1 conv, i.e. flat rows: row m of the output is row m of the residual)
        float4 r4[2][8];
        const float* rbase = nullptr;     // residual row of this lane's first row (rows 4*i+rsub are 4*res_ld apart)
        int rrows = 0;                    // how many of the lane's 8 rows exist (m < M)
        const long long rstep = 4ll * d.res_ld;
        bool prefetched = false;      // r4 already holds the first chunks of the tile about to be processed
        auto res_rows = [&](int mt_) {
            const long long m0 = (long long)mt_ * BLOCK_M + q * 32 + rsub;
            const long long left = p.M - m0;                     // rows m0, m0+4, ... < M
            rrows = left <= 0 ? 0 : (left >= 32 ? 8 : (int)((left + 3) >> 2));
            rbase = d.residual + (left <= 0 ? 0 : m0) * d.res_ld + 4 * c4;
        };
        // folded-BN scale / shift (or bias) of the lane's four channels, fetched one chunk ahead
        float4 sc_n = make_float4(1.f, 1.f, 1.f, 1.f), sh_n = make_float4(0.f, 0.f, 0.f, 0.f);
        auto load_scale_shift = [&](int cidx) {
            const bool ok = cidx < d.Cout;
            sc_n = (d.scale && ok) ? __ldg(reinterpret_cast<const float4*>(d.scale + cidx)) : make_float4(1.f, 1.f, 1.f, 1.f);
            sh_n = (d.shift && ok) ? __ldg(reinterpret_cast<const float4*>(d.shift + cidx)) : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        auto load_res = [&](int buf, int cbase) {
            const int live = (cbase + 4 * c4 < d.Cout) ? rrows : 0;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                r4[buf][i] = (i < live) ? __ldg(reinterpret_cast<const float4*>(rbase + i * rstep + cbase))
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        // Residual rows of a tile two ahead are pulled into L2 with a bulk prefetch (one row segment per lane): in
        // layers 1-2 the residual stream lives in HBM, and the register prefetch alone keeps too few bytes in
        // flight (64 KB per SM against a ~2 us DRAM round trip) to fill the memory pipe.
        auto prefetch_res_tile = [&](int t) {
            if (t >= num_tiles) return;
            const int pmt = t / p.num_n_tiles, pnt = t - pmt * p.num_n_tiles;
            const long long m = (long long)pmt * BLOCK_M + q * 32 + lane;
            const int c0 = pnt * BLOCK_N + col_begin;
            if (m < p.M && c0 < d.Cout) {
                const int ncols = min(kColsPerWarp, d.Cout - c0);
                prefetch_l2_bulk(d.residual + m * d.res_ld + c0, (uint32_t)ncols * 4u);
            }
        };
        if (HAS_RES && has_cols) prefetch_res_tile(blockIdx.x + gridDim.x);
        for (int tile = tile0; tile < num_tiles; tile += tstep) {
            const int mt = row_tile(tile), nt = tile % p.num_n_tiles;
            if (HAS_RES && has_cols) prefetch_res_tile(tile + 2 * gridDim.x);
            unsigned ooff[8];          // element offsets < 2^31 (checked on the host)
            unsigned vmask = 0;
            int uoff[8];
            float uly[8], ulx[8];
            unsigned fy = 0, fx = 0;
            {   // this lane describes accumulator row q*32+lane of the tile
                const int row = q * 32 + lane;
                int n_img, ho, wo;
                bool valid;
                if (p.patch) {
                    const int tw = mt % p.tiles_w;
                    const int t2 = mt / p.tiles_w;
                    ho = (t2 % p.tiles_h) * TH + row / TW;
                    wo = tw * TW + row % TW;
                    n_img = t2 / p.tiles_h;
                    valid = ho < d.Ho && wo < d.Wo && n_img < d.N;      // (n_img >= N: the pad tile of an odd CTA pair)
                } else {
                    const long long m = (long long)mt * BLOCK_M + row;
                    valid = m < p.M;
                    const unsigned mm = valid ? (unsigned)m : 0u;      // M < 2^31 (checked on the host)
                    const unsigned hw = (unsigned)(d.Ho * d.Wo);
                    n_img = (int)(mm / hw);
                    const unsigned rem = mm - (unsigned)n_img * hw;
                    ho = (int)(rem / (unsigned)d.Wo);
                    wo = (int)(rem - (unsigned)ho * (unsigned)d.Wo);
                }
                // one 16-byte record per row {output offset, upsample source offset, ly1, lx1} goes through the
                // (idle) staging tile; the three per-row flags travel as ballots
                const long long out_off = (long long)n_img * d.out_n_stride + (long long)ho * d.out_h_stride +
                                          (long long)wo * d.out_w_stride + d.out_coff;
                uint4 rec = make_uint4((unsigned)out_off, 0u, 0u, 0u);
                bool by = false, bx = false;
                if (HAS_UP && valid) {
                    const float sy = __fmul_rn(rh, (float)ho), sx = __fmul_rn(rw, (float)wo);
                    const int y1 = (int)sy, x1 = (int)sx;
                    by = y1 < d.UH - 1;
                    bx = x1 < d.UW - 1;
                    rec.y = (unsigned)((((long long)n_img * d.UH + y1) * d.UW + x1) * d.Cout);
                    rec.z = __float_as_uint(sy - (float)y1);
                    rec.w = __float_as_uint(sx - (float)x1);
                }
                const unsigned bal_v = __ballot_sync(0xffffffffu, valid);
                const unsigned bal_y = HAS_UP ? __ballot_sync(0xffffffffu, by) : 0u;
                const unsigned bal_x = HAS_UP ? __ballot_sync(0xffffffffu, bx) : 0u;
                sts128u(stg + lane * 16, rec);          // (the previous tile's staging reads ended with a __syncwarp)
                __syncwarp();
                // rows this lane touches in the coalesced domain: 4*i + rsub, i = 0..7
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = 4 * i + rsub;
                    const uint4 o = lds128u(stg + r * 16);
                    ooff[i] = o.x + 4u * c4 + (unsigned)(nt * BLOCK_N + col_begin);     // + the warp's first column
                    vmask |= ((bal_v >> r) & 1u) << i;
                    if (HAS_UP) {
                        uoff[i] = (int)o.y;
                        uly[i] = __uint_as_float(o.z);
                        ulx[i] = __uint_as_float(o.w);
                        fy |= ((bal_y >> r) & 1u) << i;
                        fx |= ((bal_x >> r) & 1u) << i;
                    }
                }
                __syncwarp();           // staging tile free again
            }
            const int cb0 = nt * BLOCK_N + col_begin;
            if (HAS_RES && !kResRing && has_cols) res_rows(mt);
            if (kResRing && has_cols && !prefetched) {
                // the first tile's residual rows are requested before its accumulator is complete, so their
                // latency hides behind the MMA main loop
                res_rows(mt);
                load_res(0, cb0);
                if (kChunks > 1) load_res(1, cb0 + 32);
            }
            if (has_cols) load_scale_shift(cb0 + 4 * c4);      // chunk 0's: in flight while the accumulator completes
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            if (has_cols) {
                // Each chunk runs in straight-line phases over the lane's 8 row quads (loads, math, stores): with
                // two epilogue warps per scheduler there is nothing else to hide latency behind, so the
                // instruction-level parallelism has to come from inside the warp (no per-row branches).
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BLOCK_N + col_begin);
                uint32_t v[32];
                tmem_ld32(taddr, v);
                constexpr int kUnroll = HAS_UP ? 1 : kChunks;      // (the upsample-add chunk body is register-bound: keep chunks apart)
#pragma unroll kUnroll
                for (int k = 0; k < kChunks; ++k) {
                    const int cbase = nt * BLOCK_N + col_begin + 32 * k;
                    const int cidx = cbase + 4 * c4;
                    const bool col_ok = cidx < d.Cout;
                    const unsigned live = col_ok ? vmask : 0u;
                    const float4 sc = sc_n, sh = sh_n;
                    if (k + 1 < kChunks) load_scale_shift(cb0 + 32 * (k + 1) + 4 * c4);      // for the next chunk
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        sts128(stg + (lane * 8 + (j ^ (lane & 7))) * 16,
                               make_float4(__uint_as_float(v[4 * j + 0]), __uint_as_float(v[4 * j + 1]),
                                           __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3])));
                    __syncwarp();
                    // the next chunk's accumulator columns travel TMEM -> registers while this chunk is finished
                    constexpr bool kEarlyLd = !HAS_RES && !HAS_UP && EW <= 8;   // the other variants have no registers to spare
                    if (kEarlyLd && k + 1 < kChunks) tmem_ld32(taddr + 32 * (k + 1), v);
                    // rows per pass: the upsample-add variant keeps 16 tap registers per row pair, so it walks the
                    // lane's 8 row quads in two passes of 4 to stay inside the register file
                    constexpr int XR = HAS_UP ? 4 : 8;
#pragma unroll
                    for (int pass = 0; pass < 8 / XR; ++pass) {
                        float4 x[XR];
#pragma unroll
                        for (int ii = 0; ii < XR; ++ii) {
                            const int r = 4 * (pass * XR + ii) + rsub;
                            x[ii] = lds128(stg + (r * 8 + (c4 ^ (r & 7))) * 16);
                        }
#pragma unroll
                        for (int ii = 0; ii < XR; ++ii) {
                            x[ii].x = fmaf(x[ii].x, sc.x, sh.x); x[ii].y = fmaf(x[ii].y, sc.y, sh.y);
                            x[ii].z = fmaf(x[ii].z, sc.z, sh.z); x[ii].w = fmaf(x[ii].w, sc.w, sh.w);
                        }
                        if (HAS_RES) {
                            if (kResRing && res_biased) {
#pragma unroll
                                for (int ii = 0; ii < XR; ++ii) {
                                    float4& rr = r4[k & 1][pass * XR + ii];
                                    rr.x = sb_unbias_tf32(rr.x); rr.y = sb_unbias_tf32(rr.y);
                                    rr.z = sb_unbias_tf32(rr.z); rr.w = sb_unbias_tf32(rr.w);
                                }
                            }
#pragma unroll
                            for (int ii = 0; ii < XR; ++ii) {
                                float4 rr;
                                if (kResRing) {
                                    rr = r4[k & 1][pass * XR + ii];
                                } else {
                                    const int i = pass * XR + ii;
                                    rr = (col_ok && i < rrows) ? __ldg(reinterpret_cast<const float4*>(rbase + i * rstep + cbase))
                                                               : make_float4(0.f, 0.f, 0.f, 0.f);
                                    if (res_biased) {
                                        rr.x = sb_unbias_tf32(rr.x); rr.y = sb_unbias_tf32(rr.y);
                                        rr.z = sb_unbias_tf32(rr.z); rr.w = sb_unbias_tf32(rr.w);
                                    }
                                }
                                x[ii].x += rr.x; x[ii].y += rr.y; x[ii].z += rr.z; x[ii].w += rr.w;
                            }
                        }
                        if (HAS_UP) {
                            const float* ubase = d.up_src + (col_ok ? cidx : 0);
                            const long long ustep_y = (long long)d.UW * d.Cout;
                            constexpr int UB = 2;                     // rows per batch: 4 * UB independent tap loads in flight
#pragma unroll
                            for (int hh = 0; hh < XR / UB; ++hh) {
                                float4 ta[UB], tb[UB], tg[UB], th[UB];
#pragma unroll
                                for (int jj = 0; jj < UB; ++jj) {
                                    const int i = pass * XR + hh * UB + jj;
                                    const float* u00 = ubase + uoff[i];
                                    const long long dx = ((fx >> i) & 1u) ? d.Cout : 0;
                                    const long long dy = ((fy >> i) & 1u) ? ustep_y : 0;
                                    ta[jj] = __ldg(reinterpret_cast<const float4*>(u00));
                                    tb[jj] = __ldg(reinterpret_cast<const float4*>(u00 + dx));
                                    tg[jj] = __ldg(reinterpret_cast<const float4*>(u00 + dy));
                                    th[jj] = __ldg(reinterpret_cast<const float4*>(u00 + dy + dx));
                                }
#pragma unroll
                                for (int jj = 0; jj < UB; ++jj) {
                                    const int ii = hh * UB + jj, i = pass * XR + ii;
                                    const float4 a = ta[jj], bq = tb[jj], g = tg[jj], h = th[jj];
                                    const float ly1 = uly[i], ly0 = 1.f - ly1, lx1 = ulx[i], lx0 = 1.f - lx1;
                                    x[ii].x += ly0 * (lx0 * a.x + lx1 * bq.x) + ly1 * (lx0 * g.x + lx1 * h.x);
                                    x[ii].y += ly0 * (lx0 * a.y + lx1 * bq.y) + ly1 * (lx0 * g.y + lx1 * h.y);
                                    x[ii].z += ly0 * (lx0 * a.z + lx1 * bq.z) + ly1 * (lx0 * g.z + lx1 * h.z);
                                    x[ii].w += ly0 * (lx0 * a.w + lx1 * bq.w) + ly1 * (lx0 * g.w + lx1 * h.w);
                                }
                            }
                        }
                        if (relu) {
#pragma unroll
                            for (int ii = 0; ii < XR; ++ii) {
                                x[ii].x = fmaxf(x[ii].x, 0.f); x[ii].y = fmaxf(x[ii].y, 0.f);
                                x[ii].z = fmaxf(x[ii].z, 0.f); x[ii].w = fmaxf(x[ii].w, 0.f);
                            }
                        }
                        if (out_mode == 1) {
#pragma unroll
                            for (int ii = 0; ii < XR; ++ii) {
                                x[ii].x = sb_round_tf32(x[ii].x); x[ii].y = sb_round_tf32(x[ii].y);
                                x[ii].z = sb_round_tf32(x[ii].z); x[ii].w = sb_round_tf32(x[ii].w);
                            }
                        } else if (out_mode == 2) {
#pragma unroll
                            for (int ii = 0; ii < XR; ++ii) {
                                x[ii].x = sb_bias_tf32(x[ii].x); x[ii].y = sb_bias_tf32(x[ii].y);
                                x[ii].z = sb_bias_tf32(x[ii].z); x[ii].w = sb_bias_tf32(x[ii].w);
                            }
                        }
                        if (d.out) {
#pragma unroll
                            for (int ii = 0; ii < XR; ++ii) {
                                const int i = pass * XR + ii;
                                if ((live >> i) & 1u) *reinterpret_cast<float4*>(d.out + ooff[i] + 32 * k) = x[ii];
                            }
                        }
                        if (d.out16) {   // fp16 twin (round to nearest) for the next tensor-core consumer
                            if (out_mode == 2) {
#pragma unroll
                                for (int ii = 0; ii < XR; ++ii) {
                                    x[ii].x = sb_unbias_tf32(x[ii].x); x[ii].y = sb_unbias_tf32(x[ii].y);
                                    x[ii].z = sb_unbias_tf32(x[ii].z); x[ii].w = sb_unbias_tf32(x[ii].w);
                                }
                            }
#pragma unroll
                            for (int ii = 0; ii < XR; ++ii) {
                                const int i = pass * XR + ii;
                                __half2 lo = __floats2half2_rn(x[ii].x, x[ii].y);
                                __half2 hi = __floats2half2_rn(x[ii].z, x[ii].w);
                                uint2 pk;
                                pk.x = *reinterpret_cast<uint32_t*>(&lo);
                                pk.y = *reinterpret_cast<uint32_t*>(&hi);
                                if ((live >> i) & 1u)
                                    *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(d.out16) + ooff[i] + 32 * k) = pk;
                            }
                        }
                    }
                    __syncwarp();
                    if (kResRing) {
                        // buffer k&1 is free: refill it with the chunk two ahead in the CTA's chunk sequence --
                        // of this tile, or of the CTA's next tile (whose accumulator is still being computed)
                        if (k + 2 < kChunks) {
                            load_res(k & 1, cb0 + 32 * (k + 2));
                        } else {
                            const int ntile = tile + gridDim.x;
                            const int nk = kChunks == 1 ? 0 : k + 2 - kChunks;
                            if (ntile < num_tiles) {
                                const int nmt = ntile / p.num_n_tiles, nnt = ntile - nmt * p.num_n_tiles;
                                if (nk == 0) res_rows(nmt);      // rbase / rrows now describe the next tile
                                load_res(kChunks == 1 ? 0 : (k & 1), nnt * BLOCK_N + col_begin + 32 * nk);
                                prefetched = true;
                            } else {
                                prefetched = false;
                            }
                        }
                    }
                    if (!kEarlyLd && k + 1 < kChunks) tmem_ld32(taddr + 32 * (k + 1), v);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                // CG2: the accumulator stage of the PAIR is free when the epilogue warps of both CTAs are done with it;
                // the barrier the MMA warp waits on lives in the leader
                if (CG2 && crank != 0) mbar_arrive_remote(mapa_rank(smem_u32(&tempty[acc]), 0));
                else mbar_arrive(&tempty[acc]);
            }
            if (tr && warp == 2 && lane == 0 && tile == tile0) { tr[4] = gtimer(); tr[12] = clock64(); }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }

    tc_fence_before();
    if (CG2) cluster_sync_all();      // neither CTA may retire (or free TMEM) while the other can still reach into it
    else __syncthreads();
    if (tr && threadIdx.x == 0) { tr[5] = gtimer(); tr[13] = clock64(); }
    if (warp == 1) {
        tc_fence_after();
        if (CG2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols));
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols));
    }
}

// ------------------------------------------------------------------ flat (1x1) kernel with a TMA epilogue
// The 1x1 convolutions of the bottlenecks -- conv1, conv3 (+ residual), the downsample branch -- the stem GEMM, the
// box-head FCs and the RPN head are plain [M, Cin] x [Cin, Cout] GEMMs with dense [M, Cout] outputs and only 1-32
// K-steps per tile: their time is the epilogue.  This kernel keeps the producer / MMA-issuer warps of the generic
// kernel above and replaces the epilogue by one in which global memory is touched by TMA only:
//   * each epilogue warp owns a 32-row x 32-column box of the tile per step ("chunk"); the accumulator chunk comes
//     out of TMEM with one tcgen05.ld (one row per thread), which is already the layout of a 128-byte-swizzled TMA
//     box: row r of the box is 128 contiguous bytes, its 16-byte groups XOR-permuted by (r & 7) -- conflict-free for
//     the row-per-thread 128-bit accesses, no transposition through shared memory;
//   * the residual box arrives by TMA load into a warp-private ring (three boxes: one being consumed, two in
//     flight -- issued two chunks ahead, across tile boundaries, before the accumulator is complete), the result
//     overwrites it in place and leaves by TMA store; the fp16 twin leaves through a 64-byte-swizzled half box;
//   * no address arithmetic, predicates or global LD/ST in the warps: M and Cout tails are clipped / zero-filled
//     by the tensor maps.  Buffer reuse is ordered by cp.async.bulk.wait_group.read, not by barriers between warps.
struct FlatParams {
    const float* scale;
    const float* shift;
    const float* residual;    // for the L2 bulk prefetch two tiles ahead (the data path goes through map_res)
    long long M;
    int Cout, res_ld;
    int num_m_tiles, num_n_tiles, num_k_blocks;
    int relu, has16, pdl_late;
    unsigned long long* trace;
    // STEM variant: the A operand is gathered from the NCHW fp32 image (7x7 / stride 2 / pad 3 patches), no im2col
    const float* stem_im;
    int sH, sW, sHo, sWo;
    // GEMM variant (sb_gemm_tc): out = alpha * acc + shift[col], alpha read from device memory (NULL: 1)
    const float* alpha;
};

// per epilogue warp: NB fp32 boxes + the fp16 twin's two half boxes (the GEMM variant stores no twin)
constexpr int flat_epi_warp_bytes(bool res, bool f32, bool gemm = false) {
    return f32 ? ((res ? 3 : 2) * 4096 + (gemm ? 0 : 4096)) : 4096;
}

constexpr int kStemGatherWarps = 8;       // 2 threads per A-tile row: each builds 4 of the 8 16-byte groups of a K-step
constexpr int kStemThreads = 320 + 32 * kStemGatherWarps;

// GEMM variant (sb_gemm_tc, C = alpha * A B^T + bias): A_MN / B_MN select an operand stored M/N-major ([K][ld]).  Its
// tiles arrive as 64-element-wide TMA boxes (the 128-byte swizzle span) of BLOCK_K K rows each -- 2 for A, BLOCK_N / 64
// for B, stacked 8 KB apart -- and the MMAs read them through M/N-major descriptors with the transpose bits set, so no
// transposed copy of an operand ever exists.  Everything else (pipeline, TMEM double buffer, TMA-store epilogue) is
// the conv's.
template <int BLOCK_N, int kStages, bool HAS_RES, bool F32, bool STEM = false, bool GEMM = false, bool A_MN = false,
          bool B_MN = false>
__global__ void __launch_bounds__(STEM ? kStemThreads : 320, 1)
conv_tc_flat_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const __grid_constant__ CUtensorMap map_res, const __grid_constant__ CUtensorMap map_o32,
                    const __grid_constant__ CUtensorMap map_o16, const FlatParams p) {
    static_assert(!HAS_RES || F32, "the residual epilogue produces the fp32 stream");
    static_assert(GEMM || (!A_MN && !B_MN), "M/N-major operands are a GEMM feature");
    static_assert(!B_MN || BLOCK_N % 64 == 0, "M/N-major B tiles are whole 64-element boxes");
    constexpr uint32_t kMnBox = 64 * 64 * 2;      // one M/N-major TMA box: 64 M/N elements x 64 K rows of fp16
    constexpr uint32_t kABytes = BLOCK_M * kRowBytes, kBBytes = BLOCK_N * kRowBytes;
    constexpr int BLOCK_K = 64;
    constexpr uint32_t kStageBytes = kABytes + kBBytes;
    constexpr uint32_t kTmemCols = (2 * BLOCK_N <= 32) ? 32 : (2 * BLOCK_N <= 64) ? 64 : (2 * BLOCK_N <= 128) ? 128
                                   : (2 * BLOCK_N <= 256) ? 256 : 512;
    constexpr int NB = HAS_RES ? 3 : 2;                                  // fp32 boxes per warp
    constexpr int kEpiWarpBytes = flat_epi_warp_bytes(HAS_RES, F32, GEMM);
    constexpr int kF16Off = F32 ? NB * 4096 : 0;       // (GEMM: no twin, has16 = 0)
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* epi = smem + kStages * kStageBytes;                          // 1024-aligned (stage bytes are multiples of 4096)
    uint64_t* full = reinterpret_cast<uint64_t*>(epi + 8 * kEpiWarpBytes);
    uint64_t* empty = full + kStages;
    uint64_t* tfull = empty + kStages;
    uint64_t* tempty = tfull + 2;
    uint64_t* rfull = tempty + 2;                                         // [8 warps][3]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rfull + 24);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned long long* tr = p.trace ? p.trace + (size_t)blockIdx.x * kTraceWords : nullptr;
    if (tr && threadIdx.x == 0) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        tr[0] = gtimer(); tr[8] = clock64(); tr[6] = smid;
    }
    if (warp == 0 && elect_one()) {
        prefetch_tmap(&map_a);
        prefetch_tmap(&map_b);
        if (HAS_RES) prefetch_tmap(&map_res);
        if (F32) prefetch_tmap(&map_o32);
        if (p.has16) prefetch_tmap(&map_o16);
    }
    if (warp == 1) {
        if (elect_one()) {
            // STEM: a stage is full when the weight tile has landed (1 expect_tx arrival) and the gather threads
            // have written their patch rows
            for (int i = 0; i < kStages; ++i) { mbar_init(&full[i], STEM ? 1 + 32 * kStemGatherWarps : 1); mbar_init(&empty[i], 1); }
            for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 8); }
            for (int i = 0; i < 24; ++i) mbar_init(&rfull[i], 1);
            fence_barrier_init();
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (!p.pdl_late) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (tr && threadIdx.x == 0) { tr[1] = gtimer(); tr[9] = clock64(); }

    const int num_tiles = p.num_m_tiles * p.num_n_tiles;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (elect_one()) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int mt = tile / p.num_n_tiles, nt = tile - mt * p.num_n_tiles;
                for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * kStageBytes;
                    mbar_expect_tx(&full[stage], STEM ? kBBytes : kStageBytes);
                    if (A_MN) {
#pragma unroll
                        for (int i = 0; i < BLOCK_M / 64; ++i)
                            tma_load_2d(&map_a, &full[stage], sa + i * kMnBox, mt * BLOCK_M + 64 * i, kb * BLOCK_K);
                    } else if (!STEM) {
                        tma_load_2d(&map_a, &full[stage], sa, kb * BLOCK_K, mt * BLOCK_M);
                    }
                    if (B_MN) {
#pragma unroll
                        for (int i = 0; i < BLOCK_N / 64; ++i)
                            tma_load_2d(&map_b, &full[stage], sa + kABytes + i * kMnBox, nt * BLOCK_N + 64 * i, kb * BLOCK_K);
                    } else {
                        tma_load_2d(&map_b, &full[stage], sa + kABytes, kb * BLOCK_K, nt * BLOCK_N);
                    }
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        constexpr uint32_t idesc = make_idesc_major(BLOCK_N, true, A_MN, B_MN);
        // per MMA (K = 16): K-major operands advance 32 bytes inside the swizzle row, M/N-major ones two 8-row K groups
        constexpr uint64_t kStepA = A_MN ? 2048 >> 4 : 2, kStepB = B_MN ? 2048 >> 4 : 2;
        int stage = 0;
        uint32_t phase = 0;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            mbar_wait(&tempty[acc], acc_phase ^ 1);
            tc_fence_after();
            const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
            for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                mbar_wait(&full[stage], phase);
                tc_fence_after();
                if (tr && lane == 0 && kb == 0 && tile == (int)blockIdx.x) { tr[2] = gtimer(); tr[10] = clock64(); }
                if (elect_one()) {
                    const uint32_t sa = smem_u32(smem + stage * kStageBytes);
                    const uint64_t da = A_MN ? make_smem_desc_mn(sa, kMnBox) : make_smem_desc(sa);
                    const uint64_t db = B_MN ? make_smem_desc_mn(sa + kABytes, kMnBox) : make_smem_desc(sa + kABytes);
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        umma_f16(tmem_d, da + (uint64_t)k * kStepA, db + (uint64_t)k * kStepB, idesc, (kb | k) != 0);
                    umma_commit(&empty[stage]);
                    if (kb == p.num_k_blocks - 1) umma_commit(&tfull[acc]);
                }
                __syncwarp();
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (p.pdl_late) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        if (tr && lane == 0) { tr[3] = gtimer(); tr[11] = clock64(); }
    } else if (STEM && warp >= 10) {
        // ===================== stem patch gather (warps 10..17) =====================
        // The 7x7 / stride-2 / pad-3 stem convolution (resnet.py:111) as an implicit GEMM: row gr of the A tile holds
        // the 147 taps (ci, r, s) of one output pixel, zero padded to 3 K-steps of 64 fp16, built straight from the
        // NCHW fp32 image into the 128-byte-swizzled stage (16-byte group j of row r at j ^ (r & 7)), so the 229 MB
        // patch matrix of round 1 (sb_stem_im2col16) is never written or read.  Image reads hit L1 / L2: every input
        // pixel is used by ~12 taps of neighbouring outputs.  Two threads build a row (4 groups each per K-step); all
        // loads of a K-step are issued before the first use and before the wait for the stage, so a thread exposes
        // the load latency once per K-step, not once per tap (4x faster than load-convert-store per group; measured).
        // Variants that were measured and lost (profiles/r02f_stem_fused.md): rows padded to 8 columns and loaded as
        // 8-byte words, one barrier arrival per warp, L1 prefetch of the CTA's next tile.
        constexpr int kPer = 8 / (kStemGatherWarps / 4);       // 16-byte groups per thread and K-step
        const int gt = threadIdx.x - 320;
        const int gr = gt & 127, gh = gt >> 7;
        int stage = 0;
        uint32_t phase = 0;
        const int H = p.sH, W = p.sW;
        const long long HW = (long long)H * W;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int mt = tile / p.num_n_tiles;
            const long long m = (long long)mt * BLOCK_M + gr;
            const bool valid = m < p.M;
            int n = 0, ho = 0, wo = 0;
            if (valid) {
                const int hw = p.sHo * p.sWo;
                n = (int)(m / hw);
                const int rem = (int)(m - (long long)n * hw);
                ho = rem / p.sWo;
                wo = rem - ho * p.sWo;
            }
            const int y0 = 2 * ho - 3, x0 = 2 * wo - 3;
            const float* img = p.stem_im + (long long)n * 3 * HW;
            const float* base = img + (long long)y0 * W + x0;
            const bool interior = valid && y0 >= 0 && y0 + 6 < H && x0 >= 0 && x0 + 6 < W;
#pragma unroll
            for (int kb = 0; kb < 3; ++kb) {
                float v[kPer * 8];
#pragma unroll
                for (int g = 0; g < kStemGatherWarps / 4; ++g) {          // g == gh: keeps every tap index a constant
                    if (g != gh) continue;
                    if (interior) {
#pragma unroll
                        for (int i = 0; i < kPer * 8; ++i) {
                            const int k = kb * 64 + g * kPer * 8 + i;
                            const int ci = k / 49, r = (k % 49) / 7, sx = k % 7;
                            v[i] = k < 147 ? __ldg(base + ci * HW + r * W + sx) : 0.f;
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < kPer * 8; ++i) {
                            const int k = kb * 64 + g * kPer * 8 + i;
                            const int ci = k / 49, r = (k % 49) / 7, sx = k % 7;
                            const int yy = y0 + r, xx = x0 + sx;
                            const bool ok = valid && k < 147 && yy >= 0 && yy < H && xx >= 0 && xx < W;
                            const int yc = min(max(yy, 0), H - 1), xc = min(max(xx, 0), W - 1);
                            const float t = __ldg(img + (k < 147 ? ci : 0) * HW + (long long)yc * W + xc);   // always in bounds
                            v[i] = ok ? t : 0.f;
                        }
                    }
                }
                mbar_wait(&empty[stage], phase ^ 1);
                const uint32_t row = smem_u32(smem + stage * kStageBytes) + gr * 128;
#pragma unroll
                for (int jj = 0; jj < kPer; ++jj) {
                    const int j = gh * kPer + jj;
                    uint32_t h[4];
#pragma unroll
                    for (int e2 = 0; e2 < 4; ++e2) {
                        __half2 pk = __floats2half2_rn(v[jj * 8 + 2 * e2], v[jj * 8 + 2 * e2 + 1]);
                        h[e2] = *reinterpret_cast<uint32_t*>(&pk);
                    }
                    sts128u(row + ((uint32_t)(j ^ (gr & 7)) << 4), make_uint4(h[0], h[1], h[2], h[3]));
                }
                fence_proxy_async();          // generic-proxy writes -> visible to the tensor core's async-proxy reads
                mbar_arrive(&full[stage]);
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        // ===================== epilogue (warps 2..9) =====================
        const int q = warp & 3;            // TMEM lane quarter this warp may touch
        const int ew = warp - 2;
        const int half = ew >> 2;
        constexpr int kColsPerWarp = BLOCK_N / 2 >= 32 ? BLOCK_N / 2 : 32;
        constexpr int kChunks = kColsPerWarp / 32;
        const int col_begin = half * kColsPerWarp;
        const bool has_cols = col_begin < BLOCK_N;
        uint8_t* ebase = epi + ew * kEpiWarpBytes;
        uint64_t* my_rfull = rfull + ew * 3;
        const bool has16 = p.has16 != 0;
        const bool relu = p.relu != 0;
        // (after griddepcontrol.wait: alpha may come from the kernel just before)
        const float alpha = (GEMM && p.alpha) ? __ldg(p.alpha) : 1.f;
        uint32_t g = 0;                    // running chunk number of this warp (ring position)
        // coordinates of chunk gi in this warp's chunk sequence (tiles of this CTA x chunks of the warp)
        auto issue_res = [&](uint32_t gi) {
            const uint32_t ts = gi / kChunks, k = gi - ts * kChunks;
            const long long tile = (long long)blockIdx.x + (long long)ts * gridDim.x;
            if (tile >= num_tiles) return;
            const int mt = (int)(tile / p.num_n_tiles), nt = (int)(tile - (long long)mt * p.num_n_tiles);
            const uint32_t b = gi % NB;
            mbar_expect_tx(&my_rfull[b], 4096);
            tma_load_2d(&map_res, &my_rfull[b], ebase + b * 4096, nt * BLOCK_N + col_begin + 32 * (int)k, mt * BLOCK_M + q * 32);
        };
        // residual rows two tiles ahead go to L2 with a bulk prefetch (layers 1-2: the residual stream lives in HBM)
        auto prefetch_res_tile = [&](int t) {
            if (t >= num_tiles) return;
            const int pmt = t / p.num_n_tiles, pnt = t - pmt * p.num_n_tiles;
            const long long m = (long long)pmt * BLOCK_M + q * 32 + lane;
            const int c0 = pnt * BLOCK_N + col_begin;
            if (m < p.M && c0 < p.Cout)
                prefetch_l2_bulk(p.residual + m * p.res_ld + c0, (uint32_t)min(kColsPerWarp, p.Cout - c0) * 4u);
        };
        if (HAS_RES && has_cols) {
            if (lane == 0) { issue_res(0); issue_res(1); }
            prefetch_res_tile(blockIdx.x + gridDim.x);
        }
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int mt = tile / p.num_n_tiles, nt = tile - mt * p.num_n_tiles;
            if (HAS_RES && has_cols) prefetch_res_tile(tile + 2 * gridDim.x);
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            if (has_cols) {
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BLOCK_N + col_begin);
                const int m0 = mt * BLOCK_M + q * 32;
#pragma unroll
                for (int k = 0; k < kChunks; ++k) {
                    uint32_t v[32];
                    tmem_ld32(taddr + 32 * k, v);
                    const int c0 = nt * BLOCK_N + col_begin + 32 * k;
                    const uint32_t b = F32 ? g % NB : 0;
                    uint8_t* box32 = ebase + b * 4096;
                    uint8_t* box16 = ebase + kF16Off + (g & 1) * 2048;
                    const uint32_t row32 = smem_u32(box32) + lane * 128;
                    const uint32_t row16 = smem_u32(box16) + lane * 64;
                    if (HAS_RES) mbar_wait(&my_rfull[b], (g / NB) & 1);       // this chunk's residual box has landed
                    tmem_ld_wait();
                    if (k == kChunks - 1) {      // the accumulator stage is drained: the MMA warp may reuse it
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tempty[acc]);
                    }
                    uint32_t hprev0 = 0, hprev1 = 0;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int cj = c0 + 4 * j;
                        const bool ok = cj < p.Cout;
                        float4 sc, sh;
                        if (GEMM) {      // any N: the bias of a partial column quad is read element by element
                            sc = make_float4(alpha, alpha, alpha, alpha);
                            sh = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (p.shift && cj + 4 <= p.Cout) {
                                sh = __ldg(reinterpret_cast<const float4*>(p.shift + cj));
                            } else if (p.shift && ok) {
                                sh.x = __ldg(p.shift + cj);
                                if (cj + 1 < p.Cout) sh.y = __ldg(p.shift + cj + 1);
                                if (cj + 2 < p.Cout) sh.z = __ldg(p.shift + cj + 2);
                            }
                        } else {
                            sc = (p.scale && ok) ? __ldg(reinterpret_cast<const float4*>(p.scale + cj)) : make_float4(1.f, 1.f, 1.f, 1.f);
                            sh = (p.shift && ok) ? __ldg(reinterpret_cast<const float4*>(p.shift + cj)) : make_float4(0.f, 0.f, 0.f, 0.f);
                        }
                        float4 x;
                        x.x = fmaf(__uint_as_float(v[4 * j + 0]), sc.x, sh.x);
                        x.y = fmaf(__uint_as_float(v[4 * j + 1]), sc.y, sh.y);
                        x.z = fmaf(__uint_as_float(v[4 * j + 2]), sc.z, sh.z);
                        x.w = fmaf(__uint_as_float(v[4 * j + 3]), sc.w, sh.w);
                        const uint32_t a32 = row32 + ((uint32_t)(j ^ (lane & 7)) << 4);
                        if (HAS_RES) {
                            const float4 r = lds128(a32);
                            x.x += r.x; x.y += r.y; x.z += r.z; x.w += r.w;
                        }
                        if (relu) { x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f); }
                        if (F32) sts128(a32, x);
                        if (has16) {
                            __half2 lo = __floats2half2_rn(x.x, x.y), hi = __floats2half2_rn(x.z, x.w);
                            const uint32_t h0 = *reinterpret_cast<uint32_t*>(&lo), h1 = *reinterpret_cast<uint32_t*>(&hi);
                            if (j & 1) sts128u(row16 + ((uint32_t)((j >> 1) ^ ((lane >> 1) & 3)) << 4), make_uint4(hprev0, hprev1, h0, h1));
                            else { hprev0 = h0; hprev1 = h1; }
                        }
                    }
                    fence_proxy_async();          // the boxes were written through the generic proxy; TMA reads them
                    __syncwarp();
                    if (lane == 0) {
                        if (F32) tma_store_2d(&map_o32, box32, c0, m0);
                        if (has16) tma_store_2d(&map_o16, box16, c0, m0);
                        tma_commit_group();
                        // everything but this chunk's stores has left shared memory: the box of chunk g-1 is free
                        tma_wait_group_read<1>();
                        if (HAS_RES) issue_res(g + 2);
                    }
                    __syncwarp();
                    ++g;
                }
            } else {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[acc]);
            }
            if (tr && warp == 2 && lane == 0 && tile == (int)blockIdx.x) { tr[4] = gtimer(); tr[12] = clock64(); }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (lane == 0) tma_wait_group_read<0>();      // shared memory must outlive the last stores' reads
    }

    tc_fence_before();
    __syncthreads();
    if (tr && threadIdx.x == 0) { tr[5] = gtimer(); tr[13] = clock64(); }
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols));
    }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = (EncodeTiledFn)p;
    }
    return fn;
}

bool make_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
              const cuuint32_t* box, bool f16, CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return false;
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<void*>(base), dims,
                     strides_bytes, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

// Tile-width choice.  One SM ingests ~64 B/clk from L2, so a K-step costs max(MMA cycles, bytes/64):
//   BN=128: max(256, (16+16) KB / 64) = 512 cycles     BN=256: max(512, (16+32) KB / 64) = 768 cycles
// and the persistent grid runs ceil(tiles/SMs) waves.  Pick the cheaper of the two for Cout >= 256.
int pick_block_n(int cout, long long m_tiles, int num_sms) {
    if (cout <= 32) return 32;
    if (cout <= 64) return 64;
    if (cout < 256) return 128;
    const long long t128 = m_tiles * ((cout + 127) / 128), t256 = m_tiles * ((cout + 255) / 256);
    const long long c128 = ((t128 + num_sms - 1) / num_sms) * 512, c256 = ((t256 + num_sms - 1) / num_sms) * 768;
    return c256 <= c128 ? 256 : 128;
}

// CTA-pair launch: clusters of 2, one pair per two SMs, 6 stages of 32 KB (A tile + half a weight tile)
int launch_cg2(const CUtensorMap& ma, const CUtensorMap& mb, const TcParams& p, cudaStream_t st) {
    constexpr int ST = 6, BN = 256;
    constexpr size_t smem = (size_t)ST * (BLOCK_M * kRowBytes + (BN / 2) * kRowBytes) + 1024 + 256 + epi_smem(8);
    static_assert(smem <= 227 * 1024, "smem budget");
    auto kern = conv_tc_kernel<BN, ST, false, false, true, 8, true>;
    static bool attr_done[kSbMaxDevices] = {false};
    bool& attr = attr_done[sb_cur_device()];
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    const int pair_tiles = ((p.num_m_tiles + 1) / 2) * p.num_n_tiles;
    int pairs = sb_num_sms() / 2;
    if (p.d.max_ctas > 1 && p.d.max_ctas / 2 < pairs) pairs = p.d.max_ctas / 2;
    if (pair_tiles < pairs) pairs = pair_tiles;
    static const bool use_pdl = getenv("SB_NO_PDL") == nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(64 + 32 * 8);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attrs[2];
    attrs[0].id = cudaLaunchAttributeClusterDimension;
    attrs[0].val.clusterDim.x = 2; attrs[0].val.clusterDim.y = 1; attrs[0].val.clusterDim.z = 1;
    attrs[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attrs[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attrs;
    cfg.numAttrs = use_pdl ? 2 : 1;
    cudaError_t le = cudaLaunchKernelEx(&cfg, kern, ma, mb, p);
    SB_LAUNCHED();
    if (le != cudaSuccess) return (int)le;
    SB_CHECK_LAUNCH();
    return SB_OK;
}

template <int BN, int ST, bool RES, bool UP, bool IN16, int EW>
int launch_t(const CUtensorMap& ma, const CUtensorMap& mb, const TcParams& p, cudaStream_t st) {
    constexpr size_t smem = (size_t)ST * (BLOCK_M * kRowBytes + BN * kRowBytes) + 1024 + 256 + epi_smem(EW);
    static_assert(smem * (EW == 4 ? 2 : 1) <= 227 * 1024, "smem budget");
    constexpr int kNumThreads = 64 + 32 * EW;
    static bool attr_done[kSbMaxDevices] = {false};
    bool& attr = attr_done[sb_cur_device()];
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel<BN, ST, RES, UP, IN16, EW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess && EW == 4)
            e = cudaFuncSetAttribute(conv_tc_kernel<BN, ST, RES, UP, IN16, EW>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    const int num_sms = sb_num_sms();
    const int tiles = p.num_m_tiles * p.num_n_tiles;
    int slots = num_sms * (EW == 4 ? 2 : 1);
    if (p.d.max_ctas > 0 && p.d.max_ctas < slots) slots = p.d.max_ctas;
    const int grid = tiles < slots ? tiles : slots;
    static const bool use_pdl = getenv("SB_NO_PDL") == nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kNumThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attrs[1];
    attrs[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attrs[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attrs;
    cfg.numAttrs = use_pdl ? 1 : 0;
    cudaError_t le = cudaLaunchKernelEx(&cfg, conv_tc_kernel<BN, ST, RES, UP, IN16, EW>, ma, mb, p);
    SB_LAUNCHED();
    if (le != cudaSuccess) return (int)le;
    SB_CHECK_LAUNCH();
    return SB_OK;
}

// 16 epilogue warps (576 threads): plain and residual epilogues only
template <int BN, int ST>
int launch16(const CUtensorMap& ma, const CUtensorMap& mb, const TcParams& p, cudaStream_t st) {
    const bool res = p.d.residual != nullptr;
    if (p.d.in_dtype == 1)
        return res ? launch_t<BN, ST, true, false, true, 16>(ma, mb, p, st) : launch_t<BN, ST, false, false, true, 16>(ma, mb, p, st);
    return res ? launch_t<BN, ST, true, false, false, 16>(ma, mb, p, st) : launch_t<BN, ST, false, false, false, 16>(ma, mb, p, st);
}

template <int BN, int ST, int EW>
int launch(const CUtensorMap& ma, const CUtensorMap& mb, const TcParams& p, cudaStream_t st) {
    const bool res = p.d.residual != nullptr, up = p.d.up_src != nullptr;   // never both (supported())
    if (p.d.in_dtype == 1) {
        if (up) return launch_t<BN, ST, false, true, true, EW>(ma, mb, p, st);
        return res ? launch_t<BN, ST, true, false, true, EW>(ma, mb, p, st) : launch_t<BN, ST, false, false, true, EW>(ma, mb, p, st);
    }
    if (up) return launch_t<BN, ST, false, true, false, EW>(ma, mb, p, st);
    return res ? launch_t<BN, ST, true, false, false, EW>(ma, mb, p, st) : launch_t<BN, ST, false, false, false, EW>(ma, mb, p, st);
}


template <int BN, int ST, bool RES, bool F32, bool STEM = false, bool GEMM = false, bool A_MN = false, bool B_MN = false>
int launch_flat(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mr, const CUtensorMap& mo32,
                const CUtensorMap& mo16, const FlatParams& p, int max_ctas, cudaStream_t st) {
    constexpr size_t smem = (size_t)ST * (BLOCK_M * kRowBytes + BN * kRowBytes) + 8 * (size_t)flat_epi_warp_bytes(RES, F32, GEMM) +
                            (2 * ST + 4 + 24) * 8 + 16 + 1024;
    static_assert(smem <= 227 * 1024, "smem budget");
    static bool attr_done[kSbMaxDevices] = {false};
    bool& attr = attr_done[sb_cur_device()];
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(conv_tc_flat_kernel<BN, ST, RES, F32, STEM, GEMM, A_MN, B_MN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    const int tiles = p.num_m_tiles * p.num_n_tiles;
    int slots = sb_num_sms();
    if (max_ctas > 0 && max_ctas < slots) slots = max_ctas;
    const int grid = tiles < slots ? tiles : slots;
    static const bool use_pdl = getenv("SB_NO_PDL") == nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(STEM ? kStemThreads : 320);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attrs[1];
    attrs[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attrs[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attrs;
    cfg.numAttrs = use_pdl ? 1 : 0;
    cudaError_t le = cudaLaunchKernelEx(&cfg, conv_tc_flat_kernel<BN, ST, RES, F32, STEM, GEMM, A_MN, B_MN>, ma, mb, mr, mo32, mo16, p);
    SB_LAUNCHED();
    if (le != cudaSuccess) return (int)le;
    SB_CHECK_LAUNCH();
    return SB_OK;
}

// can this conv run through the flat kernel with the TMA epilogue?  (fp16 operands, 1x1, dense [M, Cout] rows)
bool flat_eligible(const sb_conv_desc* d, bool patch) {
    static const bool on = getenv("SB_TC_FLAT") == nullptr || atoi(getenv("SB_TC_FLAT")) != 0;
    if (!on || d->in_dtype != 1 || patch || d->up_src || d->out_mode != 0 || d->res_biased || d->in_biased) return false;
    if (d->out_h_stride != (long long)d->Wo * d->out_w_stride) return false;
    if (d->N > 1 && d->out_n_stride != (long long)d->Ho * d->out_h_stride) return false;      // rows must be equally spaced
    if (d->residual && !d->out) return false;
    if (d->out && (((reinterpret_cast<uintptr_t>(d->out) + 4ull * d->out_coff) & 15) || (d->out_w_stride & 3))) return false;
    if (d->out16 && (((reinterpret_cast<uintptr_t>(d->out16) + 2ull * d->out_coff) & 15) || (d->out_w_stride & 7))) return false;
    return true;
}

}  // namespace

extern "C" int sb_conv2d_tc_supported(const sb_conv_desc* d) {
    if (!d || !d->in || !d->wgt) return 0;
    const int bk = d->in_dtype == 1 ? 64 : 32;
    if (d->in_dtype != 0 && d->in_dtype != 1) return 0;
    if (d->stride != 1 || d->Cin % bk != 0 || d->in_ld % (d->in_dtype == 1 ? 8 : 4) != 0) return 0;
    if (!d->out && !d->out16) return 0;
    const bool k1 = d->kh == 1 && d->kw == 1 && d->pad == 0;
    const bool k3 = d->kh == 3 && d->kw == 3 && d->pad == 1;
    if (!k1 && !k3) return 0;
    if (d->Cout > kMaxCout || (d->Cout & 3)) return 0;
    if (d->residual && (d->up_src || !k1)) return 0;      // the residual epilogue assumes flat (1x1) rows
    if (d->up_src && (long long)d->N * d->UH * d->UW * d->Cout >= 0x7fffffffLL) return 0;
    if ((long long)d->N * d->out_n_stride + d->out_coff >= 0x7fffffffLL) return 0;   // 32-bit element offsets in the epilogue
    if ((reinterpret_cast<uintptr_t>(d->in) & 15) || (reinterpret_cast<uintptr_t>(d->wgt) & 15) ||
        (reinterpret_cast<uintptr_t>(d->out) & 15) || (reinterpret_cast<uintptr_t>(d->out16) & 7))
        return 0;
    if ((d->out_coff & 3) || (d->out_n_stride & 3) || (d->out_h_stride & 3) || (d->out_w_stride & 3)) return 0;
    if (d->residual && ((d->res_ld & 3) || (reinterpret_cast<uintptr_t>(d->residual) & 15))) return 0;
    if ((reinterpret_cast<uintptr_t>(d->scale) & 15) || (reinterpret_cast<uintptr_t>(d->shift) & 15)) return 0;   // float4 loads
    if (d->up_src && ((d->Cout & 3) || (reinterpret_cast<uintptr_t>(d->up_src) & 15))) return 0;
    if (d->Ho != d->H || d->Wo != d->W) return 0;
    if ((long long)d->N * d->Ho * d->Wo >= 0x7fffffffLL) return 0;
    return 1;
}

// ---- optional phase trace (tools/conv_trace.py): 16 words per CTA, kTraceCtas CTAs per launch
namespace {
unsigned long long* g_trace = nullptr;
int g_trace_cap = 0, g_trace_n = 0;
struct TraceInfo { int v[12]; };
TraceInfo g_trace_info[4096];
}  // namespace

extern "C" size_t sb_conv_trace_bytes(int max_launches) {
    return (size_t)max_launches * kTraceCtas * kTraceWords * sizeof(unsigned long long);
}
extern "C" int sb_conv_trace(void* buf, int max_launches) {
    if (max_launches > 4096) return SB_EINVAL;
    g_trace = (unsigned long long*)buf;
    g_trace_cap = buf ? max_launches : 0;
    g_trace_n = 0;
    return SB_OK;
}
extern "C" int sb_conv_trace_info(int id, int* out12) {
    if (id < 0 || id >= g_trace_n) return SB_EINVAL;
    for (int i = 0; i < 12; ++i) out12[i] = g_trace_info[id].v[i];
    return SB_OK;
}
extern "C" int sb_conv_trace_count(void) { return g_trace_n; }

extern "C" int sb_conv2d_tc(const sb_conv_desc* d, sb_stream_t stream) {
    if (!sb_conv2d_tc_supported(d)) return SB_EINVAL;
    TcParams p;
    p.d = *d;
    // default: release the dependent launch once this CTA's last MMAs are issued -- an early release lets the
    // next kernel's CTAs sit in griddepcontrol.wait on SMs the other stream's chain could be using
    static const bool pdl_late = getenv("SB_PDL_LATE") == nullptr || atoi(getenv("SB_PDL_LATE")) != 0;
    p.pdl_late = pdl_late ? 1 : 0;
    // default: both CTAs' TMA loads complete on the leader's barrier (cta_group::2 TMA).  SB_CG2_DIRECT=0 selects the
    // first protocol tried -- the peer's warp 1 forwards "stage full" with a remote mbarrier arrive -- which is correct
    // but 1.7x slower (415 us for the RPN P2 conv: the extra hop sits on the operand ring's round trip).
    static const bool cg2_direct = getenv("SB_CG2_DIRECT") == nullptr || atoi(getenv("SB_CG2_DIRECT")) != 0;
    p.cg2_direct = cg2_direct ? 1 : 0;
    p.trace = nullptr;
    // spatial 8x16 tiles for 3x3 convs, and for the FPN laterals so that the bilinear upsample taps of a tile
    // (5x9 source pixels) stay in L1 instead of being re-fetched from L2 for every output row
    p.patch = (d->kh == 3 || d->up_src) ? 1 : 0;
    p.M = (long long)d->N * d->Ho * d->Wo;
    if (p.M == 0) return SB_OK;
    const bool f16 = d->in_dtype == 1;
    const int BLOCK_K = f16 ? 64 : 32;
    const int esz = f16 ? 2 : 4;
    p.kblocks_per_tap = d->Cin / BLOCK_K;
    p.num_k_blocks = d->kh * d->kw * p.kblocks_per_tap;
    p.tiles_w = (d->W + TW - 1) / TW;
    p.tiles_h = (d->H + TH - 1) / TH;
    p.num_m_tiles = p.patch ? d->N * p.tiles_h * p.tiles_w : (int)((p.M + BLOCK_M - 1) / BLOCK_M);
    const int sms = sb_num_sms();
    int BN = pick_block_n(d->Cout, p.num_m_tiles, sms);
    if (d->residual && BN == 256) BN = 128;   // residual layers are HBM-bound; the 256-wide residual epilogue spills
    // "small" variant (128x128 tiles, half the shared memory, two CTAs per SM): measured slower than the
    // one-CTA-per-SM tiles on every layer shape of this network (tools/conv_bench.py), so it is opt-in only
    bool small = false;
    if (const char* e = getenv("SB_TC_SMALL")) {
        const int v = atoi(e);   // 1: every eligible conv, 2: only convs issued with a grid cap (the L/R chains)
        small = (v == 1 || (v == 2 && d->max_ctas != 0)) && d->Cout >= 128 && !d->up_src;
    }
    if (small) BN = 128;
    if (const char* e = getenv("SB_TC_BLOCK_N")) { int v = atoi(e); if ((v == 128 || v == 256) && d->Cout >= 256 && !small) BN = v; }
    // flat kernel with the TMA epilogue: instances exist for these (tile width, outputs) combinations
    bool flat = !small && flat_eligible(d, p.patch != 0);
    if (flat) {
        if (d->out && BN == 256) BN = 128;            // fp32 boxes of a 256-wide tile do not fit beside the stages
        const bool f16only = !d->out;
        flat = (BN == 32 && d->out && !d->out16 && !d->residual) || (BN == 64 && f16only) || BN == 128 || (BN == 256 && f16only);
    }
    p.num_n_tiles = (d->Cout + BN - 1) / BN;
    // CTA pairs (cta_group::2) for the 256-wide 3x3 convs (default on; SB_TC_CG2=0 switches back to single-CTA tiles).
    // Measured on B200 (tools/conv_trace.py): RPN P2 conv 245 -> 229 us (1.43 -> 1.54 PFLOP/s), all 3x3 convs of a
    // forward 1022 -> 958 us of SM time; bench +1..3 %.
    static const bool cg2_on = getenv("SB_TC_CG2") == nullptr || atoi(getenv("SB_TC_CG2")) != 0;
    const bool cg2 = cg2_on && !flat && !small && f16 && p.patch && d->kh == 3 && !d->up_src && !d->residual && BN == 256 &&
                     d->Cout % 256 == 0 && p.num_m_tiles >= 2;
    if (g_trace && g_trace_n < g_trace_cap) {
        const int id = g_trace_n++;
        p.trace = g_trace + (size_t)id * kTraceCtas * kTraceWords;
        int* v = g_trace_info[id].v;
        v[0] = d->Cin; v[1] = d->Cout; v[2] = d->kh; v[3] = (int)p.M; v[4] = BN; v[5] = p.num_m_tiles * p.num_n_tiles;
        v[6] = p.num_k_blocks; v[7] = d->residual ? 1 : 0; v[8] = d->up_src ? 1 : 0; v[9] = small ? 1 : (flat ? 2 : (cg2 ? 3 : 0));
        v[10] = d->max_ctas; v[11] = d->N;
    }
    CUtensorMap ma, mb;
    if (p.patch) {
        cuuint64_t dims[4] = {(cuuint64_t)d->Cin, (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->N};
        cuuint64_t strides[3] = {(cuuint64_t)d->in_ld * esz, (cuuint64_t)d->W * d->in_ld * esz,
                                 (cuuint64_t)d->H * d->W * d->in_ld * esz};
        cuuint32_t box[4] = {(cuuint32_t)BLOCK_K, TW, TH, 1};
        if (!make_map(&ma, d->in, 4, dims, strides, box, f16)) return SB_EINVAL;
    } else {
        // a row may be SHORTER than Cin (in_ld < Cin: the stem's 152-wide patch rows under a 192-wide zero-padded weight):
        // the map's inner extent is then the row length and TMA zero-fills the rest of the last K-step
        cuuint64_t dims[2] = {(cuuint64_t)(d->in_ld < d->Cin ? d->in_ld : d->Cin), (cuuint64_t)p.M};
        cuuint64_t strides[1] = {(cuuint64_t)d->in_ld * esz};
        cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, BLOCK_M};
        if (!make_map(&ma, d->in, 2, dims, strides, box, f16)) return SB_EINVAL;
    }
    {
        const cuuint64_t ktot = (cuuint64_t)d->kh * d->kw * d->Cin;
        cuuint64_t dims[2] = {ktot, (cuuint64_t)d->Cout};
        cuuint64_t strides[1] = {ktot * esz};
        cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)(cg2 ? BN / 2 : BN)};     // cg2: each CTA loads half the tile
        if (!make_map(&mb, d->wgt, 2, dims, strides, box, f16)) return SB_EINVAL;
    }
    cudaStream_t st = sb_cs(stream);
    if (cg2) return launch_cg2(ma, mb, p, st);
    if (flat) {
        FlatParams fp;
        fp.scale = d->scale; fp.shift = d->shift; fp.residual = d->residual;
        fp.M = p.M; fp.Cout = d->Cout; fp.res_ld = d->res_ld;
        fp.num_m_tiles = p.num_m_tiles; fp.num_n_tiles = p.num_n_tiles; fp.num_k_blocks = p.num_k_blocks;
        fp.relu = d->relu; fp.has16 = d->out16 ? 1 : 0; fp.pdl_late = p.pdl_late; fp.trace = p.trace;
        fp.stem_im = nullptr; fp.sH = fp.sW = fp.sHo = fp.sWo = 0;
        fp.alpha = nullptr;
        CUtensorMap mr = ma, mo32 = ma, mo16 = ma;      // unused maps still need a valid descriptor
        const cuuint64_t dims[2] = {(cuuint64_t)d->Cout, (cuuint64_t)p.M};
        const cuuint32_t box[2] = {32, 32};
        if (d->residual) {
            const cuuint64_t str[1] = {(cuuint64_t)d->res_ld * 4};
            if (!make_map(&mr, d->residual, 2, dims, str, box, false)) return SB_EINVAL;
        }
        if (d->out) {
            const cuuint64_t str[1] = {(cuuint64_t)d->out_w_stride * 4};
            if (!make_map(&mo32, d->out + d->out_coff, 2, dims, str, box, false)) return SB_EINVAL;
        }
        if (d->out16) {
            const cuuint64_t str[1] = {(cuuint64_t)d->out_w_stride * 2};
            if (!make_map(&mo16, reinterpret_cast<const __half*>(d->out16) + d->out_coff, 2, dims, str, box, true,
                          CU_TENSOR_MAP_SWIZZLE_64B))
                return SB_EINVAL;
        }
        const int mc = d->max_ctas;
        if (BN == 32) return launch_flat<32, 6, false, true>(ma, mb, mr, mo32, mo16, fp, mc, st);
        if (BN == 64) return launch_flat<64, 8, false, false>(ma, mb, mr, mo32, mo16, fp, mc, st);
        if (BN == 256) return launch_flat<256, 4, false, false>(ma, mb, mr, mo32, mo16, fp, mc, st);
        if (d->residual) return launch_flat<128, 3, true, true>(ma, mb, mr, mo32, mo16, fp, mc, st);
        if (d->out) return launch_flat<128, 4, false, true>(ma, mb, mr, mo32, mo16, fp, mc, st);
        return launch_flat<128, 6, false, false>(ma, mb, mr, mo32, mo16, fp, mc, st);
    }
    if (small) return launch<128, 2, 4>(ma, mb, p, st);
    // epilogue-bound shapes (at most 8 K-steps per tile: the 1x1 convs of the bottlenecks, the deconv quarters)
    // can run with 16 epilogue warps: SB_TC_EW16 = 0 never (default), 1 by this rule, 2 whenever the tile is wide
    // enough.  Measured (tools/epi_bench.py, bench.py): no faster than 8 warps -- the epilogue is bound by the SM's
    // store / load path, not by per-warp latency -- so it stays opt-in.
    static const int ew16 = getenv("SB_TC_EW16") ? atoi(getenv("SB_TC_EW16")) : 0;
    if (BN >= 128 && !d->up_src && (ew16 == 2 || (ew16 == 1 && p.num_k_blocks <= 8)))
        return BN == 256 ? launch16<256, 3>(ma, mb, p, st) : launch16<128, 5>(ma, mb, p, st);
    switch (BN) {
        case 32: return launch<32, 9, 8>(ma, mb, p, st);
        case 64: return launch<64, 8, 8>(ma, mb, p, st);
        case 256: return launch<256, 4, 8>(ma, mb, p, st);
        default: return launch<128, 6, 8>(ma, mb, p, st);
    }
}

// The stem (resnet.py:111-112: Conv2d(3, 64, 7, stride 2, pad 3) + frozen BN + ReLU) as an implicit GEMM on the tensor
// cores, patches gathered inside the kernel (conv_tc_flat_kernel<.., STEM>): image NCHW fp32 [N,3,H,W], weights fp16
// [64][192] in (ci, r, s) order zero padded from 147, out NHWC fp16 [N,Ho,Wo,64].
extern "C" int sb_stem_conv_tc(const float* im_nchw, int N, int H, int W, const void* wgt16, const float* scale,
                               const float* shift, void* out16, sb_stream_t stream) {
    if (!im_nchw || !wgt16 || !out16 || N < 1 || H < 7 || W < 7) return SB_EINVAL;
    if ((reinterpret_cast<uintptr_t>(wgt16) & 15) || (reinterpret_cast<uintptr_t>(out16) & 15) ||
        (reinterpret_cast<uintptr_t>(scale) & 15) || (reinterpret_cast<uintptr_t>(shift) & 15))
        return SB_EINVAL;
    const int Ho = (H + 6 - 7) / 2 + 1, Wo = (W + 6 - 7) / 2 + 1;
    FlatParams fp;
    fp.scale = scale; fp.shift = shift; fp.residual = nullptr;
    fp.M = (long long)N * Ho * Wo; fp.Cout = 64; fp.res_ld = 0;
    if (fp.M >= 0x7fffffffLL) return SB_EINVAL;
    fp.num_m_tiles = (int)((fp.M + BLOCK_M - 1) / BLOCK_M); fp.num_n_tiles = 1; fp.num_k_blocks = 3;
    fp.relu = 1; fp.has16 = 1;
    static const bool pdl_late = getenv("SB_PDL_LATE") == nullptr || atoi(getenv("SB_PDL_LATE")) != 0;
    fp.pdl_late = pdl_late ? 1 : 0;
    fp.trace = nullptr;
    fp.stem_im = im_nchw; fp.sH = H; fp.sW = W; fp.sHo = Ho; fp.sWo = Wo;
    fp.alpha = nullptr;
    CUtensorMap mb, mo16;
    {
        cuuint64_t dims[2] = {192, 64};
        cuuint64_t strides[1] = {192 * 2};
        cuuint32_t box[2] = {64, 64};
        if (!make_map(&mb, wgt16, 2, dims, strides, box, true)) return SB_EINVAL;
    }
    {
        const cuuint64_t dims[2] = {64, (cuuint64_t)fp.M};
        const cuuint64_t str[1] = {64 * 2};
        const cuuint32_t box[2] = {32, 32};
        if (!make_map(&mo16, out16, 2, dims, str, box, true, CU_TENSOR_MAP_SWIZZLE_64B)) return SB_EINVAL;
    }
    return launch_flat<64, 8, false, false, true>(mb, mb, mb, mb, mo16, fp, 0, sb_cs(stream));
}

// ------------------------------------------------------------------ GEMM with transposed operands
// C[m][n] = alpha * sum_k A(m,k) B(n,k) + bias[n] through the flat kernel's pipeline (conv_tc_flat_kernel<.., GEMM>):
// 128 x 256 tiles (3 stages of 48 KB) or 128 x 128 (4 stages of 32 KB), fp32 C leaves through 32 x 32 TMA boxes.  The backward passes of the layers need
// the operands in the layout their forward stored them in: weight gradients contract over pixels / RoIs (both
// operands M/N-major), data gradients multiply by the untransposed weight (B N-major).  Tails in M, N and K are
// zero-filled by the load maps and clipped by the store map.  One CTA owns each output tile and walks K in order (no
// split-K), so C is bit-identical from run to run.
namespace {
// 256-wide tiles: 3 stages of 48 KB beside the 64 KB of fp32 boxes (the GEMM stores no fp16 twin)
template <bool A_MN, bool B_MN>
int launch_gemm(int bn, const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mo32, const FlatParams& fp,
                cudaStream_t st) {
    if (bn == 256) return launch_flat<256, 3, false, true, false, true, A_MN, B_MN>(ma, mb, mo32, mo32, mo32, fp, 0, st);
    return launch_flat<128, 4, false, true, false, true, A_MN, B_MN>(ma, mb, mo32, mo32, mo32, fp, 0, st);
}
}  // namespace

extern "C" int sb_gemm_tc(const sb_gemm_desc* d, sb_stream_t stream) {
    if (!d || !d->a || !d->b || !d->c || d->M < 1 || d->N < 1 || d->K < 1) return SB_EINVAL;
    if ((d->lda & 7) || (d->ldb & 7) || (d->ldc & 7)) return SB_EINVAL;
    if (d->lda < (d->a_mn_major ? d->M : d->K) || d->ldb < (d->b_mn_major ? d->N : d->K) || d->ldc < d->N) return SB_EINVAL;
    if ((reinterpret_cast<uintptr_t>(d->a) & 15) || (reinterpret_cast<uintptr_t>(d->b) & 15) ||
        (reinterpret_cast<uintptr_t>(d->c) & 15) || (reinterpret_cast<uintptr_t>(d->bias) & 15) ||
        (reinterpret_cast<uintptr_t>(d->alpha) & 3))
        return SB_EINVAL;
    const long long m_tiles = ((long long)d->M + BLOCK_M - 1) / BLOCK_M;
    if (m_tiles >= 0x7fffffffLL) return SB_EINVAL;
    // 256-wide tiles carry 48 KB per 512 MMA cycles instead of 32 KB per 256: the wide tile is less bound by L2 bandwidth
    // (pick_block_n's cost model, which also weighs the waves of the persistent grid)
    const int BN = (d->N >= 256 && pick_block_n(d->N, m_tiles, sb_num_sms()) == 256) ? 256 : 128;
    const long long n_tiles = ((long long)d->N + BN - 1) / BN;
    if (m_tiles * n_tiles >= 0x7fffffffLL) return SB_EINVAL;
    FlatParams fp;
    fp.scale = nullptr; fp.shift = d->bias; fp.residual = nullptr;
    fp.M = d->M; fp.Cout = d->N; fp.res_ld = 0;
    fp.num_m_tiles = (int)m_tiles; fp.num_n_tiles = (int)n_tiles; fp.num_k_blocks = (d->K + 63) / 64;
    fp.relu = 0; fp.has16 = 0;
    static const bool pdl_late = getenv("SB_PDL_LATE") == nullptr || atoi(getenv("SB_PDL_LATE")) != 0;
    fp.pdl_late = pdl_late ? 1 : 0;
    fp.trace = nullptr;
    fp.stem_im = nullptr; fp.sH = fp.sW = fp.sHo = fp.sWo = 0;
    fp.alpha = d->alpha;
    CUtensorMap ma, mb, mo;
    {   // K-major: rows of K elements, box 64 (K) x 128 rows;  M-major: rows of M elements, box 64 (M) x 64 K rows
        const cuuint64_t dims[2] = {(cuuint64_t)(d->a_mn_major ? d->M : d->K), (cuuint64_t)(d->a_mn_major ? d->K : d->M)};
        const cuuint64_t str[1] = {(cuuint64_t)d->lda * 2};
        const cuuint32_t box[2] = {64, d->a_mn_major ? 64u : (cuuint32_t)BLOCK_M};
        if (!make_map(&ma, d->a, 2, dims, str, box, true)) return SB_EINVAL;
    }
    {
        const cuuint64_t dims[2] = {(cuuint64_t)(d->b_mn_major ? d->N : d->K), (cuuint64_t)(d->b_mn_major ? d->K : d->N)};
        const cuuint64_t str[1] = {(cuuint64_t)d->ldb * 2};
        const cuuint32_t box[2] = {64, d->b_mn_major ? 64u : (cuuint32_t)BN};
        if (!make_map(&mb, d->b, 2, dims, str, box, true)) return SB_EINVAL;
    }
    {
        const cuuint64_t dims[2] = {(cuuint64_t)d->N, (cuuint64_t)d->M};
        const cuuint64_t str[1] = {(cuuint64_t)d->ldc * 4};
        const cuuint32_t box[2] = {32, 32};
        if (!make_map(&mo, d->c, 2, dims, str, box, false)) return SB_EINVAL;
    }
    cudaStream_t st = sb_cs(stream);
    if (d->a_mn_major)
        return d->b_mn_major ? launch_gemm<true, true>(BN, ma, mb, mo, fp, st) : launch_gemm<true, false>(BN, ma, mb, mo, fp, st);
    return d->b_mn_major ? launch_gemm<false, true>(BN, ma, mb, mo, fp, st) : launch_gemm<false, false>(BN, ma, mb, mo, fp, st);
}
