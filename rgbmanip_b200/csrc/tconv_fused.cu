// ConvTranspose3d(k = 3, stride 2, padding 1, output_padding 1) + folded BatchNorm + ReLU + skip add
// (ADA/lib/network_v5.py:217-258, 274-278, 287-289) as ONE tcgen05 kernel over all 8 output-parity classes.
//
// o = 2 i - 1 + k: along each axis an even output reads (k = 1, i = o/2); an odd one (k = 2, i = (o-1)/2) and
// (k = 0, i = (o+1)/2).  For a tile of 128 input positions the 27 taps therefore touch only the 8 shifted input
// tiles with offsets in {0,1}^3.  Each K step loads ONE shifted tile and issues every (class, tap) MMA that reads it
// (8, 4, 4, 2, 4, 2, 2, 1 of them) into that class's own 16/32-column TMEM region; the weights of all 27 taps stay
// resident in shared memory.  Compared with 8 separate class launches the input is fetched 8x instead of 27x per
// tile and a tile amortises its pipeline latency over 27 MMAs and 8 output voxels per input position.
#include "ptx.cuh"
#include "stages.cuh"
#include "tc_conv.cuh"
#include "tma.cuh"

namespace adp {

constexpr int TF_THREADS = 192;

struct TconvParams {
    int B, D, H, W;          // input grid
    int Cout;                // real output channels (<= BN)
    int res_cs;              // channel pitch of the skip tensor
    int f16;
    int s2d;                 // out and res are space-to-depth(2): [B, D, H, W, 8 * Cout], channel = parity * Cout + c
    int TW, TH, tiles_x, tiles_y;
    const float* scale;
    const float* bias;
    const bf16* res;         // [B, 2D, 2H, 2W, res_cs]
    bf16* out;               // [B, 2D, 2H, 2W, Cout]
    int* err;
};

template <int KC, int BN>
struct TfCfg {
    static constexpr int A_BYTES = 128 * KC * 2;
    static constexpr int W_SLOT = (BN * KC * 2 + 1023) / 1024 * 1024;
    static constexpr int W_BYTES = 27 * W_SLOT;
    static constexpr int STAGES = 6;
    static constexpr int REGION = BN;                         // TMEM columns per parity class
    static constexpr int TMEM_COLS = 2 * 8 * REGION;          // two accumulator sets
    static constexpr int SMEM = STAGES * A_BYTES + W_BYTES + 1024 + 256;
};

template <int KC, int BN>
__global__ void __launch_bounds__(TF_THREADS, 2)
tconv_fused_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, const TconvParams p, int batch) {
    using Cfg = TfCfg<KC, BN>;
    constexpr int STAGES = Cfg::STAGES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* wsm = smem + STAGES * Cfg::A_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(wsm + Cfg::W_BYTES);
    // bars: [0,S) full, [S,2S) empty, [2S,2S+2) tmem_full, [2S+2,2S+4) tmem_empty, [2S+4] weights, then the TMEM base
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 5);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = ptx::smem_u32(smem), w_base = ptx::smem_u32(wsm), bar_base = ptx::smem_u32(bars);
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
    auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
    auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + 2 + s); };
    const uint32_t w_bar = bar_base + 8u * (2 * STAGES + 4);

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmA);
        ptx::prefetch_tmap(&tmW);
        for (int s = 0; s < STAGES; ++s) { ptx::mbar_init(full_bar(s), 1); ptx::mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < 2; ++s) { ptx::mbar_init(tfull_bar(s), 1); ptx::mbar_init(tempty_bar(s), 4); }
        ptx::mbar_init(w_bar, 1);
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        ptx::tmem_alloc(ptx::smem_u32(tmem_slot), Cfg::TMEM_COLS);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int tiles_per_img = p.D * p.tiles_y * p.tiles_x;
    const int total_tiles = batch * tiles_per_img;
    const int rows_valid = p.TW * p.TH;

    if (warp == 0) {
        if (lane == 0) {
            // all 27 weight slabs, once
            ptx::mbar_arrive_expect_tx(w_bar, 27u * BN * KC * 2u);
            for (int t = 0; t < 27; ++t) ptx::tma_load_3d(&tmW, w_bar, w_base + t * Cfg::W_SLOT, 0, 0, t);
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                int t = tile;
                const int tx = t % p.tiles_x; t /= p.tiles_x;
                const int ty = t % p.tiles_y; t /= p.tiles_y;
                const int d = t % p.D;
                const int b = t / p.D;
                for (int o = 0; o < 8; ++o) {          // shifted input tile (oz, oy, ox) = bits (2, 1, 0) of o
                    ptx::mbar_wait(empty_bar(stage), phase ^ 1, p.err, 21);
                    ptx::mbar_arrive_expect_tx(full_bar(stage), (uint32_t)(rows_valid * KC * 2));
                    ptx::tma_load_5d(&tmA, full_bar(stage), smem_base + stage * Cfg::A_BYTES, 0, tx * p.TW + (o & 1),
                                     ty * p.TH + ((o >> 1) & 1), d + (o >> 2), b);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        int stage = 0, as = 0;
        uint32_t phase = 0, aphase = 0;
        const uint32_t idesc = make_idesc_n(BN, p.f16);
        const uint32_t elected = ptx::elect_one();       // warp-convergent issue, see ptx::umma_bf16_elected
        const uint32_t tbase = __shfl_sync(0xffffffffu, tmem_base, 0);
        ptx::mbar_wait(w_bar, 0, p.err, 22);
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            ptx::mbar_wait(tempty_bar(as), aphase ^ 1, p.err, 23);
            ptx::tc_fence_after();
            const uint32_t tmem_set = tbase + (uint32_t)(as * 8 * Cfg::REGION);
            for (int o = 0; o < 8; ++o) {
                ptx::mbar_wait(full_bar(stage), phase, p.err, 24);
                ptx::tc_fence_after();
                {
                    const uint64_t adesc = make_smem_desc<KC>(smem_base + stage * Cfg::A_BYTES);
                    const int oz = o >> 2, oy = (o >> 1) & 1, ox = o & 1;
                    // per axis: offset 0 serves (parity 0, k = 1) and (parity 1, k = 2); offset 1 serves (parity 1, k = 0)
                    for (int cz = 0; cz < (oz ? 1 : 2); ++cz)
                        for (int cy = 0; cy < (oy ? 1 : 2); ++cy)
                            for (int cx = 0; cx < (ox ? 1 : 2); ++cx) {
                                const int pz = oz ? 1 : cz, py = oy ? 1 : cy, px = ox ? 1 : cx;
                                const int kz = oz ? 0 : (pz ? 2 : 1), ky = oy ? 0 : (py ? 2 : 1), kx = ox ? 0 : (px ? 2 : 1);
                                const int cls = (pz << 2) | (py << 1) | px, tap = (kz * 3 + ky) * 3 + kx;
                                const uint64_t bdesc = make_smem_desc<KC>(w_base + tap * Cfg::W_SLOT);
                                const uint32_t tmem_d = tmem_set + (uint32_t)(cls * Cfg::REGION);
#pragma unroll
                                for (int k = 0; k < KC / 16; ++k)
                                    ptx::umma_bf16_elected(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc,
                                                           (o > 0 || k > 0) ? 1u : 0u, elected);
                            }
                    ptx::umma_commit_elected(empty_bar(stage), elected);
                    if (o == 7) ptx::umma_commit_elected(tfull_bar(as), elected);
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            if (++as == 2) { as = 0; aphase ^= 1; }
        }
    } else {
        const int q = warp & 3;
        const int m = q * 32 + lane;
        const int ty_l = m / p.TW, tx_l = m - ty_l * p.TW;
        int as = 0;
        uint32_t aphase = 0;
        const int oD = 2 * p.D, oH = 2 * p.H, oW = 2 * p.W;
        float sc[BN], sh[BN];          // folded BatchNorm, hoisted out of the tile / class loops (the epilogue is issue bound)
#pragma unroll
        for (int j = 0; j < BN; ++j) { sc[j] = j < p.Cout ? __ldg(p.scale + j) : 0.f; sh[j] = j < p.Cout ? __ldg(p.bias + j) : 0.f; }
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            int t = tile;
            const int tx = t % p.tiles_x; t /= p.tiles_x;
            const int ty = t % p.tiles_y; t /= p.tiles_y;
            const int d = t % p.D;
            const int b = t / p.D;
            const int x = tx * p.TW + tx_l, y = ty * p.TH + ty_l;
            const bool valid = (m < rows_valid) && (x < p.W) && (y < p.H);
            ptx::mbar_wait(tfull_bar(as), aphase, p.err, 25);
            ptx::tc_fence_after();
#pragma unroll 1
            for (int cls = 0; cls < 8; ++cls) {
                uint32_t r[32];
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * 8 * Cfg::REGION + cls * Cfg::REGION);
                ptx::tmem_ld16(taddr, r);
                if (BN == 32) ptx::tmem_ld16(taddr + 16, r + 16);
                ptx::tmem_ld_wait();
                if (valid) {
                    const int pz = cls >> 2, py = (cls >> 1) & 1, px = cls & 1;
                    const size_t pix = (((size_t)b * oD + (2 * d + pz)) * oH + (2 * y + py)) * oW + (2 * x + px);
                    size_t o = pix * p.Cout, ro = pix * p.res_cs;
                    if (p.s2d) o = ro = (((((size_t)b * p.D + d) * p.H + y) * p.W + x) * 8 + cls) * p.Cout;
#pragma unroll
                    for (int j0 = 0; j0 < BN; j0 += 8) {
                        if (j0 < p.Cout) {
                            float v[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                v[j] = fmaxf(fmaf(__uint_as_float(r[j0 + j]), sc[j0 + j], sh[j0 + j]), 0.f);
                            if (p.res) ld8_16(p.res, ro + j0, p.f16, v, true);          // skip joins after the ReLU
                            st8_16(p.out, nullptr, o + j0, p.f16, v);
                        }
                    }
                }
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(tempty_bar(as));
            if (++as == 2) { as = 0; aphase ^= 1; }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------------ host
struct TconvPlan {
    CUtensorMap tmA, tmW;
    TconvParams p;
    int num_sms;
    int (*launch)(const TconvPlan* pl, int batch, cudaStream_t stream);   // the kernel instance of (KC, BN), chosen by tconv_plan
};

template <int KC, int BN>
static int tconv_launch(const TconvPlan* pl, int batch, cudaStream_t stream) {
    using Cfg = TfCfg<KC, BN>;
    static int attr[kMaxDevices];
    ADP_TRY(ensure_dyn_smem(tconv_fused_kernel<KC, BN>, Cfg::SMEM, attr));
    const long long total = (long long)batch * pl->p.D * pl->p.tiles_y * pl->p.tiles_x;
    if (total == 0) return ADP_OK;
    const long long slots = 2LL * pl->num_sms;
    const int grid = (int)(total < slots ? total : slots);
    tconv_fused_kernel<KC, BN><<<grid, TF_THREADS, Cfg::SMEM, stream>>>(pl->tmA, pl->tmW, pl->p, batch);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

TconvPlan* tconv_alloc() { return new TconvPlan(); }
void tconv_release(TconvPlan* p) { delete p; }

int tconv_plan(TconvPlan* pl, const Act& in, const bf16* w, int Cout, const float* scale, const float* bias, const bf16* res,
               int res_cs, bf16* out, int flags, int num_sms) {
    ADP_TRY(tma_init_driver());
    ADP_CHECK_ARG((in.C == 16 || in.C == 32) && Cout % 8 == 0 && Cout <= 32, "fused transposed conv: Cin in {16,32}, Cout in {8,16,32}");
    ADP_CHECK_ARG(in.lo == nullptr, "single-plane activations only");
    const int KC = in.C;
    const int BN = Cout <= 16 ? 16 : 32;
    TconvParams& p = pl->p;
    p = TconvParams{};
    p.B = in.B; p.D = in.D; p.H = in.H; p.W = in.W; p.Cout = Cout; p.res_cs = res_cs ? res_cs : Cout; p.f16 = in.f16; p.s2d = (flags >> 1) & 1;
    tc_pick_tile(in.H, in.W, &p.TW, &p.TH);
    p.tiles_x = cdiv(in.W, p.TW); p.tiles_y = cdiv(in.H, p.TH);
    p.scale = scale; p.bias = bias; p.res = res; p.out = out; p.err = nullptr;
    const CUtensorMapSwizzle swz = KC == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    const cuuint64_t dims_a[5] = {(cuuint64_t)in.C, (cuuint64_t)in.W, (cuuint64_t)in.H, (cuuint64_t)in.D, (cuuint64_t)in.B};
    const cuuint32_t box_a[5] = {(cuuint32_t)KC, (cuuint32_t)p.TW, (cuuint32_t)p.TH, 1, 1};
    ADP_TRY(tma_encode(&pl->tmA, tma_type16(in.f16), 5, in.hi, dims_a, 2, box_a, nullptr, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                       "tconv input"));
    const cuuint64_t dims_w[3] = {(cuuint64_t)in.C, (cuuint64_t)BN, 27};
    const cuuint32_t box_w[3] = {(cuuint32_t)KC, (cuuint32_t)BN, 1};
    ADP_TRY(tma_encode(&pl->tmW, tma_type16(in.f16), 3, w, dims_w, 2, box_w, nullptr, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                       "tconv weights"));
    static const struct { int KC, BN; decltype(TconvPlan::launch) launch; } instances[] = {
        {16, 16, tconv_launch<16, 16>}, {32, 16, tconv_launch<32, 16>}, {32, 32, tconv_launch<32, 32>}, {16, 32, tconv_launch<16, 32>}};
    pl->launch = nullptr;
    for (const auto& t : instances) if (t.KC == KC && t.BN == BN) pl->launch = t.launch;
    if (!pl->launch) {
        set_last_error("no fused transposed-conv instantiation for KC=%d BN=%d", KC, BN);
        return ADP_ERR_ARG;
    }
    pl->num_sms = num_sms > 0 ? num_sms : 148;
    return ADP_OK;
}

int tconv_run(TconvPlan* pl, int batch, int* err_flag, cudaStream_t stream) {
    ADP_CHECK_ARG(batch <= pl->p.B, "batch exceeds planned capacity");
    pl->p.err = err_flag;
    return pl->launch(pl, batch, stream);
}

}  // namespace adp
