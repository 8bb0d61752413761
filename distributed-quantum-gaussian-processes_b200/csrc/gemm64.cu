// Grouped fp64 GEMM, 128x64 tile per CTA, 8 warps (4x2) each owning 32x32 = 4x4 DMMA 8x8 blocks, two CTAs per SM
// so one CTA's prologue / C read-modify-write overlaps the other's DMMA stream (v1 was 128x128, one CTA per SM:
// 60% DMMA-pipe utilisation on the K=128 trailing updates, 83% on long K; ncu profiles/r01_v1_syrk0, _lauum).
// Operands stream HBM/L2 -> shared memory through a 3-stage ring: two tensor-map boxes per 16-deep k-chunk issued by one thread
// (TMA, gemm_group_tmap_kernel, the default) or per-thread 16-byte cp.async (LDGSTS; the small-tile kernel and the fallback);
// shared-memory pitches (20 / 132 doubles) make every DMMA fragment load bank-conflict-free.
// A launch covers a *group* of independent tasks (device-resident table) so the many small products of
// the recursive triangular inverse fill the machine in one launch.  Roofline: FP64 pipe (DMMA and DFMA
// share it on B200: 37.1 TFLOP/s measured, profiles/r01_fp64_peak.json).
#include <cstring>
#include <vector>
#include "gemm64.cuh"
#include "tensormap.cuh"

namespace dqgp {

template <int ROWS, int PITCH_R, int THREADS>
__device__ __forceinline__ void gm_load_operand(double* sm, const double* __restrict__ g, int ld, int row0, int k0, int k_contig) {
    // ROWS rows x 16 k doubles as 16-byte chunks
    constexpr int CHUNKS = ROWS * GM_KC / 2;
    static_assert(CHUNKS % THREADS == 0, "operand chunks must divide over the CTA");
    if (k_contig) {
#pragma unroll
        for (int i = 0; i < CHUNKS / THREADS; ++i) {
            const int c = threadIdx.x + THREADS * i;
            const int row = c >> 3, kc = (c & 7) * 2;
            cp_async16(sm + row * GM_PITCH_K + kc, g + (size_t)(row0 + row) * ld + k0 + kc);
        }
    } else {
#pragma unroll
        for (int i = 0; i < CHUNKS / THREADS; ++i) {
            const int c = threadIdx.x + THREADS * i;
            const int k = c / (ROWS / 2), mc = (c % (ROWS / 2)) * 2;
            cp_async16(sm + k * PITCH_R + mc, g + (size_t)(k0 + k) * ld + row0 + mc);
        }
    }
}

template <typename S, int AK, int BK, bool TMAP>
__device__ __forceinline__ void gemm_tile(const GemmTask& T, int local, double* gm_smem, const CUtensorMap* tmaps = nullptr);

__device__ __forceinline__ int gm_find_task(const GemmTask* __restrict__ tasks, int n_tasks, int tile) {
    int lo = 0, hi = n_tasks - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (tasks[mid].tile_begin <= tile) lo = mid; else hi = mid - 1;
    }
    return lo;
}

template <typename S, bool TMAP>
__device__ __forceinline__ void gm_dispatch(const GemmTask* __restrict__ tasks, int n_tasks, double* gm_smem, const CUtensorMap* maps = nullptr) {
    // locate the task that owns this tile (tables are short: <= a few hundred entries)
    const int ti = gm_find_task(tasks, n_tasks, blockIdx.x);
    const GemmTask T = tasks[ti];
    const int local = blockIdx.x - T.tile_begin;
    const CUtensorMap* tm = TMAP ? maps + 2 * ti : nullptr;      // this task's A and B operand maps
    // operand layouts are compile-time inside the tile routine (no predicated duplicate fragment loads)
    if (T.a_k_contig) {
        if (T.b_k_contig) gemm_tile<S, 1, 1, TMAP>(T, local, gm_smem, tm); else gemm_tile<S, 1, 0, TMAP>(T, local, gm_smem, tm);
    } else {
        if (T.b_k_contig) gemm_tile<S, 0, 1, TMAP>(T, local, gm_smem, tm); else gemm_tile<S, 0, 0, TMAP>(T, local, gm_smem, tm);
    }
}

__global__ void __launch_bounds__(GemmBig::THREADS, 2) gemm_group_kernel(const GemmTask* __restrict__ tasks, int n_tasks) {
    extern __shared__ __align__(16) double gm_smem[];
    gm_dispatch<GemmBig, false>(tasks, n_tasks, gm_smem);
}
__global__ void __launch_bounds__(GemmSmall::THREADS, 4) gemm_small_kernel(const GemmTask* __restrict__ tasks, int n_tasks) {
    extern __shared__ __align__(16) double gm_smem[];
    gm_dispatch<GemmSmall, false>(tasks, n_tasks, gm_smem);
}
// Operand tiles as TWO tensor-map boxes per k-chunk (TMA proper, SASS UTMALDG.2D), issued by one thread: the box is as wide as the padded
// shared-memory pitch (20 for k-contiguous operands: the 4 doubles beyond the chunk are the next chunk's, never read; BM + 4 / BN + 4
// otherwise), so the fragment layout stays bank-conflict-free without a swizzle.  Used for every registered task table whose maps the
// driver accepted: same box, one issuing thread instead of 768 LDGSTS per chunk - measured on one B200 against the cp.async ring,
// alternating runs: lauum 5.73 -> 5.31 ms (32.0 -> 34.5 TF = 0.93 of the FP64 peak), triangular inverse 6.15 -> 5.80 ms, potrf
// 8.13 -> 7.79 ms, a lone n = 8192 factorisation 20.02 -> 18.89 ms, the N = 1 iteration of config 4 227.9 -> 219.2 ms; bit-identical
// results.  (A round-2 variant with one cp.async.bulk per tile row lost to the cp.async ring - dqgp_dgemm 8192^3 30.0 against
// 32.9 TFLOP/s, 192 copies and 256 threads polling an mbarrier per chunk - and was removed; what it lacked was the single issuing thread.)
__global__ void __launch_bounds__(GemmBig::THREADS, 2) gemm_group_tmap_kernel(const GemmTask* __restrict__ tasks, int n_tasks,
                                                                              const CUtensorMap* __restrict__ maps) {
    extern __shared__ __align__(128) double gm_smem_t[];
    gm_dispatch<GemmBig, true>(tasks, n_tasks, gm_smem_t, maps);
}

template <typename S, int AK, int BK, bool TMAP>
__device__ __forceinline__ void gemm_tile(const GemmTask& T, int local, double* gm_smem, const CUtensorMap* tmaps) {
    __shared__ __align__(8) unsigned long long gm_bar[GM_STAGES];
    if (TMAP) {
        if (threadIdx.x == 0) {
#pragma unroll
            for (int s = 0; s < GM_STAGES; ++s) mbar_init(&gm_bar[s], 1);
            mbar_fence_init();
        }
        __syncthreads();
    }
    constexpr int GM_BM = S::BM, GM_BN = S::BN, MI = S::MI, NI = S::NI;
    constexpr int GM_PITCH_M = S::PITCH_M, GM_PITCH_N = S::PITCH_N, GM_STAGE_DOUBLES = S::STAGE_DOUBLES, GM_A_DOUBLES = S::A_DOUBLES;
    constexpr int R = GM_BM / GM_BN;
    int tm, tn;
    if (T.lower_tiles) {
        // row block tm owns R*(tm+1) tiles; tiles before it: R*tm*(tm+1)/2
        const int q = local / R;
        tm = int((sqrt(8.0 * q + 1.0) - 1.0) * 0.5);
        while (R * (tm + 1) * (tm + 2) / 2 <= local) ++tm;
        while (R * tm * (tm + 1) / 2 > local) --tm;
        tn = local - R * tm * (tm + 1) / 2;
    } else {
        // full tile grid: enumerate so that tiles with the LONGEST contraction range come first (the triangular
        // operands clip k per tile), otherwise the last wave is a few long tiles on an idle machine
        const int tiles_n = T.N / GM_BN, tiles_m = T.M / GM_BM;
        if (T.krule == GM_KRULE_B_LOWER) {          // k >= n0: long for small tn -> column-major
            tn = local / tiles_m;
            tm = local - tn * tiles_m;
        } else if (T.krule == GM_KRULE_A_LOWER) {   // k < m0 + 128: long for large tm -> rows in descending order
            tm = tiles_m - 1 - local / tiles_n;
            tn = local % tiles_n;
        } else {
            tm = local / tiles_n;
            tn = local - tm * tiles_n;
        }
    }
    const int m0 = tm * GM_BM, n0 = tn * GM_BN;
    int kb = 0, ke = T.K;
    if (T.krule == GM_KRULE_A_LOWER) ke = min(T.K, m0 + GM_BM);
    else if (T.krule == GM_KRULE_B_LOWER) kb = (n0 / GM_KC) * GM_KC;
    else if (T.krule == GM_KRULE_LAUUM) kb = max(m0, (n0 / GM_KC) * GM_KC);
    const int n_chunks = (ke - kb) / GM_KC;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wm = warp / S::WC, wn = warp % S::WC;     // WR x WC warps, (8 MI) x (8 NI) each
    const int g = lane >> 2, t = lane & 3;
    constexpr int WROWS = 8 * MI, WCOLS = 8 * NI;

    double acc[MI][NI][2];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < NI; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    auto stage_a = [&](int s) { return gm_smem + (size_t)s * GM_STAGE_DOUBLES; };
    auto stage_b = [&](int s) { return gm_smem + (size_t)s * GM_STAGE_DOUBLES + GM_A_DOUBLES; };

    constexpr unsigned TM_BYTES = ((AK ? GM_BM * GM_PITCH_K : GM_KC * GM_PITCH_M) + (BK ? GM_BN * GM_PITCH_K : GM_KC * GM_PITCH_N)) * sizeof(double);
    auto fill = [&](int s, int c) {
        if (TMAP) {
            if (threadIdx.x == 0) {
                const int k = kb + c * GM_KC;
                mbar_arrive_expect_tx(&gm_bar[s], TM_BYTES);
                if (AK) tensor_copy_2d_g2s(stage_a(s), tmaps, k, m0, &gm_bar[s]); else tensor_copy_2d_g2s(stage_a(s), tmaps, m0, k, &gm_bar[s]);
                if (BK) tensor_copy_2d_g2s(stage_b(s), tmaps + 1, k, n0, &gm_bar[s]); else tensor_copy_2d_g2s(stage_b(s), tmaps + 1, n0, k, &gm_bar[s]);
            }
        } else {
            gm_load_operand<GM_BM, GM_PITCH_M, S::THREADS>(stage_a(s), T.A, T.lda, m0, kb + c * GM_KC, AK);
            gm_load_operand<GM_BN, GM_PITCH_N, S::THREADS>(stage_b(s), T.B, T.ldb, n0, kb + c * GM_KC, BK);
        }
    };
#pragma unroll
    for (int s = 0; s < GM_STAGES - 1; ++s) {
        if (s < n_chunks) fill(s, s);
        if (!TMAP) cp_async_commit();
    }
    for (int ch = 0; ch < n_chunks; ++ch) {
        if (TMAP) mbar_wait(&gm_bar[ch % GM_STAGES], (ch / GM_STAGES) & 1);
        else cp_async_wait<GM_STAGES - 2>();
        __syncthreads();
        {
            const int nx = ch + GM_STAGES - 1;
            if (nx < n_chunks) fill(nx % GM_STAGES, nx);
            if (!TMAP) cp_async_commit();
        }
        const double* As = stage_a(ch % GM_STAGES);
        const double* Bs = stage_b(ch % GM_STAGES);
#pragma unroll
        for (int kk = 0; kk < GM_KC / 4; ++kk) {
            double a[MI], b[NI];
            if (AK) {
#pragma unroll
                for (int i = 0; i < MI; ++i) a[i] = As[(wm * WROWS + i * 8 + g) * GM_PITCH_K + kk * 4 + t];
            } else {
#pragma unroll
                for (int i = 0; i < MI; ++i) a[i] = As[(kk * 4 + t) * GM_PITCH_M + wm * WROWS + i * 8 + g];
            }
            if (BK) {
#pragma unroll
                for (int j = 0; j < NI; ++j) b[j] = Bs[(wn * WCOLS + j * 8 + g) * GM_PITCH_K + kk * 4 + t];
            } else {
#pragma unroll
                for (int j = 0; j < NI; ++j) b[j] = Bs[(kk * 4 + t) * GM_PITCH_N + wn * WCOLS + j * 8 + g];
            }
#pragma unroll
            for (int i = 0; i < MI; ++i)
#pragma unroll
                for (int j = 0; j < NI; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
    }
    if (!TMAP) cp_async_wait<0>();

    // epilogue: each lane owns 2 adjacent doubles per 8x8 block -> 16-byte accesses
#pragma unroll
    for (int i = 0; i < MI; ++i) {
        const int r = m0 + wm * WROWS + i * 8 + g;
#pragma unroll
        for (int j = 0; j < NI; ++j) {
            const int c = n0 + wn * WCOLS + j * 8 + 2 * t;
            double2* dst = reinterpret_cast<double2*>(T.C + (size_t)r * T.ldc + c);
            double2 v = make_double2(T.alpha * acc[i][j][0], T.alpha * acc[i][j][1]);
            if (T.beta != 0.0) {
                const double2 old = *dst;
                v.x = fma(T.beta, old.x, v.x);
                v.y = fma(T.beta, old.y, v.y);
            }
            *dst = v;
        }
    }
}

int gemm_init() {
    static bool done[64] = {false};
    int dev = 0;
    DQGP_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && done[dev]) return 0;
    DQGP_CUDA(cudaFuncSetAttribute(gemm_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GemmBig::SMEM_BYTES));
    DQGP_CUDA(cudaFuncSetAttribute(gemm_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GemmSmall::SMEM_BYTES));
    DQGP_CUDA(cudaFuncSetAttribute(gemm_group_tmap_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GemmBig::SMEM_BYTES + 128));
    if (dev >= 0 && dev < 64) done[dev] = true;
    return 0;
}

// ---- tensor maps: registered task tables -> device arrays of (A map, B map) per task -----------------------------------------
struct GemmMapTable { const GemmTask* d_tasks; int n; CUtensorMap* d_maps; };
static std::vector<GemmMapTable>& gemm_map_tables() { static std::vector<GemmMapTable> t; return t; }

void gemm_register_maps(const GemmTask* d_tasks, const GemmTask* h_tasks, int n_tasks) {
    if (n_tasks <= 0) return;
    std::vector<CUtensorMap> maps(2 * (size_t)n_tasks);
    memset(maps.data(), 0, sizeof(CUtensorMap) * maps.size());
    for (int i = 0; i < n_tasks; ++i) {
        const GemmTask& t = h_tasks[i];
        // k-contiguous: rows of K values, box = (tile rows) x (chunk + padding); otherwise rows of M (N) values, box = (chunk) x (tile + padding)
        const bool oka = t.a_k_contig ? make_matrix_tensor_map(&maps[2 * i], t.A, t.K, t.M, t.lda, GM_PITCH_K, GM_BM)
                                      : make_matrix_tensor_map(&maps[2 * i], t.A, t.M, t.K, t.lda, GM_PITCH_M, GM_KC);
        const bool okb = t.b_k_contig ? make_matrix_tensor_map(&maps[2 * i + 1], t.B, t.K, t.N, t.ldb, GM_PITCH_K, GM_BN)
                                      : make_matrix_tensor_map(&maps[2 * i + 1], t.B, t.N, t.K, t.ldb, GM_PITCH_N, GM_KC);
        if (!oka || !okb) return;                  // the driver refused a map: this table stays on the cp.async ring
    }
    CUtensorMap* d_maps = nullptr;
    if (cudaMalloc(&d_maps, sizeof(CUtensorMap) * maps.size()) != cudaSuccess) { cudaGetLastError(); return; }
    if (cudaMemcpy(d_maps, maps.data(), sizeof(CUtensorMap) * maps.size(), cudaMemcpyHostToDevice) != cudaSuccess) { cudaGetLastError(); cudaFree(d_maps); return; }
    gemm_map_tables().push_back({d_tasks, n_tasks, d_maps});
}

void gemm_unregister_maps(const GemmTask* d_tasks) {
    auto& tabs = gemm_map_tables();
    for (size_t i = 0; i < tabs.size(); ++i)
        if (tabs[i].d_tasks == d_tasks) { cudaFree(tabs[i].d_maps); tabs.erase(tabs.begin() + i); return; }
}

int launch_gemm_group(const GemmTask* d_tasks, int n_tasks, int total_tiles, cudaStream_t st) {
    if (n_tasks <= 0 || total_tiles <= 0) return 0;
    int rc = gemm_init();
    if (rc) return rc;
    for (const GemmMapTable& tab : gemm_map_tables())
        if (d_tasks >= tab.d_tasks && d_tasks + n_tasks <= tab.d_tasks + tab.n) {
            gemm_group_tmap_kernel<<<total_tiles, GemmBig::THREADS, GemmBig::SMEM_BYTES + 128, st>>>(d_tasks, n_tasks, tab.d_maps + 2 * (d_tasks - tab.d_tasks));
            DQGP_LAUNCH_CHECK("gemm_group_tmap_kernel");
            return 0;
        }
    gemm_group_kernel<<<total_tiles, GemmBig::THREADS, GemmBig::SMEM_BYTES, st>>>(d_tasks, n_tasks);
    DQGP_LAUNCH_CHECK("gemm_group_kernel");
    return 0;
}

int launch_gemm_group_small(const GemmTask* d_tasks, int n_tasks, int total_tiles, cudaStream_t st) {
    if (n_tasks <= 0 || total_tiles <= 0) return 0;
    int rc = gemm_init();
    if (rc) return rc;
    gemm_small_kernel<<<total_tiles, GemmSmall::THREADS, GemmSmall::SMEM_BYTES, st>>>(d_tasks, n_tasks);
    DQGP_LAUNCH_CHECK("gemm_small_kernel");
    return 0;
}

}  // namespace dqgp
