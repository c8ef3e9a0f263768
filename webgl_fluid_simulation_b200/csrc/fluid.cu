// fluid.cu — libfluid_b200: the C ABI of include/fluid.h over the sm_100a kernels.
//
// Host-side structure mirrors the reference's globals (script.js S:950-954): five fields, three of
// them DoubleFBO-style read/write pairs with swap() (S:1079-1106).  There is no CPU fallback:
// every entry point either launches CUDA kernels on the handle's stream or fails.
#include "../../include/fluid.h"

#include <cuda.h>            // CUtensorMap types only: the encoder is fetched through cudaGetDriverEntryPoint
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <type_traits>
#include <vector>

#include "jacobi.cuh"
#include "nccl_dl.h"
#include "passes.cuh"
#include "stream_passes.cuh"
#include "postfx.cuh"
#include "half_passes.cuh"

namespace {

thread_local std::string g_create_error;

struct Pair {              // createDoubleFBO, S:1079-1106
    void* read = nullptr;
    void* write = nullptr;
    void swap() { std::swap(read, write); }
};

}  // namespace

struct fluid {
    fluid_config cfg{};
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;  // slab mode: halo exchange + boundary strips, overlapped with the interior launch
    cudaStream_t active = nullptr;   // where halo / Jacobi launches go right now (== stream except inside that overlap)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t mark[2] = {nullptr, nullptr};
    cudaEvent_t tev[8] = {};
    Pair velocity, dye, pressure;    // float2 / float4 / float
    float* divergence = nullptr;
    float* curl = nullptr;
    int* halo_flag = nullptr;        // device flag set by advection when a tap leaves the ghost zone
    uint64_t launches = 0;
    uint64_t jacobi_kernel_launches = 0;   // Jacobi kernels only (fluid_stat FLUID_STAT_JACOBI_LAUNCHES)
    uint64_t halo_kernel_launches = 0;     // halo_push / halo_wait kernels of the peer-memory transport
    uint64_t div_epoch = 1, div_sent_epoch = 0;   // slab: the divergence ghost rows are re-sent only after divergence was rewritten
    int div_sent_rows = 0;
    bool pdl_chain = false;                // the next blocked Jacobi launch directly follows another one of the same solve
    bool capturing = false;                // inside the stream capture of a step graph
    bool half = false;                     // FLUID_FLAG_HALF_STORAGE: fields are fp16 (half_passes.cuh), single GPU only
    float* scratch = nullptr;              // half mode: fp32 staging of fluid_read / fluid_write / render
    size_t scratch_floats = 0;
    float* dt_dev = nullptr;               // step()'s dt lives in device memory: one graph serves every dt
    unsigned char* tiny_map = nullptr;     // where divergence has 0 < |d| < 2^-123 (jacobi.cuh): 1 byte per 128x32 cells, GLOBAL rows
    size_t tiny_map_bytes = 0;
    // 2-D tensor maps (TMA staging of the blocked Jacobi kernel) of the two pressure buffers and divergence
    struct Tmaps { CUtensorMap p[2]; void* p_ptr[2] = {nullptr, nullptr}; CUtensorMap d; bool ok = false; } tmaps;
    double splat_radius_d = 0.25;          // config.SPLAT_RADIUS and the canvas aspect as the JS doubles they are
    double aspect_d = 1.0;                 // (correctRadius S:1457-1462 is double arithmetic, narrowed once)
    int background = 0;                    // FLUID_BACKGROUND: what render() draws the display over (0 colour, 1 checkerboard, 2 none)
    fluid_timing timing{};
    bool have_timing = false;
    std::string err;
    int jacobi_rows_override = 0;    // FLUID_JACOBI_ROWS env (tuning)
    int jacobi_warps_per_sm = 0;     // FLUID_JACOBI_WARPS env (tuning): cap on resident streams per SM used to size the chunks

    // ---- row-slab decomposition (SURVEY §8e).  Single GPU: rank 0 of 1, no ghost rows. -------------
    int rank = 0, world = 1;
    int G = 0, Gd = 0;               // ghost rows kept below and above the owned rows (sim / dye)
    int row0 = 0, row1 = 0;          // owned sim rows  [row0, row1)
    int drow0 = 0, drow1 = 0;        // owned dye rows  [drow0, drow1)
    int roff = 0, droff = 0;         // global row index of local row 0  (row0 - G, drow0 - Gd)
    ncdl::ncclComm_t comm = nullptr;
    bool v_ghost_valid = true;       // velocity valid on owned rows +-3 (what the next step needs)
    uint64_t halo_groups = 0;        // halo exchanges issued (diagnostics)
    // ---- peer-memory halo path (fluid_p2p_export / fluid_p2p_connect) -------------------------------
    char* arena = nullptr;           // slab mode: every exchanged field + the flag words live in ONE allocation
    size_t arena_bytes = 0;
    size_t off_v[2] = {0, 0}, off_p[2] = {0, 0}, off_dye[2] = {0, 0}, off_div = 0, off_flags = 0;
    int par_v = 0, par_p = 0, par_dye = 0;   // which half of a pair is .read (toggles with swap(); SPMD-identical)
    struct Peer {
        bool present = false;
        char* base = nullptr;        // neighbour's arena mapped here through CUDA IPC
        int roff = 0, droff = 0;     // neighbour's local-row-0 global row indices
        size_t off_v[2], off_p[2], off_dye[2], off_div, off_flags;
    } peer[2];                       // [0] = rank-1 (below), [1] = rank+1 (above)
    bool p2p = false;
    uint32_t p2p_seq = 0;
    // pressure ghost rows stored by the neighbours' last Jacobi launch (jacobi.cuh, TbSync): sequence number of
    // the last mirrored solve, whether pressure.read's ghost rows still hold it, and how many rows deep
    uint32_t mir_seq = 0;
    bool p_mirror_valid = false;
    int p_mirror_rows = 0;
    // fluid_pressure_solve_host pipelined over row bands (single GPU): copy streams, per-band events and the
    // band-private ping-pong rows of the intermediate launches
    struct HostPipe {
        cudaStream_t up = nullptr, down = nullptr;
        cudaEvent_t ev_start = nullptr, ev_up[16] = {}, ev_done[16] = {};
        float* s[2] = {nullptr, nullptr};
        size_t s_floats = 0;
    } hp;
    fk::TbSync tb_sync{};                      // hand-offs of the NEXT blocked launch (launch_tb: SYNC instantiation when tb_sync_on)
    bool tb_sync_on = false;
    // divergence ghost rows of the exchange about to be issued: the peer-memory wait kernel scans them (halo.cuh)
    struct { const float* div; unsigned char* map; int W, row_off, lo0, hi0, lo1, hi1; } scan{};
    bool scan_pending = false;
    // ---- step() as a CUDA graph (single GPU): one instantiated graph per (dt, config scalars, parity)
    struct StepGraph { cudaGraphExec_t exec = nullptr; int flip_v = 0, flip_p = 0, flip_dye = 0, kernels = 0, jacobi_launches = 0; };
    std::map<std::string, StepGraph> graphs;
    uint64_t graph_launches = 0, graph_captures = 0;
    float4* frame = nullptr;         // render target of fluid_render (w x h RGBA fp32), grown on demand
    size_t frame_cells = 0;
    bool slab() const { return world > 1; }
    int lrows() const { return row1 - row0 + 2 * G; }
    int ldrows() const { return drow1 - drow0 + 2 * Gd; }
};

namespace {

using namespace fk;

inline void swap_v(fluid_t* h) { h->velocity.swap(); h->par_v ^= 1; }
inline void swap_p(fluid_t* h) { h->pressure.swap(); h->par_p ^= 1; }
inline void swap_dye(fluid_t* h) { h->dye.swap(); h->par_dye ^= 1; }

void drop_graphs(fluid_t* h) {
    if (!h->graphs.empty() && h->stream) cudaStreamSynchronize(h->stream);   // an exec may still be in flight
    for (auto& kv : h->graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    h->graphs.clear();
}

int fail(fluid_t* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(h, FLUID_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                                  \
    } while (0)

inline bool is_pow2(int n) { return n > 0 && (n & (n - 1)) == 0; }

inline dim3 grid2d(int W, int rows, dim3 b) {
    return dim3((W + b.x - 1) / b.x, (rows + b.y - 1) / b.y);
}

Grid sim_grid(const fluid_t* h) { return Grid{h->cfg.sim_w, h->cfg.sim_h, h->roff, h->row0, h->row1}; }
Grid dye_grid(const fluid_t* h) { return Grid{h->cfg.dye_w, h->cfg.dye_h, h->droff, h->drow0, h->drow1}; }
// same grid, producing rows [row0-e, row1+e) clipped to the domain (redundant ghost-zone compute)
Grid sim_grid_ext(const fluid_t* h, int e) {
    Grid g = sim_grid(h);
    g.j_lo = std::max(h->row0 - e, 0); g.j_hi = std::min(h->row1 + e, h->cfg.sim_h);
    return g;
}

// LOCAL cell counts (owned + ghost rows): what the device buffers hold
size_t sim_cells(const fluid_t* h) { return (size_t)h->cfg.sim_w * h->lrows(); }
size_t dye_cells(const fluid_t* h) { return (size_t)h->cfg.dye_w * h->ldrows(); }

int check_launch(fluid_t* h, const char* what, int n = 1) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
        return fail(h, FLUID_ERR_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(e));
    h->launches += n;
    return FLUID_OK;
}

// dt of the current step()/pass, in device memory.  Stream-ordered 4-byte upload from a pageable
// host word (the driver stages it before returning), issued OUTSIDE any capture: an instantiated
// step graph therefore never bakes dt in, and the reference's calcDeltaTime() (S:1188-1194, a new
// dt every frame) replays the same graph.
int set_dt(fluid_t* h, float dt) {
    CU(cudaMemcpyAsync(h->dt_dev, &dt, sizeof(float), cudaMemcpyHostToDevice, h->stream));
    return FLUID_OK;
}

#include "halo.cuh"

// bytes per cell of each field: fp32 storage (float2 / float4 / float) or half storage (S:986-1006)
inline size_t vbytes(const fluid_t* h) { return h->half ? 4 : 8; }
inline size_t dbytes(const fluid_t* h) { return h->half ? 8 : 16; }
inline size_t sbytes(const fluid_t* h) { return h->half ? 2 : 4; }
int need_scratch(fluid_t* h, size_t floats) {
    if (floats <= h->scratch_floats) return FLUID_OK;
    CU(cudaStreamSynchronize(h->stream));
    cudaFree(h->scratch); h->scratch = nullptr; h->scratch_floats = 0;
    CU(cudaMalloc((void**)&h->scratch, floats * sizeof(float)));
    h->scratch_floats = floats;
    return FLUID_OK;
}
inline dim3 hs_grid(int W, int H) { return dim3((W + 63) / 64, (H + 3) / 4); }
const dim3 HS_BLOCK(64, 4);

// ---- the tiny-divergence map (jacobi.cuh): one byte per 128 x 32 cells of the GLOBAL grid -------------
int alloc_tiny_map(fluid_t* h) {
    cudaFree(h->tiny_map); h->tiny_map = nullptr;
    h->tiny_map_bytes = (size_t)tiny_map_w(h->cfg.sim_w) * tiny_map_h(h->cfg.sim_h);
    CU(cudaMalloc((void**)&h->tiny_map, h->tiny_map_bytes));
    CU(cudaMemsetAsync(h->tiny_map, 0, h->tiny_map_bytes, h->stream));
    return FLUID_OK;
}
// before a pass that recomputes divergence everywhere (the pass then flags cells itself)
int clear_tiny_map(fluid_t* h) {
    CU(cudaMemsetAsync(h->tiny_map, 0, h->tiny_map_bytes, h->stream));
    ++h->div_epoch;                       // every writer of divergence comes through here
    return FLUID_OK;
}
// divergence rows [j_lo, j_hi) came from outside (host write, neighbour rank): flag their cells
int scan_tiny(fluid_t* h, int j_lo, int j_hi) {
    if (j_hi <= j_lo) return FLUID_OK;
    dim3 b(256), g((h->cfg.sim_w + 255) / 256, j_hi - j_lo);
    tiny_scan_kernel<<<g, b, 0, h->active>>>(h->divergence, h->tiny_map, h->cfg.sim_w, h->roff, j_lo, j_hi);
    return check_launch(h, "tiny_scan_kernel");
}

// ---- Jacobi dispatch -----------------------------------------------------------------------------

constexpr int KMAX = 12;

// cuTensorMapEncodeTiled through the runtime (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) { cudaGetLastError(); return nullptr; }
        return (EncodeTiledFn)p;
    }();
    return fn;
}

// fp32 field of `rows` x W as a 2-D tensor; box = 128 columns x 3 rows, no swizzle, out-of-range
// elements read as zero (the blocked kernel never lets them reach a valid output)
bool encode_rows_map(CUtensorMap* tm, void* base, int W, int rows) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc || W % 4 != 0) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)W, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)W * sizeof(float)};
    const cuuint32_t box[2] = {128, 3};
    const cuuint32_t estr[2] = {1, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// (re)build the tensor maps after the pressure / divergence buffers were allocated
void build_tmaps(fluid_t* h) {
    h->tmaps.ok = false;
    if (h->half || h->cfg.sim_w % 4 != 0 || h->cfg.sim_w < 16) return;
    const int rows = h->lrows();
    h->tmaps.p_ptr[0] = h->pressure.read; h->tmaps.p_ptr[1] = h->pressure.write;
    h->tmaps.ok = encode_rows_map(&h->tmaps.p[0], h->pressure.read, h->cfg.sim_w, rows) &&
                  encode_rows_map(&h->tmaps.p[1], h->pressure.write, h->cfg.sim_w, rows) &&
                  encode_rows_map(&h->tmaps.d, h->divergence, h->cfg.sim_w, rows);
}

// staging of the blocked kernel.  Default: the per-lane cp.async (LDGSTS) ring — measured 4-6 % faster
// than the 2-D TMA boxes on B200 at 4096^2 x 50 (0.2575 vs 0.2685 ms per solve; the elected-lane issue +
// mbarrier poll sit in a one-warp CTA's only instruction stream; profiles/r02_jacobi_staging.md).
// FLUID_TB_STAGE=tma selects the tensor-map path (bit-identical results).
bool tb_use_tma(const fluid_t* h) {
    static const bool want_tma = getenv("FLUID_TB_STAGE") && !strcmp(getenv("FLUID_TB_STAGE"), "tma");
    return h->tmaps.ok && want_tma;
}

template <int K, bool SCALE>
int launch_tb(fluid_t* h, const JacobiArgs& a) {
    using T = TB<K>;
    const int nxw = (a.W + T::VALID - 1) / T::VALID;
    int nch = (a.out_hi - a.out_lo + a.rows_per_chunk - 1) / a.rows_per_chunk;
    if (a.nch1 > 0) nch = a.nch1 + (a.seg2_hi - a.seg2_lo + a.rows_per_chunk - 1) / a.rows_per_chunk;
    TmapPair maps;
    memset(&maps, 0, sizeof maps);
    // chained to the previous launch of the same solve by programmatic dependent launch (jacobi.cuh);
    // not while a graph is being captured, FLUID_PDL=0 turns it off
    static const bool pdl_off = getenv("FLUID_PDL") && !strcmp(getenv("FLUID_PDL"), "0");
    // tuning: run the SYNC instantiation everywhere (all hand-offs null) to time it against the plain one
    static const bool force_sync = getenv("FLUID_TB_FORCE_SYNC") && !strcmp(getenv("FLUID_TB_FORCE_SYNC"), "1");
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(nxw * nch); lc.blockDim = dim3(32); lc.stream = h->active;
    // FLUID_PDL_GRAPH=1: also while a step graph is captured (the launch becomes a programmatic edge)
    static const bool pdl_graph = getenv("FLUID_PDL_GRAPH") && !strcmp(getenv("FLUID_PDL_GRAPH"), "1");
    lc.attrs = attr; lc.numAttrs = (h->pdl_chain && !pdl_off && (!h->capturing || pdl_graph)) ? 1 : 0;
    if (tb_use_tma(h)) {
        const int k = (a.pin == h->tmaps.p_ptr[0]) ? 0 : 1;
        memcpy(maps.p, &h->tmaps.p[k], sizeof(CUtensorMap));
        memcpy(maps.d, &h->tmaps.d, sizeof(CUtensorMap));
        lc.dynamicSmemBytes = T::SMEM_TMA;
        { TbArgs<false> ta; static_cast<JacobiArgs&>(ta) = a; cudaLaunchKernelEx(&lc, jacobi_tb_kernel<K, SCALE, true, false>, ta, maps); }   // one warp per CTA
    } else if (h->tb_sync_on || force_sync) {         // slab launch with hand-offs (run_jacobi fills h->tb_sync)
        lc.dynamicSmemBytes = T::SMEM_LDGSTS;
        TbArgs<true> ta; static_cast<JacobiArgs&>(ta) = a; ta.sy = h->tb_sync;
        cudaLaunchKernelEx(&lc, jacobi_tb_kernel<K, SCALE, false, true>, ta, maps);
    } else {
        lc.dynamicSmemBytes = T::SMEM_LDGSTS;
        TbArgs<false> ta; static_cast<JacobiArgs&>(ta) = a;
        cudaLaunchKernelEx(&lc, jacobi_tb_kernel<K, SCALE, false, false>, ta, maps);
    }
    ++h->jacobi_kernel_launches;
    return check_launch(h, "jacobi_tb_kernel");
}

template <int K>
int launch_tb_k(fluid_t* h, const JacobiArgs& a, bool scale) {
    return scale ? launch_tb<K, true>(h, a) : launch_tb<K, false>(h, a);
}

// rows per warp stream: enough chunks that every SM holds its full complement of resident warps
// (single wave), rounded so that a stream's step count R + 2K is a multiple of the unroll U.
template <int K>
int tb_rows(const fluid_t* h, int W, int rows, int reserve = 0) {
    if (h->jacobi_rows_override > 0) return h->jacobi_rows_override;
    using T = TB<K>;
    const int nxw = (W + T::VALID - 1) / T::VALID;
    int occ = 0;
    if (tb_use_tma(h)) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, jacobi_tb_kernel<K, false, true, false>, 32, T::SMEM_TMA);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, jacobi_tb_kernel<K, false, false, false>, 32, T::SMEM_LDGSTS);
    if (occ < 1) occ = 1;
    if (h->jacobi_warps_per_sm > 0) occ = std::min(occ, h->jacobi_warps_per_sm);
    const int resident_warps = std::max(nxw, h->sm_count * occ - reserve);
    const int nch = std::max(1, resident_warps / nxw);
    int r = (rows + nch - 1) / nch;
    r = std::max(r, 4 * K);                 // keep the 2K warm-up rows a bounded fraction
    // round R up so that (R + 2K) % U == 0: no partially wasted unrolled block
    const int rem = (r + 2 * K) % T::U;
    if (rem) r += T::U - rem;
    return std::min(r, rows);
}

// rows_fixed > 0: use that chunk height (the boundary strips of a slab are one chunk each);
// reserve: resident streams to leave free on the chip (for a launch that runs beside this one)
int launch_tb_dyn(fluid_t* h, int K, JacobiArgs a, bool scale, int rows_fixed = 0, int reserve = 0) {
    const int rows = a.out_hi - a.out_lo;
    switch (K) {
#define CASE(KK) case KK: a.rows_per_chunk = rows_fixed > 0 ? rows_fixed : tb_rows<KK>(h, a.W, rows, reserve); return launch_tb_k<KK>(h, a, scale);
        CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) CASE(10) CASE(11) CASE(12)
#undef CASE
    }
    return fail(h, FLUID_ERR_INVALID, "temporal block depth %d out of range", K);
}

bool tb_eligible(const fluid_t* h) {
    return !h->half && (h->cfg.sim_w % 4 == 0) && h->cfg.sim_w >= 16 && h->cfg.sim_h >= 2;
}

// `iters` sweeps reading pressure.read, result in pressure.read (swaps like S:1265).
// scale_first: fold p <- PRESSURE*p (clear pass) into the first sweep's loads.
// On a slab: before a launch of depth K the neighbours' K rows of p are exchanged (K+1 for the last
// launch, which also produces one row beyond each slab edge so that gradientSubtract needs no
// message of its own); divergence ghosts are exchanged once per solve (it is constant in the loop).
int run_jacobi(fluid_t* h, int iters, bool scale_first, int* launches_out) {
    int nl = 0;
    const bool p_ghosts_mirrored = h->p_mirror_valid;    // every path below rewrites pressure
    h->p_mirror_valid = false;
    const int W = h->cfg.sim_w, H = h->cfg.sim_h;
    JacobiArgs a{};
    a.div = h->divergence; a.W = W; a.H = H; a.row_off = h->roff; a.out_lo = h->row0; a.out_hi = h->row1;
    a.scale = h->cfg.pressure;
    a.err = h->halo_flag;
    a.tiny_map = h->tiny_map;
    int kb = h->cfg.jacobi_block > 0 ? h->cfg.jacobi_block : 10;  // tuned on B200: profiles/r01_tune_jacobi.txt
    kb = std::min(kb, KMAX);
    if (h->slab()) kb = std::max(1, std::min(kb, h->G - 1));
    const bool naive = (h->cfg.flags & FLUID_FLAG_NAIVE_JACOBI) || kb == 1;
    if (h->half) {                                   // fp16 storage: the literal loop, every sweep rounds to fp16 (S:1253-1266)
        const int n = W * H;
        if (scale_first) {
            hs::scale_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>((const hs::h1*)h->pressure.read, (hs::h1*)h->pressure.write, n, h->cfg.pressure);
            int rc = check_launch(h, "hs::scale_kernel"); if (rc) return rc;
            swap_p(h); ++nl;
        }
        for (int k = 0; k < iters; ++k) {
            if (W % 8 == 0 && W >= 64) {
                dim3 b(32, 8), g((W / 8 + 31) / 32, (H + 7) / 8);
                hs::jacobi8_kernel<<<g, b, 0, h->stream>>>((const hs::h1*)h->pressure.read, (const hs::h1*)h->divergence, (hs::h1*)h->pressure.write, W, H);
            } else {
                hs::jacobi_kernel<<<hs_grid(W, H), HS_BLOCK, 0, h->stream>>>((const hs::h1*)h->pressure.read, (const hs::h1*)h->divergence, (hs::h1*)h->pressure.write, W, H);
            }
            ++h->jacobi_kernel_launches;
            int rc = check_launch(h, "hs::jacobi_kernel"); if (rc) return rc;
            swap_p(h); ++nl;
        }
        if (launches_out) *launches_out = nl;
        return FLUID_OK;
    }
    if (iters <= 0) {
        if (scale_first) {   // clear pass alone (owned + ghost rows; ghosts are refreshed before use anyway)
            const size_t n = sim_cells(h);
            scale_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(
                (const float*)h->pressure.read, (float*)h->pressure.write, n, h->cfg.pressure);
            int rc = check_launch(h, "scale_kernel"); if (rc) return rc;
            swap_p(h); ++nl;
        }
        if (launches_out) *launches_out = nl;
        return FLUID_OK;
    }
    const bool blocked = tb_eligible(h) && !naive;
    const int nlaunch = blocked ? (iters + kb - 1) / kb : iters;
    const int base = iters / nlaunch, extra = iters % nlaunch;
    // Slab halos.  Communication-avoiding form (deep): ONE group per solve carries iters+1 rows of
    // pressure and iters rows of divergence; launch i then produces owned rows +- (sweeps still to
    // come + 1), so later launches find their input already there (~1 % redundant rows instead of
    // one latency-bound message per launch).  If the ghost zone is too thin for that (iterations
    // raised after creation) fall back to one K-row message per launch.
    const bool deep = h->slab() && (iters + 1 <= h->G) && (iters + 1 <= h->row1 - h->row0);
    // Optional overlap (deep + blocked, either transport): the exchange and the two boundary strips of
    // launch 1 — the only rows of it that read ghost rows — go to a second stream, the interior rows
    // [row0+K1, row1-K1) of launch 1 run meanwhile on the compute stream.
    // Default OFF: measured on 2 B200 (4096 x 4096 per rank, 50 iterations) the split costs more than it hides —
    // 0.327 ms per solve with it, 0.277 ms without (same box, profiles/r02_scaling.md); FLUID_HALO_OVERLAP=1 enables it.
    static const bool overlap_off = !(getenv("FLUID_HALO_OVERLAP") && !strcmp(getenv("FLUID_HALO_OVERLAP"), "1"));
    const int K1 = base + (extra ? 1 : 0);
    const bool overlap = deep && blocked && !overlap_off && h->stream2 && (h->row1 - h->row0) >= 2 * K1 + 4 * K1;
    // Peer-memory transport, two or more blocked launches: the last launch of this solve stores the pressure
    // rows the neighbours need next time into their ghost rows itself (TbSync in jacobi.cuh), and if the
    // previous solve did so — nothing wrote pressure since — this solve starts without a pressure message.
    // FLUID_HALO_MIRROR=1 enables it (default: the explicit exchange).
    static const bool mirror_off = !(getenv("FLUID_HALO_MIRROR") && !strcmp(getenv("FLUID_HALO_MIRROR"), "1"));
    const bool mirror = deep && blocked && h->p2p && nlaunch >= 2 && !mirror_off && !overlap && !tb_use_tma(h);
    const bool p_in_place = mirror && p_ghosts_mirrored && h->p_mirror_rows >= iters + 1;
    unsigned* const my_flags = h->slab() ? (unsigned*)(h->arena + h->off_flags) : nullptr;
    auto peer_flags = [&](int side) { return (unsigned*)(h->peer[side].base + h->peer[side].off_flags); };
    if (h->slab()) {
        if (overlap) {
            CU(cudaEventRecord(h->ev_fork, h->stream));
            CU(cudaStreamWaitEvent(h->stream2, h->ev_fork, 0));
            h->active = h->stream2;
        }
        if (deep) {
            const HaloItem itp = {h->pressure.read, (size_t)W * sizeof(float), h->roff, h->row0, h->row1, iters + 1, HB_PRESSURE};
            const HaloItem itd = {h->divergence, (size_t)W * sizeof(float), h->roff, h->row0, h->row1, iters, HB_DIVERGENCE};
            // divergence is constant during a solve and often across solves (a host that iterates the solve on
            // one right-hand side, bench.py's loop): its ghost rows — and their tiny-value flags — are still in
            // place unless some pass rewrote divergence since they were last received (SPMD-identical decision)
            const bool send_div = h->div_sent_epoch != h->div_epoch || h->div_sent_rows < iters;
            HaloItem it[2];
            int nitems = 0;
            if (!p_in_place) it[nitems++] = itp;
            if (send_div) it[nitems++] = itd;
            // the neighbours' divergence rows get their tiny values flagged like the local producers do:
            // inside the wait kernel on the peer-memory path, by a scan kernel after the NCCL group
            h->scan.div = h->divergence; h->scan.map = h->tiny_map; h->scan.W = W; h->scan.row_off = h->roff;
            h->scan.lo0 = std::max(h->row0 - iters, 0); h->scan.hi0 = h->row0;
            h->scan.lo1 = h->row1; h->scan.hi1 = std::min(h->row1 + iters, H);
            h->scan_pending = h->p2p && send_div;
            int rc = nitems ? exchange_many(h, it, nitems) : FLUID_OK;
            if (send_div) { h->div_sent_epoch = h->div_epoch; h->div_sent_rows = iters; }
            if (!rc && !h->p2p && send_div) {
                rc = scan_tiny(h, h->scan.lo0, h->scan.hi0);
                if (!rc) rc = scan_tiny(h, h->scan.lo1, h->scan.hi1);
            }
            h->scan_pending = false;
            if (rc) { h->active = h->stream; return rc; }
        } else {
            const int kmax = base + (extra ? 1 : 0);
            int rc = exchange_rows(h, HB_DIVERGENCE, h->divergence, (size_t)W * sizeof(float), h->roff, h->row0, h->row1, kmax);
            if (rc) return rc;
            if ((rc = scan_tiny(h, std::max(h->row0 - kmax, 0), h->row0))) return rc;
            if ((rc = scan_tiny(h, h->row1, std::min(h->row1 + kmax, H)))) return rc;
        }
    }
    int remaining = iters;
    for (int k = 0; k < nlaunch; ++k) {
        const int K = base + (k < extra ? 1 : 0);
        const bool last = (k == nlaunch - 1);
        remaining -= K;
        a.pin = (const float*)h->pressure.read; a.pout = (float*)h->pressure.write;
        a.out_lo = h->row0; a.out_hi = h->row1;
        if (h->slab()) {
            int ext;
            if (deep) {
                ext = remaining + 1;
            } else {
                ext = last ? 1 : 0;
                int rc = exchange_rows(h, HB_PRESSURE, h->pressure.read, (size_t)W * sizeof(float), h->roff, h->row0, h->row1, K + ext);
                if (rc) return rc;
            }
            a.out_lo = std::max(h->row0 - ext, 0); a.out_hi = std::min(h->row1 + ext, H);
        }
        h->tb_sync = TbSync{}; h->tb_sync_on = false;
        if (mirror) {
            const unsigned seq = h->mir_seq + 1;
            h->tb_sync_on = (k == 0 && p_in_place) || k == nlaunch - 2 || last;
            static const bool dbg = getenv("FLUID_DEBUG_HALO_TIMING") != nullptr;
            if (dbg) h->tb_sync.dbg = (unsigned long long*)(h->arena + h->off_flags + 512);
            h->tb_sync.own_lo = h->row0; h->tb_sync.own_hi = h->row1;
            if (k == 0 && p_in_place) {                          // wait for the previous solve's mirrored rows
                for (int s = 0; s < 2; ++s)
                    if (h->peer[s].present) h->tb_sync.pre_wait[s] = my_flags + 66 + s;
                h->tb_sync.pre_seq = h->mir_seq;
            }
            if (k == nlaunch - 2) {                              // last reader of the ghost rows the neighbours will overwrite
                h->tb_sync.ticket = my_flags + 72;
                for (int s = 0; s < 2; ++s)
                    if (h->peer[s].present) h->tb_sync.done_flag[s] = peer_flags(s) + (s == 0 ? 65 : 64);
                h->tb_sync.done_seq = seq;
            }
            if (last) {
                const int pidx = ((char*)h->pressure.write == h->arena + h->off_p[0]) ? 0 : 1;
                for (int s = 0; s < 2; ++s) {
                    const fluid::Peer& P = h->peer[s];
                    if (!P.present) continue;
                    h->tb_sync.mirror[s] = (float*)(P.base + P.off_p[pidx]) - (ptrdiff_t)P.roff * W;
                    h->tb_sync.mir_lo[s] = s == 0 ? h->row0 : h->row1 - (iters + 1);
                    h->tb_sync.mir_hi[s] = s == 0 ? h->row0 + (iters + 1) : h->row1;
                    h->tb_sync.mir_wait[s] = my_flags + 64 + s;
                    h->tb_sync.done_flag[s] = peer_flags(s) + (s == 0 ? 67 : 66);
                }
                h->tb_sync.mir_seq = seq; h->tb_sync.ticket = my_flags + 73; h->tb_sync.done_seq = seq;
            }
        }
        const bool sc = scale_first && k == 0;
        int rc;
        if (blocked && overlap && k == 0) {
            // boundary strips [out_lo, row0+K) and [row1-K, out_hi) behind the exchange on stream2 ...
            const int nxw = (W + 127) / 128 + 8;             // upper bound of the strips' stream count (any K)
            JacobiArgs bnd = a;
            bnd.out_lo = a.out_lo; bnd.out_hi = std::min(h->row0 + K, a.out_hi);
            bnd.seg2_lo = std::max(h->row1 - K, bnd.out_hi); bnd.seg2_hi = a.out_hi;
            const int strip = std::max(bnd.out_hi - bnd.out_lo, bnd.seg2_hi - bnd.seg2_lo);
            bnd.nch1 = 1;
            rc = launch_tb_dyn(h, K, bnd, sc, strip);        // h->active == stream2
            h->active = h->stream;
            if (rc) return rc;
            CU(cudaEventRecord(h->ev_join, h->stream2));
            // ... the interior meanwhile on the compute stream, sized to leave the strips' slots free
            JacobiArgs in = a;
            in.out_lo = bnd.out_hi; in.out_hi = bnd.seg2_lo;
            rc = launch_tb_dyn(h, K, in, sc, 0, 2 * nxw);
            if (rc) return rc;
            CU(cudaStreamWaitEvent(h->stream, h->ev_join, 0));
        } else if (blocked) {
            // programmatic dependent launch: behind another blocked launch of this solve, and — first launch —
            // behind whatever kernel precedes it on the stream (the previous solve's last launch in a host loop
            // of solves; a kernel without griddepcontrol.launch_dependents simply triggers at its end)
            h->pdl_chain = !(overlap && k <= 1);
            rc = launch_tb_dyn(h, K, a, sc);
            h->pdl_chain = false; h->tb_sync_on = false;
        } else if (tb_eligible(h)) {
            dim3 b(32, 8);
            dim3 g((W / 4 + b.x - 1) / b.x, (a.out_hi - a.out_lo + b.y - 1) / b.y);
            if (sc) jacobi_sweep_kernel<true><<<g, b, 0, h->stream>>>(a);
            else jacobi_sweep_kernel<false><<<g, b, 0, h->stream>>>(a);
            ++h->jacobi_kernel_launches;
            rc = check_launch(h, "jacobi_sweep_kernel");
        } else {
            dim3 b(64, 4);
            jacobi_scalar_kernel<<<grid2d(W, a.out_hi - a.out_lo, b), b, 0, h->stream>>>(a, sc);
            ++h->jacobi_kernel_launches;
            rc = check_launch(h, "jacobi_scalar_kernel");
        }
        if (rc) return rc;
        swap_p(h); ++nl;
    }
    if (mirror) { ++h->mir_seq; h->p_mirror_valid = true; h->p_mirror_rows = iters + 1; }
    if (launches_out) *launches_out = nl;
    return FLUID_OK;
}

int alloc_fields(fluid_t* h) {
    const size_t n = sim_cells(h), nd = dye_cells(h);
    if (h->slab()) {
        // one allocation, so that a single CUDA IPC handle maps everything a neighbour may write into
        auto al = [](size_t b) { return (b + 1023) & ~(size_t)1023; };
        size_t o = 0;
        h->off_flags = o; o += 1024;
        for (int k = 0; k < 2; ++k) { h->off_v[k] = o; o += al(n * sizeof(float2)); }
        for (int k = 0; k < 2; ++k) { h->off_p[k] = o; o += al(n * sizeof(float)); }
        for (int k = 0; k < 2; ++k) { h->off_dye[k] = o; o += al(nd * sizeof(float4)); }
        h->off_div = o; o += al(n * sizeof(float));
        const size_t off_curl = o; o += al(n * sizeof(float));
        h->arena_bytes = o;
        CU(cudaMalloc((void**)&h->arena, o));
        CU(cudaMemsetAsync(h->arena, 0, o, h->stream));
        h->velocity.read = h->arena + h->off_v[0]; h->velocity.write = h->arena + h->off_v[1];
        h->pressure.read = h->arena + h->off_p[0]; h->pressure.write = h->arena + h->off_p[1];
        h->dye.read = h->arena + h->off_dye[0]; h->dye.write = h->arena + h->off_dye[1];
        h->divergence = (float*)(h->arena + h->off_div); h->curl = (float*)(h->arena + off_curl);
        h->par_v = h->par_p = h->par_dye = 0;
    } else {
        CU(cudaMalloc(&h->velocity.read, n * vbytes(h)));
        CU(cudaMalloc(&h->velocity.write, n * vbytes(h)));
        CU(cudaMalloc(&h->dye.read, nd * dbytes(h)));
        CU(cudaMalloc(&h->dye.write, nd * dbytes(h)));
        CU(cudaMalloc(&h->pressure.read, n * sbytes(h)));
        CU(cudaMalloc(&h->pressure.write, n * sbytes(h)));
        CU(cudaMalloc((void**)&h->divergence, n * sbytes(h)));
        CU(cudaMalloc((void**)&h->curl, n * sbytes(h)));
        CU(cudaMemsetAsync(h->velocity.read, 0, n * vbytes(h), h->stream));
        CU(cudaMemsetAsync(h->velocity.write, 0, n * vbytes(h), h->stream));
        CU(cudaMemsetAsync(h->pressure.read, 0, n * sbytes(h), h->stream));
        CU(cudaMemsetAsync(h->pressure.write, 0, n * sbytes(h), h->stream));
        CU(cudaMemsetAsync(h->divergence, 0, n * sbytes(h), h->stream));
        CU(cudaMemsetAsync(h->curl, 0, n * sbytes(h), h->stream));
    }
    { int rc = alloc_tiny_map(h); if (rc) return rc; }
    build_tmaps(h);
    h->div_sent_epoch = 0;                               // fresh buffers: no divergence ghost rows in place yet
    if (h->half) {
        hs::fill_alpha_kernel<<<(unsigned)((nd + 255) / 256), 256, 0, h->stream>>>((hs::h4*)h->dye.read, nd);
        hs::fill_alpha_kernel<<<(unsigned)((nd + 255) / 256), 256, 0, h->stream>>>((hs::h4*)h->dye.write, nd);
    } else {
        fill_alpha_kernel<<<(unsigned)((nd + 255) / 256), 256, 0, h->stream>>>((float4*)h->dye.read, nd);
        fill_alpha_kernel<<<(unsigned)((nd + 255) / 256), 256, 0, h->stream>>>((float4*)h->dye.write, nd);
    }
    return check_launch(h, "fill_alpha_kernel", 2);
}

void free_fields(fluid_t* h) {
    if (h->arena) {
        for (auto& p : h->peer) if (p.present && p.base) { cudaIpcCloseMemHandle(p.base); p.base = nullptr; p.present = false; }
        cudaFree(h->arena); h->arena = nullptr;
    } else {
        cudaFree(h->velocity.read); cudaFree(h->velocity.write);
        cudaFree(h->dye.read); cudaFree(h->dye.write);
        cudaFree(h->pressure.read); cudaFree(h->pressure.write);
        cudaFree(h->divergence); cudaFree(h->curl);
    }
    h->velocity = Pair{}; h->dye = Pair{}; h->pressure = Pair{};
    h->divergence = h->curl = nullptr;
    cudaFree(h->tiny_map); h->tiny_map = nullptr;
    h->tmaps.ok = false;
}

// pointer to the first OWNED row of a field's .read buffer, plus its owned extent
int field_info(const fluid_t* h, int field, void** ptr, int* w, int* rows, int* ch) {
    const size_t so = (size_t)h->G * h->cfg.sim_w, doff_ = (size_t)h->Gd * h->cfg.dye_w;
    switch (field) {
        case FLUID_FIELD_VELOCITY: *ptr = (float2*)h->velocity.read + so; *w = h->cfg.sim_w; *rows = h->row1 - h->row0; *ch = 2; return 0;
        case FLUID_FIELD_DYE: *ptr = (float4*)h->dye.read + doff_; *w = h->cfg.dye_w; *rows = h->drow1 - h->drow0; *ch = 4; return 0;
        case FLUID_FIELD_PRESSURE: *ptr = (float*)h->pressure.read + so; *w = h->cfg.sim_w; *rows = h->row1 - h->row0; *ch = 1; return 0;
        case FLUID_FIELD_DIVERGENCE: *ptr = h->divergence + so; *w = h->cfg.sim_w; *rows = h->row1 - h->row0; *ch = 1; return 0;
        case FLUID_FIELD_CURL: *ptr = h->curl + so; *w = h->cfg.sim_w; *rows = h->row1 - h->row0; *ch = 1; return 0;
    }
    return -1;
}

// Multi-GPU: an advection back-trace that needed a row outside the ghost zone set the device flag;
// never clamp silently (SURVEY §7) — report it at the next synchronisation point.
int check_halo(fluid_t* h) {
    int flag = 0;
    CU(cudaMemcpyAsync(&flag, h->halo_flag, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (flag) CU(cudaMemsetAsync(h->halo_flag, 0, sizeof(int), h->stream));   // report once; the caller decides what to do next
    if (flag == 2)
        return fail(h, FLUID_ERR_HALO, "peer-memory halo exchange timed out waiting for a neighbour rank");
    if (flag == 3)
        return fail(h, FLUID_ERR_CUDA, "jacobi_tb_kernel: a TMA staging barrier never completed");
    if (flag)
        return fail(h, FLUID_ERR_HALO, "advection back-trace left the %d-row ghost zone: |v|*dt exceeds it; "
                    "re-create the slab handle with a taller halo (FLUID_HALO_ROWS)", h->G);
    return FLUID_OK;
}

int not_on_slab(fluid_t* h, const char* what) {
    return fail(h, FLUID_ERR_INVALID, "%s is a single-GPU test entry point; a slab handle supports "
                "fluid_step / fluid_splat / fluid_pass_pressure_solve / fluid_pass_jacobi / read / write", what);
}

// Row ownership + ghost-zone heights of rank `rank` of `world` for a sim_h / dye_h grid (DESIGN.md §7).
// Returns false when the slabs are too short for the minimum 14-row halo.
bool slab_geometry(fluid_t* h, int H, int Hd, int iters) {
    const int rank = h->rank, world = h->world;
    h->row0 = (int)((long long)H * rank / world);  h->row1 = (int)((long long)H * (rank + 1) / world);
    h->drow0 = (int)((long long)Hd * rank / world); h->drow1 = (int)((long long)Hd * (rank + 1) / world);
    h->G = h->Gd = 0;
    if (world > 1) {
        // ghost rows: enough for the advection back-trace (3 ghost-compute rows + dt*|v|max + 2)
        // and for the deep Jacobi halo (iterations + 1).
        // 64 rows: a back-trace of up to (64 - 5) rows per step, i.e. |v| up to 3540 texels/s at the reference's
        // dt <= 1/60 (vorticity clamps |v| to 1000, a pointer flick of half the canvas splats 3000); the rows
        // cost ~4 MB of halo traffic per step per neighbour at 4096 columns, microseconds on NVLink
        int g = std::max(64, iters + 2);
        if (const char* e = getenv("FLUID_HALO_ROWS")) g = std::max(14, atoi(e));
        // every rank must arrive at the SAME halo height (message sizes must match), so clip with
        // the height of the shortest slab, which all ranks can compute: floor(H / world)
        const int per = std::max(1, (Hd + H - 1) / H);
        g = std::min(g, std::min(H / world, (Hd / world) / per));
        h->G = g;
        h->Gd = g * per;                              // same physical reach on the dye grid
        if (g < 14) return false;
    }
    h->roff = h->row0 - h->G; h->droff = h->drow0 - h->Gd;
    return true;
}

// shared by fluid_create and fluid_create_slab
int create_common(const fluid_config* cfg, int rank, int world, const void* uid, fluid_t** out) {
    fluid_t* h = nullptr;
    if (!cfg || !out) return fail(h, FLUID_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->sim_w < 1 || cfg->sim_h < 1 || cfg->dye_w < 1 || cfg->dye_h < 1)
        return fail(h, FLUID_ERR_INVALID, "bad resolution %dx%d / %dx%d", cfg->sim_w, cfg->sim_h,
                    cfg->dye_w, cfg->dye_h);
    if (world < 1 || rank < 0 || rank >= world) return fail(h, FLUID_ERR_INVALID, "bad rank %d of %d", rank, world);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(h, FLUID_ERR_NO_DEVICE, "no CUDA device: libfluid_b200 has no CPU path");
    }
    int dev = cfg->device;
    if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) dev = 0; }
    if (dev >= ndev) return fail(h, FLUID_ERR_INVALID, "device %d of %d", dev, ndev);
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess || prop.major != 10)
        return fail(h, FLUID_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only",
                    dev, prop.major, prop.minor);
    if (cudaSetDevice(dev) != cudaSuccess) return fail(h, FLUID_ERR_CUDA, "cudaSetDevice(%d)", dev);

    h = new fluid();
    h->cfg = *cfg;
    h->device = dev;
    h->sm_count = prop.multiProcessorCount;
    if (!(h->cfg.aspect > 0.0f)) h->cfg.aspect = (float)((double)cfg->sim_w / (double)cfg->sim_h);
    h->aspect_d = (cfg->aspect > 0.0f) ? (double)cfg->aspect : (double)cfg->sim_w / (double)cfg->sim_h;
    h->splat_radius_d = (double)cfg->splat_radius;
    h->rank = rank; h->world = world;
    h->half = (cfg->flags & FLUID_FLAG_HALF_STORAGE) != 0;
    if (h->half && world > 1) {
        int rc = fail(nullptr, FLUID_ERR_INVALID, "FLUID_FLAG_HALF_STORAGE is a single-GPU mode");
        delete h; return rc;
    }
    if (!slab_geometry(h, cfg->sim_h, cfg->dye_h, cfg->pressure_iterations)) {
        int rc = fail(nullptr, FLUID_ERR_INVALID, "slabs of %d rows are too short for a 14-row halo: use fewer GPUs", cfg->sim_h / world);
        delete h; return rc;
    }
    if (const char* e = getenv("FLUID_JACOBI_ROWS")) h->jacobi_rows_override = atoi(e);
    if (const char* e = getenv("FLUID_JACOBI_WARPS")) h->jacobi_warps_per_sm = atoi(e);
    auto body = [&]() -> int {
        CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        h->active = h->stream;
        if (world > 1) {
            CU(cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking));
            CU(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
        }
        for (auto& e : h->mark) CU(cudaEventCreate(&e));
        for (auto& e : h->tev) CU(cudaEventCreate(&e));
        CU(cudaMalloc((void**)&h->halo_flag, sizeof(int)));
        CU(cudaMemsetAsync(h->halo_flag, 0, sizeof(int), h->stream));
        CU(cudaMalloc((void**)&h->dt_dev, sizeof(float)));
        CU(cudaMemsetAsync(h->dt_dev, 0, sizeof(float), h->stream));
        int r = alloc_fields(h); if (r) return r;
        CU(cudaStreamSynchronize(h->stream));
        if (world > 1) {
            ncdl::Api& N = ncdl::api();
            if (!N.handle) return fail(h, FLUID_ERR_NCCL, "NCCL not available: %s", N.why);
            ncdl::ncclUniqueId id;
            memcpy(&id, uid, sizeof id);
            int rc = N.CommInitRank(&h->comm, world, id, rank);
            if (rc) return fail(h, FLUID_ERR_NCCL, "ncclCommInitRank failed: %s", N.GetErrorString(rc));
        }
        return FLUID_OK;
    };
    int rc = body();
    if (rc != FLUID_OK) { g_create_error = h->err; fluid_destroy(h); return rc; }
    *out = h;
    return FLUID_OK;
}

// createFBO's clear to (0,0,0,1) (S:1059) of the bloom FBO, for either storage
inline void clear_fbo(float4* p, size_t n, cudaStream_t s) { fill_alpha_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(p, n); }
inline void clear_fbo(hs::h4* p, size_t n, cudaStream_t s) { hs::fill_alpha_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(p, n); }

// The post-FX chain of fluid_render_postfx on T4 / T1 textures: float4 / float for fp32 storage,
// hs::h4 / hs::h1 for FLUID_FLAG_HALF_STORAGE, where (as in the reference, S:1012-1043 and S:1300)
// the bloom FBO, the pyramid, both sunrays FBOs and the mask in dye.write are fp16.  `tmp` collects
// the per-call device allocations; the caller frees them.
template <typename T4, typename T1>
int render_postfx_chain(fluid_t* h, int width, int height, const fluid_postfx* fx, const float* dither_rgb, int dw, int dh,
                        float back_r, float back_g, float back_b, float* host_rgba, float* host_bloom, float* host_sunrays,
                        int bw, int bh, int sw, int sh, std::vector<void*>& tmp) {
    constexpr bool half = !std::is_same<T4, float4>::value;
    auto dalloc = [&](size_t bytes) -> void* { void* p = nullptr; if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr; tmp.push_back(p); return p; };
    const size_t cells = (size_t)width * height;
    if (cells > h->frame_cells) {
        CU(cudaStreamSynchronize(h->stream));
        cudaFree(h->frame); h->frame = nullptr; h->frame_cells = 0;
        CU(cudaMalloc((void**)&h->frame, cells * sizeof(float4)));
        h->frame_cells = cells;
    }
    const int Wd = h->cfg.dye_w, Hd = h->cfg.dye_h;
    const T4* dye = (const T4*)h->dye.read;
    dim3 b(32, 8);
    T4* bloom = (T4*)dalloc((size_t)bw * bh * sizeof(T4));
    T1* sun = (T1*)dalloc((size_t)sw * sh * sizeof(T1));
    T1* sun2 = (T1*)dalloc((size_t)sw * sh * sizeof(T1));
    float* dith = (float*)dalloc((size_t)dw * dh * 3 * sizeof(float));
    if (!bloom || !sun || !sun2 || !dith) return fail(h, FLUID_ERR_NOMEM, "out of device memory for the post-FX targets");
    // fp16 storage: host_bloom / host_sunrays are the fp16 textures widened (exactly) on the device
    float* wide_bloom = nullptr; float* wide_sun = nullptr;
    if (half && host_bloom && !(wide_bloom = (float*)dalloc((size_t)bw * bh * 4 * sizeof(float))))
        return fail(h, FLUID_ERR_NOMEM, "out of device memory for the bloom read-back");
    if (half && host_sunrays && !(wide_sun = (float*)dalloc((size_t)sw * sh * sizeof(float))))
        return fail(h, FLUID_ERR_NOMEM, "out of device memory for the sunrays read-back");
    CU(cudaMemcpyAsync(dith, dither_rgb, (size_t)dw * dh * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    clear_fbo(bloom, (size_t)bw * bh, h->stream);
    // ---- applyBloom(dye.read, bloom) ----------------------------------------------------------
    struct Lv { T4* p; int w, h; };
    std::vector<Lv> pyr;
    for (int i = 0; i < fx->bloom_iterations; ++i) {
        const int pw = bw >> (i + 1), ph = bh >> (i + 1);
        if (pw < 2 || ph < 2) break;
        T4* p = (T4*)dalloc((size_t)pw * ph * sizeof(T4));
        if (!p) return fail(h, FLUID_ERR_NOMEM, "out of device memory for the bloom pyramid");
        pyr.push_back({p, pw, ph});
    }
    int nk = 1;
    if (pyr.size() >= 2) {
        const double knee = fx->bloom_threshold * fx->bloom_soft_knee + 0.0001;
        bloom_prefilter_kernel<<<grid2d(bw, bh, b), b, 0, h->stream>>>(
            dye, Wd, Hd, bloom, bw, bh, (float)(fx->bloom_threshold - knee),
            (float)(knee * 2), (float)(0.25 / knee), (float)fx->bloom_threshold);
        ++nk;
        Lv last{bloom, bw, bh};
        for (auto& d : pyr) {
            box4_kernel<<<grid2d(d.w, d.h, b), b, 0, h->stream>>>(last.p, last.w, last.h, d.p, d.w, d.h, 1.0f, 0);
            last = d; ++nk;
        }
        for (int i = (int)pyr.size() - 2; i >= 0; --i) {
            box4_kernel<<<grid2d(pyr[i].w, pyr[i].h, b), b, 0, h->stream>>>(last.p, last.w, last.h, pyr[i].p, pyr[i].w, pyr[i].h, 1.0f, 1);
            last = pyr[i]; ++nk;
        }
        box4_kernel<<<grid2d(bw, bh, b), b, 0, h->stream>>>(last.p, last.w, last.h, bloom, bw, bh, (float)fx->bloom_intensity, 0);
        ++nk;
    }
    // ---- applySunrays(dye.read, dye.write, sunrays); blur(sunrays, sunraysTemp, 1) ---------------
    sunrays_mask_kernel<<<grid2d(Wd, Hd, b), b, 0, h->stream>>>(dye, (T4*)h->dye.write, Wd, Hd);
    sunrays_kernel<<<grid2d(sw, sh, b), b, 0, h->stream>>>((const T4*)h->dye.write, Wd, Hd, sun, sw, sh, (float)fx->sunrays_weight);
    blur3_kernel<<<grid2d(sw, sh, b), b, 0, h->stream>>>(sun, sun2, sw, sh, (float)(1.0 / (double)sw), 0.0f);
    blur3_kernel<<<grid2d(sw, sh, b), b, 0, h->stream>>>(sun2, sun, sw, sh, 0.0f, (float)(1.0 / (double)sh));
    // ---- drawColor + drawDisplay ---------------------------------------------------------------------
    display_full_kernel<<<grid2d(width, height, b), b, 0, h->stream>>>(
        dye, Wd, Hd, bloom, bw, bh, sun, sw, sh, dith, dw, dh, h->frame, width, height,
        back_r, back_g, back_b, h->background, h->cfg.aspect,
        make_float4((float)(1.0 / (double)width), (float)(1.0 / (double)height), (float)((double)width / (double)dw), (float)((double)height / (double)dh)));
    nk += 5;
    const float* out_bloom = (const float*)bloom;
    const float* out_sun = (const float*)sun;
    if (wide_bloom) {
        const size_t n = (size_t)bw * bh * 4;
        hs::widen_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((const hs::h1*)bloom, wide_bloom, n);
        out_bloom = wide_bloom; ++nk;
    }
    if (wide_sun) {
        const size_t n = (size_t)sw * sh;
        hs::widen_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((const hs::h1*)sun, wide_sun, n);
        out_sun = wide_sun; ++nk;
    }
    int r = check_launch(h, "post-FX kernels", nk); if (r) return r;
    CU(cudaMemcpyAsync(host_rgba, h->frame, cells * sizeof(float4), cudaMemcpyDeviceToHost, h->stream));
    if (host_bloom) CU(cudaMemcpyAsync(host_bloom, out_bloom, (size_t)bw * bh * 4 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (host_sunrays) CU(cudaMemcpyAsync(host_sunrays, out_sun, (size_t)sw * sh * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return FLUID_OK;
}

}  // namespace

// ================================================================================================
extern "C" {

int fluid_abi_version(void) { return FLUID_ABI_VERSION; }

void fluid_config_default(fluid_config* c) {
    memset(c, 0, sizeof *c);
    c->sim_w = c->sim_h = 128;            // SIM_RESOLUTION  S:60
    c->dye_w = c->dye_h = 1024;           // DYE_RESOLUTION  S:61
    c->density_dissipation = 1.0f;        // S:63
    c->velocity_dissipation = 0.2f;       // S:64
    c->pressure = 0.8f;                   // S:65
    c->pressure_iterations = 20;          // S:66
    c->curl = 30.0f;                      // S:67
    c->splat_radius = 0.25f;              // S:68
    c->aspect = 1.0f;
    c->device = -1;
    c->flags = 0;
    c->jacobi_block = 0;
}

// getResolution, S:1612-1624
void fluid_get_resolution(int resolution, int canvas_w, int canvas_h, int* out_w, int* out_h) {
    double aspect = (double)canvas_w / (double)canvas_h;
    if (aspect < 1.0) aspect = 1.0 / aspect;
    // Math.round: half away from zero for positive values == floor(x + 0.5)
    const int mn = (int)(resolution + 0.5);
    const int mx = (int)((double)resolution * aspect + 0.5);
    if (canvas_w > canvas_h) { *out_w = mx; *out_h = mn; }
    else { *out_w = mn; *out_h = mx; }
}

const char* fluid_last_error(fluid_t* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int fluid_create(const fluid_config* cfg, fluid_t** out) { return create_common(cfg, 0, 1, nullptr, out); }

int fluid_nccl_unique_id(void* out_uid, size_t uid_bytes) {
    if (!out_uid || uid_bytes < sizeof(ncdl::ncclUniqueId)) return fail(nullptr, FLUID_ERR_INVALID, "uid buffer must hold 128 bytes");
    ncdl::Api& N = ncdl::api();
    if (!N.handle) return fail(nullptr, FLUID_ERR_NCCL, "NCCL not available: %s", N.why);
    ncdl::ncclUniqueId id;
    int rc = N.GetUniqueId(&id);
    if (rc) return fail(nullptr, FLUID_ERR_NCCL, "ncclGetUniqueId failed: %s", N.GetErrorString(rc));
    memcpy(out_uid, &id, sizeof id);
    return FLUID_OK;
}

int fluid_create_slab(const fluid_config* cfg, int rank, int world, const void* nccl_uid,
                      size_t uid_bytes, fluid_t** out) {
    if (world > 1 && (!nccl_uid || uid_bytes < sizeof(ncdl::ncclUniqueId)))
        return fail(nullptr, FLUID_ERR_INVALID, "nccl_uid must be the 128 bytes from fluid_nccl_unique_id()");
    return create_common(cfg, rank, world, nccl_uid, out);
}

// ---- peer-memory halo path -------------------------------------------------------------------------
struct P2PBlob {            // what fluid_p2p_export hands to the launcher (opaque to it), 256 bytes
    cudaIpcMemHandle_t mem;
    int32_t rank, roff, droff, reserved;
    uint64_t off_v[2], off_p[2], off_dye[2], off_div, off_flags, arena_bytes;
    char pad[256 - sizeof(cudaIpcMemHandle_t) - 16 - 9 * 8];
};
static_assert(sizeof(P2PBlob) == 256, "blob layout");

int fluid_p2p_export(fluid_t* h, void* blob, size_t blob_bytes) {
    if (!h || !blob || blob_bytes < sizeof(P2PBlob)) return fail(h, FLUID_ERR_INVALID, "blob must hold 256 bytes");
    if (!h->slab() || !h->arena) return fail(h, FLUID_ERR_INVALID, "fluid_p2p_export needs a slab handle");
    // halo_push_kernel moves rows as 16-byte words: every exchanged row (4*W pressure / divergence,
    // 8*W velocity, 16*Wd dye) must be a multiple of 16 bytes.  Otherwise refuse, so that the
    // launcher keeps ALL ranks on the byte-exact NCCL transport.
    if (h->cfg.sim_w % 4 != 0)
        return fail(h, FLUID_ERR_INVALID, "peer-memory halos need sim width %% 4 == 0 (got %d): staying on NCCL", h->cfg.sim_w);
    P2PBlob b{};
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaIpcGetMemHandle(&b.mem, h->arena));
    b.rank = h->rank; b.roff = h->roff; b.droff = h->droff;
    for (int k = 0; k < 2; ++k) { b.off_v[k] = h->off_v[k]; b.off_p[k] = h->off_p[k]; b.off_dye[k] = h->off_dye[k]; }
    b.off_div = h->off_div; b.off_flags = h->off_flags; b.arena_bytes = h->arena_bytes;
    memcpy(blob, &b, sizeof b);
    return FLUID_OK;
}

// blob_below / blob_above: the 256-byte exports of rank-1 / rank+1 (NULL at the domain ends).
// Collective in spirit: every rank of the slab group must connect before the next fluid_step.
int fluid_p2p_connect(fluid_t* h, const void* blob_below, const void* blob_above) {
    if (!h || !h->slab() || !h->arena) return fail(h, FLUID_ERR_INVALID, "fluid_p2p_connect needs a slab handle");
    const void* blobs[2] = {blob_below, blob_above};
    for (int side = 0; side < 2; ++side) {
        const bool need = (side == 0) ? h->rank > 0 : h->rank + 1 < h->world;
        if (!need) continue;
        if (!blobs[side]) return fail(h, FLUID_ERR_INVALID, "missing neighbour blob (side %d)", side);
        P2PBlob b; memcpy(&b, blobs[side], sizeof b);
        if (b.rank != h->rank + (side == 0 ? -1 : 1)) return fail(h, FLUID_ERR_INVALID, "blob of rank %d passed as side %d of rank %d", b.rank, side, h->rank);
        void* base = nullptr;
        CU(cudaIpcOpenMemHandle(&base, b.mem, cudaIpcMemLazyEnablePeerAccess));
        fluid::Peer& P = h->peer[side];
        P.present = true; P.base = (char*)base; P.roff = b.roff; P.droff = b.droff;
        for (int k = 0; k < 2; ++k) { P.off_v[k] = b.off_v[k]; P.off_p[k] = b.off_p[k]; P.off_dye[k] = b.off_dye[k]; }
        P.off_div = b.off_div; P.off_flags = b.off_flags;
    }
    h->p2p = true;
    return FLUID_OK;
}

// Back to the NCCL transport (used by launchers when ANY rank failed to map its neighbours, so
// that all ranks keep using the same one).
int fluid_p2p_disable(fluid_t* h) {
    if (!h) return FLUID_ERR_INVALID;
    if (h->stream) CU(cudaStreamSynchronize(h->stream));
    for (auto& p : h->peer) if (p.present && p.base) { cudaIpcCloseMemHandle(p.base); p.base = nullptr; p.present = false; }
    h->p2p = false; h->p_mirror_valid = false;
    return FLUID_OK;
}

void fluid_destroy(fluid_t* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    drop_graphs(h);
    if (h->p2p && getenv("FLUID_DEBUG_HALO_TIMING")) {
        unsigned long long d[5] = {};
        cudaMemcpy(d, h->arena + h->off_flags + 128, sizeof d, cudaMemcpyDeviceToHost);
        unsigned long long m[9] = {};
        cudaMemcpy(m, h->arena + h->off_flags + 512, sizeof m, cudaMemcpyDeviceToHost);
        if (m[6] || m[8])
            fprintf(stderr, "[mirror rank %d] streams that waited for mirror-ready: %llu, avg %.1f us; mirroring warps: %llu, waited %.1f us for done-reading, "
                            "copied for %.1f us; stream life (hand-off launches): %.1f us touching ghost rows (%llu), %.1f us others (%llu)\n",
                    h->rank, m[1], m[1] ? m[0] / 1e3 / m[1] : 0.0, m[4], m[4] ? m[2] / 1e3 / m[4] : 0.0, m[4] ? m[3] / 1e3 / m[4] : 0.0,
                    m[6] ? m[5] / 1e3 / m[6] : 0.0, m[6], m[8] ? m[7] / 1e3 / m[8] : 0.0, m[8]);
        if (d[3]) fprintf(stderr, "[halo rank %d] exchanges %llu: wait-free %.1f us, push (start->published) %.1f us, wait-ready %.1f us\n",
                          h->rank, d[3], d[0] / 1e3 / d[3], d[1] / 1e3 / d[3], d[2] / 1e3 / d[3]);
    }
    free_fields(h);
    cudaFree(h->halo_flag);
    cudaFree(h->dt_dev);
    cudaFree(h->scratch);
    cudaFree(h->frame);
    if (h->comm) { ncdl::api().CommDestroy(h->comm); h->comm = nullptr; }
    for (auto& e : h->mark) if (e) cudaEventDestroy(e);
    for (auto& e : h->tev) if (e) cudaEventDestroy(e);
    if (h->hp.up) { cudaStreamSynchronize(h->hp.up); cudaStreamDestroy(h->hp.up); }
    if (h->hp.down) { cudaStreamSynchronize(h->hp.down); cudaStreamDestroy(h->hp.down); }
    if (h->hp.ev_start) cudaEventDestroy(h->hp.ev_start);
    for (auto& e : h->hp.ev_up) if (e) cudaEventDestroy(e);
    for (auto& e : h->hp.ev_done) if (e) cudaEventDestroy(e);
    cudaFree(h->hp.s[0]); cudaFree(h->hp.s[1]);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->stream2) { cudaStreamSynchronize(h->stream2); cudaStreamDestroy(h->stream2); }
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int fluid_set_param(fluid_t* h, int key, float v) {
    if (!h) return FLUID_ERR_INVALID;
    switch (key) {
        case FLUID_DENSITY_DISSIPATION: h->cfg.density_dissipation = v; break;
        case FLUID_VELOCITY_DISSIPATION: h->cfg.velocity_dissipation = v; break;
        case FLUID_PRESSURE: h->cfg.pressure = v; break;
        case FLUID_PRESSURE_ITERATIONS: h->cfg.pressure_iterations = (int)(v + 0.5f); break;
        case FLUID_CURL: h->cfg.curl = v; break;
        case FLUID_SPLAT_RADIUS: h->cfg.splat_radius = v; h->splat_radius_d = (double)v; break;
        case FLUID_ASPECT: h->cfg.aspect = v; h->aspect_d = (double)v; break;
        case FLUID_JACOBI_BLOCK: h->cfg.jacobi_block = (int)(v + 0.5f); break;
        case FLUID_BACKGROUND: h->background = (int)(v + 0.5f); break;
        default: return fail(h, FLUID_ERR_INVALID, "unknown param key %d", key);
    }
    return FLUID_OK;
}

// The JS config values are doubles; two of them enter double arithmetic on the host before the
// single narrowing of gl.uniform1f (correctRadius S:1457-1462: SPLAT_RADIUS / 100 * aspectRatio),
// so a host mirror passes them at full precision.  Every other key narrows like fluid_set_param.
int fluid_set_param_f64(fluid_t* h, int key, double v) {
    if (!h) return FLUID_ERR_INVALID;
    int rc = fluid_set_param(h, key, (float)v);
    if (rc) return rc;
    if (key == FLUID_SPLAT_RADIUS) h->splat_radius_d = v;
    if (key == FLUID_ASPECT) h->aspect_d = v;
    return FLUID_OK;
}

int fluid_get_param(fluid_t* h, int key, float* v) {
    if (!h || !v) return FLUID_ERR_INVALID;
    switch (key) {
        case FLUID_DENSITY_DISSIPATION: *v = h->cfg.density_dissipation; break;
        case FLUID_VELOCITY_DISSIPATION: *v = h->cfg.velocity_dissipation; break;
        case FLUID_PRESSURE: *v = h->cfg.pressure; break;
        case FLUID_PRESSURE_ITERATIONS: *v = (float)h->cfg.pressure_iterations; break;
        case FLUID_CURL: *v = h->cfg.curl; break;
        case FLUID_SPLAT_RADIUS: *v = h->cfg.splat_radius; break;
        case FLUID_ASPECT: *v = h->cfg.aspect; break;
        case FLUID_JACOBI_BLOCK: *v = (float)h->cfg.jacobi_block; break;
        case FLUID_BACKGROUND: *v = (float)h->background; break;
        default: return fail(h, FLUID_ERR_INVALID, "unknown param key %d", key);
    }
    return FLUID_OK;
}

// ---- passes ---------------------------------------------------------------------------------------
// do_*: launch on an explicit row range (owned rows, or owned +- e for redundant ghost compute on a
// slab); the public fluid_pass_* wrappers are the single-GPU, one-blit-per-call test surface.

static int do_curl(fluid_t* h, Grid g) {
    if (h->half) {
        hs::curl_kernel<<<hs_grid(g.W, g.H), HS_BLOCK, 0, h->stream>>>((const hs::h2*)h->velocity.read, (hs::h1*)h->curl, g.W, g.H);
        return check_launch(h, "hs::curl_kernel");
    }
    dim3 b(64, 4);
    curl_kernel<<<grid2d(g.W, g.j_hi - g.j_lo, b), b, 0, h->stream>>>((const float2*)h->velocity.read, h->curl, g);
    return check_launch(h, "curl_kernel");
}
static int do_vorticity(fluid_t* h, Grid g) {
    if (h->half) {
        hs::vorticity_kernel<<<hs_grid(g.W, g.H), HS_BLOCK, 0, h->stream>>>((const hs::h2*)h->velocity.read, (const hs::h1*)h->curl,
                                                                            (hs::h2*)h->velocity.write, g.W, g.H, h->cfg.curl, h->dt_dev);
        int rc = check_launch(h, "hs::vorticity_kernel"); if (rc) return rc;
        swap_v(h);
        return FLUID_OK;
    }
    dim3 b(64, 4);
    vorticity_kernel<<<grid2d(g.W, g.j_hi - g.j_lo, b), b, 0, h->stream>>>(
        (const float2*)h->velocity.read, h->curl, (float2*)h->velocity.write, g, h->cfg.curl, h->dt_dev);
    int rc = check_launch(h, "vorticity_kernel"); if (rc) return rc;
    swap_v(h);                                   // S:1246
    return FLUID_OK;
}
static int do_divergence(fluid_t* h, Grid g) {
    if (h->half) {
        hs::divergence_kernel<<<hs_grid(g.W, g.H), HS_BLOCK, 0, h->stream>>>((const hs::h2*)h->velocity.read, (hs::h1*)h->divergence, g.W, g.H);
        return check_launch(h, "hs::divergence_kernel");
    }
    dim3 b(64, 4);
    { int rc = clear_tiny_map(h); if (rc) return rc; }
    divergence_kernel<<<grid2d(g.W, g.j_hi - g.j_lo, b), b, 0, h->stream>>>(
        (const float2*)h->velocity.read, h->divergence, g, h->tiny_map);
    return check_launch(h, "divergence_kernel");
}
// rows per warp stream of the row-streaming kernels: one full wave of resident warps (`warps_per_sm`
// from the occupancy calculator), at least `rmin` rows each so that the halo rows a stream re-reads
// stay a bounded fraction.  Grids too small to give every SM a warp use the tiled kernels instead.
static StreamArgs stream_args(const fluid_t* h, Grid g, int cols_per_window, int rmin, int warps_per_sm, int round_to) {
    StreamArgs a{};
    a.g = g;
    a.nxw = (g.W + cols_per_window - 1) / cols_per_window;
    const int rows = g.j_hi - g.j_lo;
    const int chunks = std::max(1, h->sm_count * warps_per_sm / a.nxw);
    int r = std::max((rows + chunks - 1) / chunks, rmin);
    r = (r + round_to - 1) / round_to * round_to;
    a.rows_per_chunk = std::min(r, std::max(rows, 1));
    return a;
}
static int stream_warps(const StreamArgs& a) {
    return a.nxw * ((a.g.j_hi - a.g.j_lo + a.rows_per_chunk - 1) / a.rows_per_chunk);
}
static bool streaming_ok(const fluid_t* h) {
    return h->cfg.sim_w % 4 == 0 && h->cfg.sim_w >= 8 && !(h->cfg.flags & FLUID_FLAG_TILED_PASSES);
}

static int do_curl(fluid_t* h, Grid g);
static int do_vorticity(fluid_t* h, Grid g);
static int do_divergence(fluid_t* h, Grid g);
static int do_cvd(fluid_t* h, Grid g) {
    if (h->half) {                                   // one launch per reference blit (each rounds to fp16)
        int rc = do_curl(h, g); if (rc) return rc;
        if ((rc = do_vorticity(h, g))) return rc;
        return do_divergence(h, g);
    }
    { int rc = clear_tiny_map(h); if (rc) return rc; }
    static int cvd_occ = 0;
    if (!cvd_occ) {
        int blocks = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, cvd_stream_kernel, 32 * CVD2_WARPS, CVD2_SMEM);
        cvd_occ = std::max(1, blocks) * CVD2_WARPS;
    }
    const StreamArgs a = stream_args(h, g, CVD2_VALID, 16, cvd_occ, 1);
    const int nwarps = stream_warps(a);
    if (streaming_ok(h) && nwarps >= h->sm_count) {
        cvd_stream_kernel<<<(nwarps + CVD2_WARPS - 1) / CVD2_WARPS, 32 * CVD2_WARPS, CVD2_SMEM, h->stream>>>(
            (const float2*)h->velocity.read, h->curl, (float2*)h->velocity.write, h->divergence, a, h->cfg.curl,
            h->dt_dev, h->tiny_map);
        int rc = check_launch(h, "cvd_stream_kernel"); if (rc) return rc;
        swap_v(h);
        return FLUID_OK;
    }
    dim3 b(64, 4);
    dim3 grid((g.W + CVD_TX - 1) / CVD_TX, (g.j_hi - g.j_lo + CVD_TY - 1) / CVD_TY);
    curl_vorticity_divergence_kernel<<<grid, b, 0, h->stream>>>(
        (const float2*)h->velocity.read, h->curl, (float2*)h->velocity.write, h->divergence, g,
        h->cfg.curl, h->dt_dev, h->tiny_map);
    int rc = check_launch(h, "curl_vorticity_divergence_kernel"); if (rc) return rc;
    swap_v(h);
    return FLUID_OK;
}
static int do_gradient(fluid_t* h, Grid g) {
    if (h->half) {
        hs::gradient_kernel<<<hs_grid(g.W, g.H), HS_BLOCK, 0, h->stream>>>((const hs::h1*)h->pressure.read, (const hs::h2*)h->velocity.read,
                                                                           (hs::h2*)h->velocity.write, g.W, g.H);
        int rc = check_launch(h, "hs::gradient_kernel"); if (rc) return rc;
        swap_v(h);
        return FLUID_OK;
    }
    const StreamArgs a = stream_args(h, g, 128, 8, 32, GS_U);
    const int nwarps = stream_warps(a);
    if (streaming_ok(h) && nwarps >= h->sm_count) {
        gradient_stream_kernel<<<(nwarps + GS_WARPS - 1) / GS_WARPS, 32 * GS_WARPS, 0, h->stream>>>(
            (const float*)h->pressure.read, (const float2*)h->velocity.read, (float2*)h->velocity.write, a);
        int rc = check_launch(h, "gradient_stream_kernel"); if (rc) return rc;
        swap_v(h);                                   // S:1273
        return FLUID_OK;
    }
    dim3 b(64, 4);
    gradient_subtract_kernel<<<grid2d(g.W, g.j_hi - g.j_lo, b), b, 0, h->stream>>>(
        (const float*)h->pressure.read, (const float2*)h->velocity.read, (float2*)h->velocity.write, g);
    int rc = check_launch(h, "gradient_subtract_kernel"); if (rc) return rc;
    swap_v(h);                                   // S:1273
    return FLUID_OK;
}
// valid source rows of a slab buffer: owned + ghost, clipped to the domain
static void valid_rows(int r0, int r1, int g, int H, int* lo, int* hi) {
    *lo = std::max(r0 - g, 0); *hi = std::min(r1 + g, H);
}
static int do_advect_velocity(fluid_t* h, Grid out) {
    if (h->half) {
        hs::advect_kernel<hs::h2, float2><<<hs_grid(out.W, out.H), HS_BLOCK, 0, h->stream>>>(
            (const hs::h2*)h->velocity.read, out.W, out.H, (const hs::h2*)h->velocity.read, (hs::h2*)h->velocity.write, out.W, out.H,
            h->dt_dev, h->cfg.velocity_dissipation, (float)(1.0 / (double)out.W), (float)(1.0 / (double)out.H),
            (float)(1.0 / (double)out.W), (float)(1.0 / (double)out.H));
        int rc = check_launch(h, "hs::advect_kernel"); if (rc) return rc;
        swap_v(h);
        return FLUID_OK;
    }
    dim3 b(64, 4);
    AdvectArgs a{};
    a.vel = sim_grid(h); a.src = out;
    valid_rows(h->row0, h->row1, h->G, h->cfg.sim_h, &a.vel_lo, &a.vel_hi);
    a.src_lo = a.vel_lo; a.src_hi = a.vel_hi;
    a.dtp = h->dt_dev; a.dissipation = h->cfg.velocity_dissipation; a.halo_violation = h->halo_flag;
    a.tsx = a.dsx = (float)(1.0 / (double)h->cfg.sim_w); a.tsy = a.dsy = (float)(1.0 / (double)h->cfg.sim_h);
    const bool p2 = is_pow2(h->cfg.sim_w) && is_pow2(h->cfg.sim_h);
    if (p2 && h->cfg.sim_w >= 128 && !(h->cfg.flags & FLUID_FLAG_TILED_PASSES)) {    // 4 cells per thread, 32 apart
        dim3 b4(32, 8), g4(out.W / 128, (out.j_hi - out.j_lo + 7) / 8);
        if (h->slab()) advect_velocity4_kernel<true><<<g4, b4, 0, h->stream>>>((const float2*)h->velocity.read, (float2*)h->velocity.write, a);
        else advect_velocity4_kernel<false><<<g4, b4, 0, h->stream>>>((const float2*)h->velocity.read, (float2*)h->velocity.write, a);
    } else if (p2) advect_velocity_kernel<true><<<grid2d(out.W, out.j_hi - out.j_lo, b), b, 0, h->stream>>>(
        (const float2*)h->velocity.read, (float2*)h->velocity.write, a);
    else advect_velocity_kernel<false><<<grid2d(out.W, out.j_hi - out.j_lo, b), b, 0, h->stream>>>(
        (const float2*)h->velocity.read, (float2*)h->velocity.write, a);
    int rc = check_launch(h, "advect_velocity_kernel"); if (rc) return rc;
    swap_v(h);                                   // S:1285
    return FLUID_OK;
}
static int do_advect_dye(fluid_t* h) {
    if (h->half) {
        hs::advect_kernel<hs::h4, float4><<<hs_grid(h->cfg.dye_w, h->cfg.dye_h), HS_BLOCK, 0, h->stream>>>(
            (const hs::h2*)h->velocity.read, h->cfg.sim_w, h->cfg.sim_h, (const hs::h4*)h->dye.read, (hs::h4*)h->dye.write,
            h->cfg.dye_w, h->cfg.dye_h, h->dt_dev, h->cfg.density_dissipation, (float)(1.0 / (double)h->cfg.sim_w),
            (float)(1.0 / (double)h->cfg.sim_h), (float)(1.0 / (double)h->cfg.dye_w), (float)(1.0 / (double)h->cfg.dye_h));
        int rc = check_launch(h, "hs::advect_kernel"); if (rc) return rc;
        swap_dye(h);
        return FLUID_OK;
    }
    dim3 b(64, 4);
    AdvectArgs a{};
    a.vel = sim_grid(h); a.src = dye_grid(h);
    // after the velocity advection the slab holds valid velocity on owned rows +- 3
    valid_rows(h->row0, h->row1, h->slab() ? 3 : 0, h->cfg.sim_h, &a.vel_lo, &a.vel_hi);
    valid_rows(h->drow0, h->drow1, h->Gd, h->cfg.dye_h, &a.src_lo, &a.src_hi);
    a.dtp = h->dt_dev; a.dissipation = h->cfg.density_dissipation; a.halo_violation = h->halo_flag;
    a.tsx = (float)(1.0 / (double)h->cfg.sim_w); a.tsy = (float)(1.0 / (double)h->cfg.sim_h);
    a.dsx = (float)(1.0 / (double)h->cfg.dye_w); a.dsy = (float)(1.0 / (double)h->cfg.dye_h);
    const bool p2 = is_pow2(h->cfg.sim_w) && is_pow2(h->cfg.sim_h) && is_pow2(h->cfg.dye_w) && is_pow2(h->cfg.dye_h);
    const bool same = h->cfg.sim_w == h->cfg.dye_w && h->cfg.sim_h == h->cfg.dye_h;
    const dim3 gr = grid2d(a.src.W, a.src.j_hi - a.src.j_lo, b);
    const float2* V = (const float2*)h->velocity.read; const float4* Dr = (const float4*)h->dye.read; float4* Dw = (float4*)h->dye.write;
    if (p2 && a.src.W >= 128 && !(h->cfg.flags & FLUID_FLAG_TILED_PASSES)) {         // 4 cells per thread, 32 apart
        dim3 b4(32, 8), g4(a.src.W / 128, (a.src.j_hi - a.src.j_lo + 7) / 8);
        if (same && h->slab()) advect_dye4_kernel<true, true><<<g4, b4, 0, h->stream>>>(V, Dr, Dw, a);
        else if (same) advect_dye4_kernel<true, false><<<g4, b4, 0, h->stream>>>(V, Dr, Dw, a);
        else if (h->slab()) advect_dye4_kernel<false, true><<<g4, b4, 0, h->stream>>>(V, Dr, Dw, a);
        else advect_dye4_kernel<false, false><<<g4, b4, 0, h->stream>>>(V, Dr, Dw, a);
    } else if (p2 && same) advect_dye_kernel<true, true><<<gr, b, 0, h->stream>>>(V, Dr, Dw, a);
    else if (p2) advect_dye_kernel<true, false><<<gr, b, 0, h->stream>>>(V, Dr, Dw, a);
    else advect_dye_kernel<false, false><<<gr, b, 0, h->stream>>>(V, Dr, Dw, a);
    int rc = check_launch(h, "advect_dye_kernel"); if (rc) return rc;
    swap_dye(h);                                        // S:1293
    return FLUID_OK;
}

int fluid_pass_curl(fluid_t* h) {
    if (!h) return FLUID_ERR_INVALID;
    if (h->slab()) return not_on_slab(h, "fluid_pass_curl");
    return do_curl(h, sim_grid(h));
}
int fluid_pass_vorticity(fluid_t* h, float dt) {
    if (!h) return FLUID_ERR_INVALID;
    if (h->slab()) return not_on_slab(h, "fluid_pass_vorticity");
    int rc = set_dt(h, dt); if (rc) return rc;
    return do_vorticity(h, sim_grid(h));
}
int fluid_pass_divergence(fluid_t* h) {
    if (!h) return FLUID_ERR_INVALID;
    if (h->slab()) return not_on_slab(h, "fluid_pass_divergence");
    return do_divergence(h, sim_grid(h));
}
int fluid_pass_curl_vorticity_divergence(fluid_t* h, float dt) {
    if (!h) return FLUID_ERR_INVALID;
    if (h->slab()) return not_on_slab(h, "fluid_pass_curl_vorticity_divergence");
    int rc = set_dt(h, dt); if (rc) return rc;
    return do_cvd(h, sim_grid(h));
}
int fluid_pass_clear_pressure(fluid_t* h) {
    if (!h) return FLUID_ERR_INVALID;
    return run_jacobi(h, 0, true, nullptr);
}
int fluid_pass_jacobi(fluid_t* h, int iters) {
    if (!h) return FLUID_ERR_INVALID;
    if (iters < 0) return fail(h, FLUID_ERR_INVALID, "iters < 0");
    return run_jacobi(h, iters, false, nullptr);
}
int fluid_pass_pressure_solve(fluid_t* h) {
    if (!h) return FLUID_ERR_INVALID;
    return run_jacobi(h, h->cfg.pressure_iterations, true, nullptr);
}
int fluid_pass_gradient_subtract(fluid_t* h) {
    if (!h) return FLUID_ERR_INVALID;
    if (h->slab()) return not_on_slab(h, "fluid_pass_gradient_subtract");
    return do_gradient(h, sim_grid(h));
}
int fluid_pass_advect_velocity(fluid_t* h, float dt) {
    if (!h) return FLUID_ERR_INVALID;
    if (h->slab()) return not_on_slab(h, "fluid_pass_advect_velocity");
    int rc = set_dt(h, dt); if (rc) return rc;
    return do_advect_velocity(h, sim_grid(h));
}
int fluid_pass_advect_dye(fluid_t* h, float dt) {
    if (!h) return FLUID_ERR_INVALID;
    if (h->slab()) return not_on_slab(h, "fluid_pass_advect_dye");
    int rc = set_dt(h, dt); if (rc) return rc;
    return do_advect_dye(h);
}

// step(dt), S:1231-1294.
// On a slab the only messages are the Jacobi halos (inside run_jacobi) and the two advection
// halos below; curl / vorticity / divergence / gradientSubtract read ghost rows that the previous
// step's advection (velocity on owned rows +- 3) and the last Jacobi launch (pressure on owned
// rows +- 1) already computed redundantly.
static int step_enqueue(fluid_t* h, bool timed) {
    const uint64_t l0 = h->launches;
    const int W = h->cfg.sim_w;
    int rc;
    int jl = 0;
    if (timed) cudaEventRecord(h->tev[0], h->stream);
    if (h->slab() && !h->v_ghost_valid) {   // after fluid_write(velocity): rebuild the +-3 ghost rows
        if ((rc = exchange_rows(h, HB_VELOCITY, h->velocity.read, (size_t)W * sizeof(float2), h->roff, h->row0, h->row1, 3))) return rc;
        h->v_ghost_valid = true;
    }
    if (h->cfg.flags & FLUID_FLAG_UNFUSED) {
        if ((rc = do_curl(h, sim_grid_ext(h, h->slab() ? 2 : 0)))) return rc;
        if ((rc = do_vorticity(h, sim_grid_ext(h, h->slab() ? 1 : 0)))) return rc;
        if ((rc = do_divergence(h, sim_grid(h)))) return rc;
    } else {
        if ((rc = do_cvd(h, sim_grid(h)))) return rc;
    }
    if (timed) cudaEventRecord(h->tev[1], h->stream);
    if ((rc = run_jacobi(h, h->cfg.pressure_iterations, true, &jl))) return rc;
    if (timed) cudaEventRecord(h->tev[2], h->stream);
    if ((rc = do_gradient(h, sim_grid(h)))) return rc;
    if (timed) cudaEventRecord(h->tev[3], h->stream);
    if (h->slab()) {   // advection halo #1: G rows of the projected velocity
        if ((rc = exchange_rows(h, HB_VELOCITY, h->velocity.read, (size_t)W * sizeof(float2), h->roff, h->row0, h->row1, h->G))) return rc;
    }
    if ((rc = do_advect_velocity(h, sim_grid_ext(h, h->slab() ? 3 : 0)))) return rc;
    if (timed) cudaEventRecord(h->tev[4], h->stream);
    if (h->slab()) {   // advection halo #2: Gd rows of dye
        if ((rc = exchange_rows(h, HB_DYE, h->dye.read, (size_t)h->cfg.dye_w * sizeof(float4), h->droff, h->drow0, h->drow1, h->Gd))) return rc;
    }
    if ((rc = do_advect_dye(h))) return rc;
    if (timed) cudaEventRecord(h->tev[5], h->stream);
    h->timing.jacobi_launches = jl;
    h->timing.total_launches = (int)(h->launches - l0);
    h->have_timing = timed;
    return FLUID_OK;
}

// The reference pays one draw call per pass (7 + PRESSURE_ITERATIONS per step) and is bound by
// that at its default 128^2 grid.  Here a step is 4 + ceil(iters/10) kernels, and on a single GPU
// they are replayed as ONE instantiated CUDA graph.  A graph bakes in kernel arguments, so the
// cache key holds everything they depend on: the config scalars, the grid sizes and which half of
// each ping-pong pair is currently `.read`.  dt is NOT part of the key: kernels read it from
// device memory (set_dt), so the reference's frame loop — calcDeltaTime() yields a different dt
// on every frame (S:1188-1194) — replays the same two graphs (one per ping-pong parity).
int fluid_step(fluid_t* h, float dt) {
    if (!h) return FLUID_ERR_INVALID;
    const bool no_graph = (h->cfg.flags & FLUID_FLAG_NO_GRAPH) != 0;
    { int rc = set_dt(h, dt); if (rc) return rc; }
    if (no_graph || h->slab()) return step_enqueue(h, no_graph);
    char key[256];
    const fluid_config& c = h->cfg;
    snprintf(key, sizeof key, "%a|%a|%a|%a|%d|%d|%u|%d%d%d|%dx%d|%dx%d",
             c.curl, c.pressure, c.velocity_dissipation, c.density_dissipation, c.pressure_iterations, c.jacobi_block,
             c.flags, h->par_v, h->par_p, h->par_dye, c.sim_w, c.sim_h, c.dye_w, c.dye_h);
    auto it = h->graphs.find(key);
    if (it == h->graphs.end()) {
        if (h->graphs.size() > 64) drop_graphs(h);          // config sliders dragged for a long time: stay bounded
        const int pv = h->par_v, pp = h->par_p, pd = h->par_dye;
        const uint64_t l0 = h->launches, j0 = h->jacobi_kernel_launches;
        cudaGraph_t g = nullptr;
        CU(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        h->capturing = true;
        int rc = step_enqueue(h, false);
        h->capturing = false;
        cudaError_t e = cudaStreamEndCapture(h->stream, &g);
        if (rc) { if (g) cudaGraphDestroy(g); return rc; }
        if (e != cudaSuccess) return fail(h, FLUID_ERR_CUDA, "stream capture of step() failed: %s", cudaGetErrorString(e));
        fluid::StepGraph sg;
        e = cudaGraphInstantiate(&sg.exec, g, 0);
        cudaGraphDestroy(g);
        if (e != cudaSuccess) return fail(h, FLUID_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(e));
        sg.flip_v = pv ^ h->par_v; sg.flip_p = pp ^ h->par_p; sg.flip_dye = pd ^ h->par_dye;
        sg.kernels = (int)(h->launches - l0); sg.jacobi_launches = (int)(h->jacobi_kernel_launches - j0);
        h->launches = l0; h->jacobi_kernel_launches = j0;    // captured, not yet executed
        ++h->graph_captures;
        it = h->graphs.emplace(key, sg).first;
        // the capture already performed the host-side swaps of this step
    } else {
        const fluid::StepGraph& sg = it->second;
        if (sg.flip_v) swap_v(h);
        if (sg.flip_p) swap_p(h);
        if (sg.flip_dye) swap_dye(h);
    }
    CU(cudaGraphLaunch(it->second.exec, h->stream));
    h->launches += it->second.kernels;
    h->jacobi_kernel_launches += it->second.jacobi_launches;
    h->timing.jacobi_launches = it->second.jacobi_launches;
    h->timing.total_launches = it->second.kernels;
    h->have_timing = false;
    ++h->graph_launches;
    return FLUID_OK;
}

// splat(x,y,dx,dy,color), S:1441-1455
int fluid_splat(fluid_t* h, float x, float y, float dx, float dy, float r, float g, float b) {
    if (!h) return FLUID_ERR_INVALID;
    // correctRadius(config.SPLAT_RADIUS / 100.0): JS double arithmetic, narrowed by gl.uniform1f
    double rad = h->splat_radius_d / 100.0;
    if (h->aspect_d > 1.0) rad *= h->aspect_d;
    const float radius = (float)rad;
    if (h->half) {
        const int W = h->cfg.sim_w, H = h->cfg.sim_h, Wd = h->cfg.dye_w, Hd = h->cfg.dye_h;
        hs::splat_velocity_kernel<<<hs_grid(W, H), HS_BLOCK, 0, h->stream>>>((const hs::h2*)h->velocity.read, (hs::h2*)h->velocity.write, W, H,
                                                                             h->cfg.aspect, x, y, dx, dy, radius);
        int rc = check_launch(h, "hs::splat_velocity_kernel"); if (rc) return rc;
        swap_v(h);
        hs::splat_dye_kernel<<<hs_grid(Wd, Hd), HS_BLOCK, 0, h->stream>>>((const hs::h4*)h->dye.read, (hs::h4*)h->dye.write, Wd, Hd,
                                                                          h->cfg.aspect, x, y, r, g, b, radius);
        rc = check_launch(h, "hs::splat_dye_kernel"); if (rc) return rc;
        swap_dye(h);
        return FLUID_OK;
    }
    dim3 bl(64, 4);
    // a splat is point-wise, so the +-3 velocity ghost rows are simply splatted as well
    Grid gs = sim_grid_ext(h, h->slab() ? 3 : 0), gd = dye_grid(h);
    SplatArgs sa{};
    sa.aspect = h->cfg.aspect; sa.px = x; sa.py = y; sa.radius = radius;
    sa.g = gs; sa.pow2 = is_pow2(gs.W) && is_pow2(gs.H);
    sa.tsx = (float)(1.0 / (double)gs.W); sa.tsy = (float)(1.0 / (double)gs.H);
    splat_velocity_kernel<<<grid2d(gs.W, gs.j_hi - gs.j_lo, bl), bl, 0, h->stream>>>(
        (const float2*)h->velocity.read, (float2*)h->velocity.write, sa, dx, dy);
    int rc = check_launch(h, "splat_velocity_kernel"); if (rc) return rc;
    swap_v(h);                                   // S:1449
    sa.g = gd; sa.pow2 = is_pow2(gd.W) && is_pow2(gd.H);
    sa.tsx = (float)(1.0 / (double)gd.W); sa.tsy = (float)(1.0 / (double)gd.H);
    splat_dye_kernel<<<grid2d(gd.W, gd.j_hi - gd.j_lo, bl), bl, 0, h->stream>>>(
        (const float4*)h->dye.read, (float4*)h->dye.write, sa, r, g, b);
    rc = check_launch(h, "splat_dye_kernel"); if (rc) return rc;
    swap_dye(h);                                        // S:1454
    return FLUID_OK;
}

// initFramebuffers() on a live simulation: S:982-1010 + resizeDoubleFBO S:1116-1126
int fluid_resize(fluid_t* h, int sim_w, int sim_h, int dye_w, int dye_h) {
    if (!h) return FLUID_ERR_INVALID;
    if (sim_w < 1 || sim_h < 1 || dye_w < 1 || dye_h < 1) return fail(h, FLUID_ERR_INVALID, "bad size");
    if (h->slab()) {
        // Collective among the ranks of the group (all call it with the same sizes).  The new rows a rank
        // owns sample old rows it owns +- ceil(old/new) + 2: refresh that many ghost rows of the old
        // velocity and dye, resample into a NEW arena, drop the old one.  Peer mappings die with the old
        // arena: the group is back on NCCL until the launcher exports / connects again
        // (distributed.connect_peers).
        const int ow = h->cfg.sim_w, oh = h->cfg.sim_h, odw = h->cfg.dye_w, odh = h->cfg.dye_h;
        const int need_v = (oh + sim_h - 1) / sim_h + 2, need_d = (odh + dye_h - 1) / dye_h + 2;
        if (need_v > h->G || need_d > h->Gd)
            return fail(h, FLUID_ERR_HALO, "resize by this factor needs %d / %d ghost rows, the slab keeps %d / %d", need_v, need_d, h->G, h->Gd);
        int rc;
        if ((rc = exchange_rows(h, HB_VELOCITY, h->velocity.read, (size_t)ow * sizeof(float2), h->roff, h->row0, h->row1, need_v))) return rc;
        if ((rc = exchange_rows(h, HB_DYE, h->dye.read, (size_t)odw * sizeof(float4), h->droff, h->drow0, h->drow1, need_d))) return rc;
        CU(cudaStreamSynchronize(h->stream));
        // keep the old arena alive while the new one is filled
        char* old_arena = h->arena; const float2* old_v = (const float2*)h->velocity.read; const float4* old_d = (const float4*)h->dye.read;
        const int old_roff = h->roff, old_droff = h->droff;
        for (auto& p : h->peer) if (p.present && p.base) { cudaIpcCloseMemHandle(p.base); p.base = nullptr; p.present = false; }
        h->p2p = false; h->p_mirror_valid = false;
        h->arena = nullptr;
        h->cfg.sim_w = sim_w; h->cfg.sim_h = sim_h; h->cfg.dye_w = dye_w; h->cfg.dye_h = dye_h;
        if (!slab_geometry(h, sim_h, dye_h, h->cfg.pressure_iterations)) {
            cudaFree(old_arena);
            return fail(h, FLUID_ERR_INVALID, "new slabs of %d rows are too short for a 14-row halo", sim_h / h->world);
        }
        cudaFree(h->tiny_map); h->tiny_map = nullptr;
        if ((rc = alloc_fields(h))) { cudaFree(old_arena); return rc; }
        dim3 b(64, 4);
        resample_slab_kernel<<<grid2d(sim_w, h->row1 - h->row0, b), b, 0, h->stream>>>(old_v, ow, oh, old_roff, (float2*)h->velocity.read, sim_w, sim_h,
                                                                                         h->roff, h->row0, h->row1);
        resample_slab_kernel<<<grid2d(dye_w, h->drow1 - h->drow0, b), b, 0, h->stream>>>(old_d, odw, odh, old_droff, (float4*)h->dye.read, dye_w, dye_h,
                                                                                           h->droff, h->drow0, h->drow1);
        rc = check_launch(h, "resample_slab_kernel", 2);
        CU(cudaStreamSynchronize(h->stream));
        cudaFree(old_arena);
        h->v_ghost_valid = false;                            // the +-3 velocity ghost rows are rebuilt by the next step
        return rc;
    }
    CU(cudaStreamSynchronize(h->stream));
    drop_graphs(h);                                          // graphs hold the old buffers' addresses
    if (h->half) {
        // fp16 storage: widen the old texture, draw the copy through the LINEAR sampler in fp32, round the
        // new texture to fp16 (what the reference's blit into an RGBA16F / RG16F target does)
        auto redo = [&](Pair& f, int ow_, int oh_, int nw_, int nh_, int ch, bool alpha) -> int {
            const size_t on = (size_t)ow_ * oh_ * ch, nn = (size_t)nw_ * nh_ * ch;
            float *wide = nullptr, *res = nullptr; void *nr = nullptr, *nwp = nullptr;
            CU(cudaMalloc((void**)&wide, on * 4)); CU(cudaMalloc((void**)&res, nn * 4));
            CU(cudaMalloc(&nr, nn * 2)); CU(cudaMalloc(&nwp, nn * 2));
            hs::widen_kernel<<<(unsigned)((on + 255) / 256), 256, 0, h->stream>>>((const hs::h1*)f.read, wide, on);
            dim3 b(64, 4);
            if (ch == 4) resample_kernel<float4><<<grid2d(nw_, nh_, b), b, 0, h->stream>>>((const float4*)wide, ow_, oh_, (float4*)res, nw_, nh_);
            else resample_kernel<float2><<<grid2d(nw_, nh_, b), b, 0, h->stream>>>((const float2*)wide, ow_, oh_, (float2*)res, nw_, nh_);
            hs::narrow_kernel<<<(unsigned)((nn + 255) / 256), 256, 0, h->stream>>>(res, (hs::h1*)nr, nn);
            if (alpha) hs::fill_alpha_kernel<<<(unsigned)((nn / 4 + 255) / 256), 256, 0, h->stream>>>((hs::h4*)nwp, nn / 4);
            else CU(cudaMemsetAsync(nwp, 0, nn * 2, h->stream));
            int rc = check_launch(h, "half resize", 3); if (rc) return rc;
            CU(cudaStreamSynchronize(h->stream));
            cudaFree(wide); cudaFree(res); cudaFree(f.read); cudaFree(f.write);
            f.read = nr; f.write = nwp;
            return FLUID_OK;
        };
        const int ow = h->cfg.sim_w, oh = h->cfg.sim_h, odw = h->cfg.dye_w, odh = h->cfg.dye_h;
        int rc;
        if ((dye_w != odw || dye_h != odh) && (rc = redo(h->dye, odw, odh, dye_w, dye_h, 4, true))) return rc;
        if ((sim_w != ow || sim_h != oh) && (rc = redo(h->velocity, ow, oh, sim_w, sim_h, 2, false))) return rc;
        const size_t n = (size_t)sim_w * sim_h;
        cudaFree(h->pressure.read); cudaFree(h->pressure.write); cudaFree(h->divergence); cudaFree(h->curl);
        h->pressure = Pair{}; h->divergence = h->curl = nullptr;
        CU(cudaMalloc(&h->pressure.read, n * 2)); CU(cudaMalloc(&h->pressure.write, n * 2));
        CU(cudaMalloc((void**)&h->divergence, n * 2)); CU(cudaMalloc((void**)&h->curl, n * 2));
        CU(cudaMemsetAsync(h->pressure.read, 0, n * 2, h->stream)); CU(cudaMemsetAsync(h->pressure.write, 0, n * 2, h->stream));
        CU(cudaMemsetAsync(h->divergence, 0, n * 2, h->stream)); CU(cudaMemsetAsync(h->curl, 0, n * 2, h->stream));
        h->cfg.sim_w = sim_w; h->cfg.sim_h = sim_h; h->cfg.dye_w = dye_w; h->cfg.dye_h = dye_h;
        h->row0 = 0; h->row1 = sim_h; h->drow0 = 0; h->drow1 = dye_h;
        return alloc_tiny_map(h);
    }
    const int ow = h->cfg.sim_w, oh = h->cfg.sim_h, odw = h->cfg.dye_w, odh = h->cfg.dye_h;
    dim3 b(64, 4);
    const size_t n = (size_t)sim_w * sim_h, nd = (size_t)dye_w * dye_h;
    if (dye_w != odw || dye_h != odh) {
        float4 *nr = nullptr, *nw = nullptr;
        CU(cudaMalloc((void**)&nr, nd * sizeof(float4)));
        CU(cudaMalloc((void**)&nw, nd * sizeof(float4)));
        resample_kernel<float4><<<grid2d(dye_w, dye_h, b), b, 0, h->stream>>>(
            (const float4*)h->dye.read, odw, odh, nr, dye_w, dye_h);
        fill_alpha_kernel<<<(unsigned)((nd + 255) / 256), 256, 0, h->stream>>>(nw, nd);
        int rc = check_launch(h, "resample_kernel", 2); if (rc) return rc;
        CU(cudaStreamSynchronize(h->stream));
        cudaFree(h->dye.read); cudaFree(h->dye.write);
        h->dye.read = nr; h->dye.write = nw;
    }
    if (sim_w != ow || sim_h != oh) {
        float2 *nr = nullptr, *nw = nullptr;
        CU(cudaMalloc((void**)&nr, n * sizeof(float2)));
        CU(cudaMalloc((void**)&nw, n * sizeof(float2)));
        resample_kernel<float2><<<grid2d(sim_w, sim_h, b), b, 0, h->stream>>>(
            (const float2*)h->velocity.read, ow, oh, nr, sim_w, sim_h);
        int rc = check_launch(h, "resample_kernel"); if (rc) return rc;
        CU(cudaMemsetAsync(nw, 0, n * sizeof(float2), h->stream));
        CU(cudaStreamSynchronize(h->stream));
        cudaFree(h->velocity.read); cudaFree(h->velocity.write);
        h->velocity.read = nr; h->velocity.write = nw;
    }
    // divergence, curl, pressure are always re-created (createFBO / createDoubleFBO, S:1004-1006)
    cudaFree(h->pressure.read); cudaFree(h->pressure.write); cudaFree(h->divergence); cudaFree(h->curl);
    h->pressure = Pair{}; h->divergence = h->curl = nullptr;
    CU(cudaMalloc(&h->pressure.read, n * sizeof(float)));
    CU(cudaMalloc(&h->pressure.write, n * sizeof(float)));
    CU(cudaMalloc((void**)&h->divergence, n * sizeof(float)));
    CU(cudaMalloc((void**)&h->curl, n * sizeof(float)));
    CU(cudaMemsetAsync(h->pressure.read, 0, n * sizeof(float), h->stream));
    CU(cudaMemsetAsync(h->pressure.write, 0, n * sizeof(float), h->stream));
    CU(cudaMemsetAsync(h->divergence, 0, n * sizeof(float), h->stream));
    CU(cudaMemsetAsync(h->curl, 0, n * sizeof(float), h->stream));
    h->cfg.sim_w = sim_w; h->cfg.sim_h = sim_h; h->cfg.dye_w = dye_w; h->cfg.dye_h = dye_h;
    h->row0 = 0; h->row1 = sim_h; h->drow0 = 0; h->drow1 = dye_h; h->roff = 0; h->droff = 0;
    { int rc = alloc_tiny_map(h); if (rc) return rc; }
    build_tmaps(h);
    return FLUID_OK;
}

// ---- data in / out --------------------------------------------------------------------------------

size_t fluid_field_elems(fluid_t* h, int field) {
    void* p; int w, rows, ch;
    if (!h || field_info(h, field, &p, &w, &rows, &ch)) return 0;
    return (size_t)w * rows * ch;
}

int fluid_field_dims(fluid_t* h, int field, int* w, int* rows, int* ch, int* row0) {
    void* p; int ww, rr, cc;
    if (!h || field_info(h, field, &p, &ww, &rr, &cc)) return FLUID_ERR_INVALID;
    if (w) *w = ww; if (rows) *rows = rr; if (ch) *ch = cc;
    if (row0) *row0 = (field == FLUID_FIELD_DYE) ? h->drow0 : h->row0;
    return FLUID_OK;
}

int fluid_read(fluid_t* h, int field, float* host, size_t n_floats) {
    void* p; int w, rows, ch;
    if (!h || !host || field_info(h, field, &p, &w, &rows, &ch)) return fail(h, FLUID_ERR_INVALID, "bad field %d", field);
    const size_t n = (size_t)w * rows * ch;
    if (n_floats != n) return fail(h, FLUID_ERR_INVALID, "field %d has %zu floats, caller passed %zu", field, n, n_floats);
    if (h->half) {                                   // the ABI speaks fp32: widen on the device, then copy
        int rc = need_scratch(h, n); if (rc) return rc;
        hs::widen_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((const hs::h1*)p, h->scratch, n);
        if ((rc = check_launch(h, "hs::widen_kernel"))) return rc;
        p = h->scratch;
    }
    CU(cudaMemcpyAsync(host, p, n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return check_halo(h);
}

int fluid_write(fluid_t* h, int field, const float* host, size_t n_floats) {
    void* p; int w, rows, ch;
    if (!h || !host || field_info(h, field, &p, &w, &rows, &ch)) return fail(h, FLUID_ERR_INVALID, "bad field %d", field);
    const size_t n = (size_t)w * rows * ch;
    if (n_floats != n) return fail(h, FLUID_ERR_INVALID, "field %d has %zu floats, caller passed %zu", field, n, n_floats);
    if (h->half) {                                   // narrow with round-to-nearest-even, like a texture upload would
        int rc = need_scratch(h, n); if (rc) return rc;
        CU(cudaMemcpyAsync(h->scratch, host, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
        hs::narrow_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->scratch, (hs::h1*)p, n);
        if ((rc = check_launch(h, "hs::narrow_kernel"))) return rc;
        CU(cudaStreamSynchronize(h->stream));
        return FLUID_OK;
    }
    CU(cudaMemcpyAsync(p, host, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (field == FLUID_FIELD_VELOCITY) h->v_ghost_valid = false;   // ghosts rebuilt by the next step
    if (field == FLUID_FIELD_PRESSURE) h->p_mirror_valid = false;  // the neighbours' ghost copies are stale now
    if (field == FLUID_FIELD_DIVERGENCE) {                          // host-provided divergence: rebuild the map
        int rc = clear_tiny_map(h); if (rc) return rc;
        if ((rc = scan_tiny(h, h->row0, h->row1))) return rc;
    }
    return FLUID_OK;
}

// fluid_pressure_solve_host on one GPU is PCIe-bound (4096^2: 128 MiB up, 64 MiB down, 3.7 of its 3.96 ms), so
// the solve is hidden behind the copies: the grid is cut into row bands, band b is solved as soon as its rows
// (+ `iters` rows beyond it) have arrived and is copied back while the later bands still upload — the slab
// decomposition of section 7 applied in time instead of across GPUs, the host standing in for the
// neighbours.  Communication-avoiding schedule as on a slab: launch k of a band produces its rows +- (sweeps
// still to come), out of band-private ping-pong rows; the first launch reads the uploaded field, the last one
// writes the band's rows of the result field.  Bit-identical to the one-piece solve (same kernel, same
// per-cell arithmetic; which rows a launch covers does not enter the values).
int solve_host_banded(fluid_t* h, const float* div_host, float* p_host, int iters, int nb) {
    const int W = h->cfg.sim_w, H = h->cfg.sim_h;
    fluid::HostPipe& hp = h->hp;
    if (!hp.up) {
        CU(cudaStreamCreateWithFlags(&hp.up, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&hp.down, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&hp.ev_start, cudaEventDisableTiming));
        for (auto& e : hp.ev_up) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : hp.ev_done) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    int kb = h->cfg.jacobi_block > 0 ? h->cfg.jacobi_block : 10;
    kb = std::min(kb, KMAX);
    const int nlaunch = (iters + kb - 1) / kb;
    const int base = iters / nlaunch, extra = iters % nlaunch;
    const int band = (H + nb - 1) / nb, halo = iters;
    const size_t need = (size_t)(band + 2 * halo) * W;
    if (hp.s_floats < need) {
        cudaFree(hp.s[0]); cudaFree(hp.s[1]); hp.s[0] = hp.s[1] = nullptr; hp.s_floats = 0;
        CU(cudaMalloc((void**)&hp.s[0], need * sizeof(float)));
        CU(cudaMalloc((void**)&hp.s[1], need * sizeof(float)));
        hp.s_floats = need;
    }
    float* const p_in = (float*)h->pressure.read;
    float* const result = (float*)h->pressure.write;
    h->p_mirror_valid = false;
    int rc = clear_tiny_map(h); if (rc) return rc;
    CU(cudaEventRecord(hp.ev_start, h->stream));          // the copies overwrite fields earlier work on the stream may still read
    CU(cudaStreamWaitEvent(hp.up, hp.ev_start, 0));
    for (int b = 0; b < nb; ++b) {
        const int b_lo = std::min(b * band, H), b_hi = std::min(b_lo + band, H);
        if (b_hi <= b_lo) break;
        // upload chunk b = what band b needs beyond what the earlier chunks brought: rows up to b_hi + halo
        const int up_lo = b == 0 ? 0 : std::min(b_lo + halo, H), up_hi = (b_hi == H) ? H : std::min(b_hi + halo, H);
        if (up_hi > up_lo) {
            const size_t o = (size_t)up_lo * W, n = (size_t)(up_hi - up_lo) * W * sizeof(float);
            CU(cudaMemcpyAsync(h->divergence + o, div_host + o, n, cudaMemcpyHostToDevice, hp.up));
            CU(cudaMemcpyAsync(p_in + o, p_host + o, n, cudaMemcpyHostToDevice, hp.up));
        }
        CU(cudaEventRecord(hp.ev_up[b], hp.up));
        CU(cudaStreamWaitEvent(h->stream, hp.ev_up[b], 0));
        if ((rc = scan_tiny(h, up_lo, up_hi))) return rc;
        const int loc = b_lo - halo;                      // global row of local row 0 of the band-private rows (may be < 0)
        int remaining = iters;
        for (int k = 0; k < nlaunch; ++k) {
            const int K = base + (k < extra ? 1 : 0);
            const bool last = (k == nlaunch - 1);
            remaining -= K;
            JacobiArgs a{};
            a.W = W; a.H = H; a.scale = h->cfg.pressure; a.err = h->halo_flag; a.tiny_map = h->tiny_map;
            a.out_lo = std::max(b_lo - remaining, 0); a.out_hi = std::min(b_hi + remaining, H);
            // the kernel addresses all three fields as "local row 0 + (row - row_off)": a whole-grid field G is
            // passed as G + loc*W (only rows inside the grid are ever dereferenced)
            a.row_off = loc;
            a.div = h->divergence + (ptrdiff_t)loc * W;
            a.pin = (k == 0) ? p_in + (ptrdiff_t)loc * W : hp.s[(k - 1) & 1];
            a.pout = last ? result + (ptrdiff_t)loc * W : hp.s[k & 1];
            h->pdl_chain = (k > 0);
            rc = launch_tb_dyn(h, K, a, k == 0);
            h->pdl_chain = false;
            if (rc) return rc;
        }
        CU(cudaEventRecord(hp.ev_done[b], h->stream));
        CU(cudaStreamWaitEvent(hp.down, hp.ev_done[b], 0));
        const size_t o = (size_t)b_lo * W;
        CU(cudaMemcpyAsync(p_host + o, result + o, (size_t)(b_hi - b_lo) * W * sizeof(float), cudaMemcpyDeviceToHost, hp.down));
    }
    swap_p(h);                                            // pressure.read = the result, like S:1265 after the loop
    CU(cudaStreamSynchronize(hp.down));
    CU(cudaStreamSynchronize(h->stream));
    return FLUID_OK;
}

int fluid_pressure_solve_host(fluid_t* h, const float* div_host, float* p_host, int iters) {
    if (!h || !div_host || !p_host || iters < 0) return fail(h, FLUID_ERR_INVALID, "bad argument");
    if (h->half) {
        int rc = fluid_write(h, FLUID_FIELD_DIVERGENCE, div_host, (size_t)h->cfg.sim_w * h->cfg.sim_h);
        if (!rc) rc = fluid_write(h, FLUID_FIELD_PRESSURE, p_host, (size_t)h->cfg.sim_w * h->cfg.sim_h);
        if (!rc) rc = run_jacobi(h, iters, true, nullptr);
        if (!rc) rc = fluid_read(h, FLUID_FIELD_PRESSURE, p_host, (size_t)h->cfg.sim_w * h->cfg.sim_h);
        return rc;
    }
    // one GPU, blocked kernel: solve band by band behind the copies (FLUID_E2E_BANDS=1 keeps the one-piece path)
    if (!h->slab() && iters > 0 && tb_eligible(h) && !(h->cfg.flags & FLUID_FLAG_NAIVE_JACOBI) && h->cfg.jacobi_block != 1 && !tb_use_tma(h)) {
        static const int bands_env = getenv("FLUID_E2E_BANDS") ? atoi(getenv("FLUID_E2E_BANDS")) : 16;
        int nb = std::min(std::min(bands_env, 16), h->cfg.sim_h / std::max(256, 4 * iters));
        if (nb >= 2) return solve_host_banded(h, div_host, p_host, iters, nb);
    }
    const size_t n = (size_t)h->cfg.sim_w * (h->row1 - h->row0);   // owned rows
    const size_t go = (size_t)h->G * h->cfg.sim_w;
    // Host buffers may be pageable; pinned ones (cudaHostAlloc / cudaHostRegister by the caller)
    // make the copies asynchronous DMA.  Either way all three copies are inside this call.
    CU(cudaMemcpyAsync(h->divergence + go, div_host, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync((float*)h->pressure.read + go, p_host, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    h->p_mirror_valid = false;
    int rc = clear_tiny_map(h); if (rc) return rc;
    if ((rc = scan_tiny(h, h->row0, h->row1))) return rc;
    rc = run_jacobi(h, iters, true, nullptr); if (rc) return rc;
    CU(cudaMemcpyAsync(p_host, (float*)h->pressure.read + go, n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return FLUID_OK;
}

// The band of a width x height target this handle draws: the whole target on one GPU, rows
// [height*rank/world, height*(rank+1)/world) on a slab rank (the same fractions as the dye rows it owns).
int fluid_render_band(fluid_t* h, int height, int* y0, int* y1) {
    if (!h || height < 1 || !y0 || !y1) return FLUID_ERR_INVALID;
    *y0 = (int)((long long)height * h->rank / h->world);
    *y1 = (int)((long long)height * (h->rank + 1) / h->world);
    return FLUID_OK;
}

// render(target) of S:1296-1317 for config.BLOOM = config.SUNRAYS = false: the background selected by
// FLUID_BACKGROUND (colour / checkerboard / none), then the display shader (optionally SHADING) blended over it.
int fluid_render(fluid_t* h, int width, int height, int shading, float back_r, float back_g,
                 float back_b, float* host_rgba, size_t n_floats) {
    if (!h || !host_rgba || width < 1 || height < 1) return fail(h, FLUID_ERR_INVALID, "bad argument");
    int y0, y1;
    fluid_render_band(h, height, &y0, &y1);
    const size_t cells = (size_t)width * (y1 - y0);
    if (n_floats != 4 * cells) return fail(h, FLUID_ERR_INVALID, "render target band has %zu floats, caller passed %zu", 4 * cells, n_floats);
    if (cells == 0) return FLUID_OK;
    if (cells > h->frame_cells) {
        CU(cudaStreamSynchronize(h->stream));
        cudaFree(h->frame); h->frame = nullptr; h->frame_cells = 0;
        CU(cudaMalloc((void**)&h->frame, cells * sizeof(float4)));
        h->frame_cells = cells;
    }
    if (h->slab()) {
        // the band's display + shading taps reach ceil(Hd / height) + 2 dye rows beyond the owned ones:
        // refresh that many ghost rows (the ghost rows of dye.read are stale after advection)
        const int need = std::min(h->Gd, (h->cfg.dye_h + height - 1) / height + 2);
        int rc = exchange_rows(h, HB_DYE, h->dye.read, (size_t)h->cfg.dye_w * sizeof(float4), h->droff, h->drow0, h->drow1, need);
        if (rc) return rc;
        if ((h->cfg.dye_h + height - 1) / height + 2 > h->Gd)
            return fail(h, FLUID_ERR_HALO, "render target of %d rows needs %d dye ghost rows, the slab keeps %d", height,
                        (h->cfg.dye_h + height - 1) / height + 2, h->Gd);
    }
    const float4* dye_src = (const float4*)h->dye.read;
    if (h->half) {                                   // the sampler widens fp16 texels exactly; shading is fp32 as in the shader
        const size_t nd = (size_t)h->cfg.dye_w * h->cfg.dye_h * 4;
        int rc = need_scratch(h, nd); if (rc) return rc;
        hs::widen_kernel<<<(unsigned)((nd + 255) / 256), 256, 0, h->stream>>>((const hs::h1*)h->dye.read, h->scratch, nd);
        if ((rc = check_launch(h, "hs::widen_kernel"))) return rc;
        dye_src = (const float4*)h->scratch;
    }
    dim3 b(32, 8);
    display_kernel<<<grid2d(width, y1 - y0, b), b, 0, h->stream>>>(dye_src, h->cfg.dye_w, h->cfg.dye_h,
                                                                   h->frame, width, height, shading, back_r, back_g, back_b,
                                                                   make_float2((float)(1.0 / (double)width), (float)(1.0 / (double)height)),
                                                                   h->background, h->cfg.aspect, h->droff, y0, y1);
    int rc = check_launch(h, "display_kernel"); if (rc) return rc;
    CU(cudaMemcpyAsync(host_rgba, h->frame, cells * sizeof(float4), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return FLUID_OK;
}


// render(null) of S:1296-1317 with config.SHADING = BLOOM = SUNRAYS = true (the reference's desktop
// defaults S:70-84), TRANSPARENT = false: applyBloom (S:1350-1394), applySunrays + blur(…, 1)
// (S:1396-1419; the mask is drawn into dye.write exactly like S:1300), drawColor, drawDisplay.
// FBO sizes follow initBloomFramebuffers / initSunraysFramebuffers (S:1012-1043).
int fluid_render_postfx(fluid_t* h, int width, int height, const fluid_postfx* fx, const float* dither_rgb,
                        int dw, int dh, float back_r, float back_g, float back_b, float* host_rgba,
                        size_t n_floats, float* host_bloom, float* host_sunrays) {
    if (!h || !fx || !dither_rgb || !host_rgba || width < 1 || height < 1 || dw < 1 || dh < 1)
        return fail(h, FLUID_ERR_INVALID, "bad argument");
    if (h->slab()) return not_on_slab(h, "fluid_render_postfx");
    const size_t cells = (size_t)width * height;
    if (n_floats != 4 * cells) return fail(h, FLUID_ERR_INVALID, "render target has %zu floats, caller passed %zu", 4 * cells, n_floats);
    int bw, bh, sw, sh;
    fluid_get_resolution(fx->bloom_resolution, width, height, &bw, &bh);
    fluid_get_resolution(fx->sunrays_resolution, width, height, &sw, &sh);
    if (bw < 1 || bh < 1 || sw < 1 || sh < 1) return fail(h, FLUID_ERR_INVALID, "bad post-FX resolution");
    std::vector<void*> tmp;
    const int rc = h->half
        ? render_postfx_chain<hs::h4, hs::h1>(h, width, height, fx, dither_rgb, dw, dh, back_r, back_g, back_b, host_rgba,
                                              host_bloom, host_sunrays, bw, bh, sw, sh, tmp)
        : render_postfx_chain<float4, float>(h, width, height, fx, dither_rgb, dw, dh, back_r, back_g, back_b, host_rgba,
                                             host_bloom, host_sunrays, bw, bh, sw, sh, tmp);
    cudaStreamSynchronize(h->stream);
    for (void* p : tmp) cudaFree(p);
    return rc;
}

void* fluid_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (bytes == 0 || cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void fluid_host_free(void* p) { if (p) cudaFreeHost(p); }

int fluid_sync(fluid_t* h) {
    if (!h) return FLUID_ERR_INVALID;
    CU(cudaStreamSynchronize(h->stream));
    return check_halo(h);
}

int fluid_timing_last(fluid_t* h, fluid_timing* out) {
    if (!h || !out) return FLUID_ERR_INVALID;
    if (!h->have_timing) return fail(h, FLUID_ERR_INVALID, "per-pass timing needs FLUID_FLAG_NO_GRAPH");
    CU(cudaStreamSynchronize(h->stream));
    float ms[5];
    for (int k = 0; k < 5; ++k) CU(cudaEventElapsedTime(&ms[k], h->tev[k], h->tev[k + 1]));
    h->timing.curl_vort_div_ms = ms[0]; h->timing.jacobi_ms = ms[1]; h->timing.gradient_ms = ms[2];
    h->timing.advect_velocity_ms = ms[3]; h->timing.advect_dye_ms = ms[4];
    CU(cudaEventElapsedTime(&h->timing.total_ms, h->tev[0], h->tev[5]));
    *out = h->timing;
    return FLUID_OK;
}

int fluid_mark(fluid_t* h, int slot) {
    if (!h || slot < 0 || slot > 1) return FLUID_ERR_INVALID;
    CU(cudaEventRecord(h->mark[slot], h->stream));
    return FLUID_OK;
}

int fluid_elapsed_ms(fluid_t* h, float* ms) {
    if (!h || !ms) return FLUID_ERR_INVALID;
    CU(cudaEventSynchronize(h->mark[1]));
    CU(cudaEventElapsedTime(ms, h->mark[0], h->mark[1]));
    return FLUID_OK;
}

uint64_t fluid_launch_count(fluid_t* h) { return h ? h->launches : 0; }

uint64_t fluid_stat(fluid_t* h, int key) {
    if (!h) return 0;
    switch (key) {
        case FLUID_STAT_LAUNCHES: return h->launches;
        case FLUID_STAT_JACOBI_LAUNCHES: return h->jacobi_kernel_launches;
        case FLUID_STAT_HALO_LAUNCHES: return h->halo_kernel_launches;
        case FLUID_STAT_HALO_EXCHANGES: return h->halo_groups;
        case FLUID_STAT_GRAPH_CAPTURES: return h->graph_captures;
        case FLUID_STAT_GRAPH_LAUNCHES: return h->graph_launches;
        case FLUID_STAT_HALO_TRANSPORT_P2P: return h->p2p ? 1 : 0;
    }
    return 0;
}

void* fluid_device_ptr(fluid_t* h, int field) {
    void* p; int w, rows, ch;
    if (!h || field_info(h, field, &p, &w, &rows, &ch)) return nullptr;
    return p;
}

}  // extern "C"
