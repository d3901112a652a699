// C-ABI glue of libbsplat.so: utility entry points, the rasterizer entry and the fused
// render path (render.py:63-101 of the reference chained on one stream).
#include <stdio.h>
#include <string.h>

#include "binning.cuh"

namespace bsplat {
int bin2_begin(int64_t N, void* workspace, size_t workspace_bytes, cudaStream_t stream);
void bin2_prep_targets(void* workspace, int64_t N, bool compact, uint2** rects_in, uint32_t** dkeys, uint32_t** hist);
int bin2_prepare(int64_t N, const float* means2d, const void* radii, int radii_is_float, const float* depths,
                 const BinParams& p, void* workspace, size_t workspace_bytes, cudaStream_t stream, bool have_prep,
                 bool compact, bool use_candidates);
int bin2_band_candidates(int64_t N, const float* means3d, const float* log_scales, const bsplat_camera& cam,
                         float eps2d, const BinParams& p, void* workspace, size_t workspace_bytes,
                         cudaStream_t stream, const int32_t** list, const unsigned long long** list_n);
int bin2_finish(int64_t N, int64_t M, bool device_m, const BinParams& p, void* workspace, size_t workspace_bytes,
                int32_t* sorted_ids, int32_t* tile_ranges, int32_t* tile_order, cudaStream_t stream, bool compact,
                bsplat_bin_info* info_host = nullptr);
int project_fwd_launch(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                       const float* opacities, const bsplat_camera& cam, float eps2d, int semantics,
                       float* means2d, float* conics, float* depths, int32_t* radii, cudaStream_t stream,
                       const bsplat_camera* cam_dev, const ProjExtra* extra, int variant);
int rasterize_launch(int64_t N, int channels, const float* means2d, const float* conics, const float* colors,
                     const float* opacities, const float* background_dev, const int32_t* tile_ranges,
                     const int32_t* tile_order, const int32_t* sorted_ids, int W, int H, int tile_size,
                     int row_begin, int row_end, int mode, float* image, unsigned long long* stats,
                     const unsigned long long* m_dev, void* rec_ws, cudaStream_t stream,
                     const PeerImages* peers = nullptr, const int32_t* rec_list = nullptr,
                     const unsigned long long* rec_list_n = nullptr, bool rec_ready = false,
                     int32_t* surv = nullptr, uint32_t* chunk_cnt = nullptr, uint32_t* long_barrier = nullptr);
uint32_t* bin2_spare_counter(void* workspace, int64_t N, int64_t M, int64_t n_tiles);
void bin2_band_list(void* workspace, int64_t N, const int32_t** perm, const unsigned long long** n_band);
size_t raster_workspace_bytes(int64_t N);
size_t raster_long_surv_bytes(int64_t M_cap);
size_t raster_long_cnt_bytes(int64_t M_cap, int64_t n_tiles);
int tile_order_launch(int first_tile, int n_tiles, const int32_t* tile_ranges, int32_t* order,
                      cudaStream_t stream);
}  // namespace bsplat

using namespace bsplat;

extern "C" int bsplat_version(void) { return BSPLAT_VERSION; }

extern "C" const char* bsplat_error_string(int code) {
    switch (code) {
        case BSPLAT_OK: return "ok";
        case BSPLAT_E_ARG: return "bsplat: invalid argument";
        case BSPLAT_E_WORKSPACE: return "bsplat: workspace too small";
        case BSPLAT_E_OVERFLOW: return "bsplat: too many tile intersections (>= 2^30)";
        case BSPLAT_E_NODEVICE: return "bsplat: no sm_100 CUDA device";
        default: break;
    }
    if (code > 0) return cudaGetErrorString(static_cast<cudaError_t>(code));
    return "bsplat: unknown error";
}

extern "C" int bsplat_check_device(int device) {
    int dev = device;
    if (dev < 0) {
        if (cudaGetDevice(&dev) != cudaSuccess) return BSPLAT_E_NODEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return BSPLAT_E_NODEVICE;
    return (prop.major == 10) ? BSPLAT_OK : BSPLAT_E_NODEVICE;
}

extern "C" int bsplat_rasterize_fwd(int64_t N, int32_t channels, const float* means2d, const float* conics,
                                    const float* colors, const float* opacities, const float* background,
                                    const int32_t* tile_ranges, const int32_t* tile_order,
                                    const int32_t* sorted_ids, int64_t M, int32_t width, int32_t height,
                                    int32_t tile_size, int32_t tile_row_begin, int32_t tile_row_end,
                                    int32_t mode, float* image, void* workspace, size_t workspace_bytes,
                                    void* stream) {
    if (N < 0 || M < 0 || !tile_ranges || !image || !background) return BSPLAT_E_ARG;
    if (M > 0 && (!sorted_ids || !means2d || !conics || !colors || !opacities)) return BSPLAT_E_ARG;
    // the record workspace is optional: without it the fast mode runs the (slower) workspace-free kernel
    void* rec_ws = (workspace && workspace_bytes >= raster_workspace_bytes(N)) ? workspace : nullptr;
    return rasterize_launch(N, channels, means2d, conics, colors, opacities, background, tile_ranges, tile_order,
                            sorted_ids, width, height, tile_size, tile_row_begin, tile_row_end, mode, image,
                            nullptr, nullptr, rec_ws, (cudaStream_t)stream);
}

extern "C" size_t bsplat_rasterize_workspace_bytes(int64_t N) { return N < 0 ? 0 : raster_workspace_bytes(N); }

extern "C" int bsplat_tile_order(int32_t first_tile, int32_t n_tiles, const int32_t* tile_ranges,
                                 int32_t* tile_order, void* stream) {
    if (first_tile < 0 || n_tiles < 0 || !tile_ranges || !tile_order) return BSPLAT_E_ARG;
    return tile_order_launch(first_tile, n_tiles, tile_ranges, tile_order, (cudaStream_t)stream);
}

// Same as bsplat_rasterize_fwd but always the faithful kernel, and counts the evaluated /
// contributing (pixel, Gaussian) pairs into stats[2] (device, uint64, caller-zeroed): the
// algorithmic work figures E_all / E_pass of SURVEY.md 8d.
extern "C" int bsplat_rasterize_stats(int64_t N, int32_t channels, const float* means2d, const float* conics,
                                      const float* colors, const float* opacities, const float* background,
                                      const int32_t* tile_ranges, const int32_t* sorted_ids, int64_t M,
                                      int32_t width, int32_t height, int32_t tile_size, float* image,
                                      uint64_t* stats, void* stream) {
    if (N < 0 || M < 0 || !tile_ranges || !image || !background || !stats) return BSPLAT_E_ARG;
    return rasterize_launch(N, channels, means2d, conics, colors, opacities, background, tile_ranges, nullptr,
                            sorted_ids, width, height, tile_size, 0, 1 << 30, BSPLAT_RASTER_FAITHFUL, image,
                            reinterpret_cast<unsigned long long*>(stats), nullptr, nullptr, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------
// fused render
// ------------------------------------------------------------------------------------------
namespace bsplat {
size_t bin2_workspace_bytes(int64_t N, int64_t M, int64_t n_tiles);
bsplat_bin_info* bin2_info_ptr(void* workspace, int64_t N);
}  // namespace bsplat

namespace {

constexpr size_t kAlign = 256;
inline size_t align_up(size_t v) { return (v + kAlign - 1) / kAlign * kAlign; }

struct RenderWs {
    float* means2d; float* conics; float* depths; int32_t* radii;
    int32_t* tile_ranges; int32_t* tile_order; int32_t* sorted_ids;
    bsplat_camera* cam_dev;  // indirect camera of captured frames
    void* raster_rec;        // 48 B per Gaussian: raster records (projection epilogue / raster_pair_prep_kernel)
    int32_t* long_surv;      // [M] survivor ids of the long-list pre-pass
    uint32_t* long_cnt;      // per-chunk survivor counts of the long-list pre-pass
    void* bin_ws; size_t bin_bytes;
    size_t total;
};

RenderWs carve_render(void* base, int64_t N, int64_t M, int W, int H, int tile_size) {
    RenderWs w;
    char* p = static_cast<char*>(base);
    size_t off = 0;
    auto take = [&](size_t bytes) { void* r = p ? p + off : nullptr; off += align_up(bytes); return r; };
    const size_t n = (size_t)(N > 0 ? N : 1), m = (size_t)(M > 0 ? M : 1);
    const int tiles_w = (W + tile_size - 1) / tile_size, tiles_h = (H + tile_size - 1) / tile_size;
    w.means2d = (float*)take(n * 2 * sizeof(float));
    w.conics = (float*)take(n * 3 * sizeof(float));
    w.depths = (float*)take(n * sizeof(float));
    w.radii = (int32_t*)take(n * 2 * sizeof(int32_t));
    w.tile_ranges = (int32_t*)take((size_t)tiles_w * tiles_h * 2 * sizeof(int32_t));
    w.tile_order = (int32_t*)take((size_t)tiles_w * tiles_h * sizeof(int32_t));
    w.cam_dev = (bsplat_camera*)take(sizeof(bsplat_camera));
    w.raster_rec = take(raster_workspace_bytes(N));
    // the N-dependent part of the binning scratch comes first so that it survives the re-carve with M
    w.bin_bytes = bin2_workspace_bytes(N, M, (int64_t)tiles_w * tiles_h);
    w.bin_ws = take(w.bin_bytes);
    w.sorted_ids = (int32_t*)take(m * sizeof(int32_t));
    w.long_surv = (int32_t*)take(raster_long_surv_bytes(M));
    w.long_cnt = (uint32_t*)take(raster_long_cnt_bytes(M, (int64_t)tiles_w * tiles_h));
    w.total = off;
    return w;
}

// The arguments of a fused frame after the checks every frame entry point shares, and what follows from them.  Each
// entry point adds its own rules (N > 0, M, streams, which Gaussian arrays must be present).
struct Frame {
    int64_t N;
    const float *means3d, *log_scales, *quats, *opacities, *colors, *background;
    float* image;
    const bsplat_camera* cam;
    int channels, tile_size, semantics, flags, raster_mode;
    bool fast_raster;  // the fast kernel with raster records and the longest-first tile order (16x16 tiles, RGB)
    int W, H, tiles_w, tiles_h;
    int row0, row1;    // tile rows that are binned and rasterized: all of them unless a band entry narrows them
};

int make_frame(int64_t N, const float* means3d, const float* log_scales, const float* quats, const float* opacities,
               const float* colors, int channels, const bsplat_camera* cam, const float* background, int tile_size,
               int semantics, int flags, float* image, Frame* f) {
    if (!cam || N < 0 || tile_size <= 0 || tile_size > 32) return BSPLAT_E_ARG;
    if (semantics != BSPLAT_SEM_TORCH && semantics != BSPLAT_SEM_GSPLAT) return BSPLAT_E_ARG;
    if (cam->width <= 0 || cam->height <= 0) return BSPLAT_E_ARG;
    f->N = N;
    f->means3d = means3d; f->log_scales = log_scales; f->quats = quats; f->opacities = opacities;
    f->colors = colors; f->background = background; f->image = image;
    f->cam = cam;
    f->channels = channels; f->tile_size = tile_size; f->semantics = semantics; f->flags = flags;
    f->raster_mode = flags & 0xff;
    f->fast_raster = (f->raster_mode == BSPLAT_RASTER_FAST || f->raster_mode == BSPLAT_RASTER_FAST_NOCULL) &&
                     tile_size == 16 && channels == 3;
    f->W = cam->width; f->H = cam->height;
    f->tiles_w = (f->W + tile_size - 1) / tile_size;
    f->tiles_h = (f->H + tile_size - 1) / tile_size;
    f->row0 = 0; f->row1 = f->tiles_h;
    return BSPLAT_OK;
}

// CUDA events of the per-stage timing; destroyed on every exit path
struct StageEvents {
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    bool on = false;
    int create() {
        on = true;
        for (auto& e : ev) BSPLAT_CUDA_TRY(cudaEventCreate(&e));
        return BSPLAT_OK;
    }
    int record(int k, cudaStream_t s) {
        if (on) BSPLAT_CUDA_TRY(cudaEventRecord(ev[k], s));
        return BSPLAT_OK;
    }
    ~StageEvents() {
        for (auto& e : ev)
            if (e) cudaEventDestroy(e);
    }
};

// Front half of a frame: control words zeroed, projection with the fused epilogue (tile rectangles, depth keys +
// histograms, raster records), [compaction,] depth sort, count + scan.  o_*: also store the reference's four projection
// outputs (needed by the faithful rasterizer, the aux outputs and nobody else); nullptr skips them.
int frame_front(const Frame& f, const bsplat_camera* cam_dev, bool want_rec, float* o_means2d, float* o_conics,
                float* o_depths, int32_t* o_radii, const RenderWs& w, cudaStream_t stream,
                cudaEvent_t ev_after_projection = nullptr) {
    BinParams p;
    int rc = make_bin_params(f.W, f.H, f.tile_size, f.row0, f.row1, f.semantics, &p);
    if (rc != BSPLAT_OK) return rc;
    const bool compact = (f.flags & BSPLAT_FLAG_PACKED) != 0 || p.row_begin > 0 || p.row_end < p.tiles_h;
    rc = bin2_begin(f.N, w.bin_ws, w.bin_bytes, stream);
    if (rc != BSPLAT_OK) return rc;
    ProjExtra ex;
    bin2_prep_targets(w.bin_ws, f.N, compact, &ex.rects, &ex.dkeys, &ex.hist);
    ex.rec = want_rec ? w.raster_rec : nullptr;
    ex.colors = f.colors;
    ex.opac = f.opacities;
    ex.tile_size = f.tile_size;
    ex.rec_row_begin = p.row_begin;
    ex.rec_row_end = p.row_end;
    // Row bands under the torch rules (and nobody asking for the stage outputs): a cheap conservative pre-test on
    // the raw inputs first lists the Gaussians whose rectangle can reach the band at all; only those are projected
    // and compacted.  (What every rank of a band split repeats shrinks from all N to its candidates.)
    const bool band = p.row_begin > 0 || p.row_end < p.tiles_h;
    const bool pretest = band && f.semantics == BSPLAT_SEM_TORCH && cam_dev == nullptr && o_means2d == nullptr &&
                         (f.flags & BSPLAT_FLAG_NO_BAND_PRETEST) == 0 && f.N > 0;
    if (pretest) {
        rc = bin2_band_candidates(f.N, f.means3d, f.log_scales, *f.cam, 0.3f, p, w.bin_ws, w.bin_bytes, stream,
                                  &ex.list, &ex.list_n);
        if (rc != BSPLAT_OK) return rc;
    }
    rc = project_fwd_launch(f.N, f.means3d, f.log_scales, f.quats, f.opacities, *f.cam, 0.3f, f.semantics, o_means2d,
                            o_conics, o_depths, o_radii, stream, cam_dev, &ex, 0);
    if (rc != BSPLAT_OK) return rc;
    if (ev_after_projection) BSPLAT_CUDA_TRY(cudaEventRecord(ev_after_projection, stream));
    return bin2_prepare(f.N, nullptr, nullptr, 0, nullptr, p, w.bin_ws, w.bin_bytes, stream, /*have_prep=*/true, compact,
                        pretest);
}

// Back half of a frame: emission, tile sort, tile ranges and tile order (bin2_finish), then the rasterizer.
// M is the pair count the caller read back or, with device_m, the capacity of the pair buffers (the real count stays on
// the device).  Binning runs on sb, the rasterizer on sr; when they differ, event_bin_done orders the two.
// rec_ready: the front half built the raster records.  info_host (nullable): pinned host block that receives the frame's
// bin info.  te (nullable): stage-timing marks 2 (before the emission) and 3 (before the rasterizer).
int frame_back(const Frame& f, const RenderWs& w, int64_t M, bool device_m, const float* means2d, const float* conics,
               int32_t* tile_ranges, bool rec_ready, const PeerImages* peers, cudaStream_t sb, cudaStream_t sr,
               cudaEvent_t event_bin_done, bsplat_bin_info* info_host, StageEvents* te) {
    BinParams p;
    int rc = make_bin_params(f.W, f.H, f.tile_size, f.row0, f.row1, f.semantics, &p);
    if (rc != BSPLAT_OK) return rc;
    if (te && (rc = te->record(2, sb)) != BSPLAT_OK) return rc;
    // the bin info reaches the host as a store from the last binning kernel when the block is device-accessible
    // (pinned memory under UVA); a copy-engine transfer would queue behind image downloads of earlier frames
    bool info_direct = false;
    if (info_host) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, info_host) == cudaSuccess && attr.type == cudaMemoryTypeHost &&
            attr.devicePointer == (void*)info_host)
            info_direct = true;
        else
            (void)cudaGetLastError();
    }
    rc = bin2_finish(f.N, M, device_m, p, w.bin_ws, w.bin_bytes, w.sorted_ids, tile_ranges, w.tile_order, sb,
                     (f.flags & BSPLAT_FLAG_PACKED) != 0, info_direct ? info_host : nullptr);
    if (rc != BSPLAT_OK) return rc;
    const bsplat_bin_info* d_info = bin2_info_ptr(w.bin_ws, f.N);
    if (info_host && !info_direct)
        BSPLAT_CUDA_TRY(cudaMemcpyAsync(info_host, d_info, sizeof(bsplat_bin_info), cudaMemcpyDeviceToHost, sb));
    if (sr != sb) {
        BSPLAT_CUDA_TRY(cudaEventRecord(event_bin_done, sb));
        BSPLAT_CUDA_TRY(cudaStreamWaitEvent(sr, event_bin_done, 0));
    }
    const unsigned long long* m_dev = nullptr;
    if (device_m) {
        // "no intersections at all => all-zero image" (render.py:73-76) is a whole-frame rule: a partial band decides
        // it from the number of Gaussians that own a tile anywhere in the frame (counted by the compaction pass)
        m_dev = reinterpret_cast<const unsigned long long*>(d_info);
        if (f.row0 > 0 || f.row1 < f.tiles_h) {
            const int32_t* perm;
            const unsigned long long* n_band;
            bin2_band_list(w.bin_ws, f.N, &perm, &n_band);
            m_dev = n_band + 1;
        }
    }
    if (te && (rc = te->record(3, sr)) != BSPLAT_OK) return rc;
    return rasterize_launch(f.N, f.channels, means2d, conics, f.colors, f.opacities, f.background, tile_ranges,
                            f.fast_raster ? w.tile_order : nullptr, w.sorted_ids, f.W, f.H, f.tile_size, f.row0,
                            f.row1, f.raster_mode, f.image, nullptr, m_dev, w.raster_rec, sr, peers, nullptr, nullptr,
                            rec_ready, w.long_surv, w.long_cnt,
                            bin2_spare_counter(w.bin_ws, f.N, M, (int64_t)f.tiles_w * f.tiles_h));
}

}  // namespace

extern "C" size_t bsplat_render_workspace_bytes(int64_t N, int64_t M_capacity, int32_t width, int32_t height,
                                                int32_t tile_size) {
    if (N < 0 || M_capacity < 0 || width <= 0 || height <= 0 || tile_size <= 0) return 0;
    return carve_render(nullptr, N, M_capacity, width, height, tile_size).total;
}

extern "C" int bsplat_render_fwd(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                                 const float* opacities, const float* colors, int32_t channels,
                                 const bsplat_camera* cam, const float* background, int32_t tile_size,
                                 int32_t semantics, int32_t flags, float* image, void* workspace,
                                 size_t workspace_bytes, size_t* needed_bytes, bsplat_render_aux* aux,
                                 void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    Frame f;
    int rc = make_frame(N, means3d, log_scales, quats, opacities, colors, channels, cam, background, tile_size,
                        semantics, flags, image, &f);
    if (rc != BSPLAT_OK) return rc;
    if (!image || !background || channels <= 0) return BSPLAT_E_ARG;
    if (N > 0 && (!means3d || !log_scales || !quats || !opacities || !colors)) return BSPLAT_E_ARG;
    const size_t image_bytes = (size_t)f.W * f.H * channels * sizeof(float);
    if (aux) { aux->n_isect = 0; aux->n_launches = 0; aux->sort_passes = 0; aux->key_bits = 0; }

    // fixed (N-dependent) part must fit before anything runs
    RenderWs w = carve_render(workspace, N, 0, f.W, f.H, tile_size);
    if (!workspace || workspace_bytes < w.total) {
        if (needed_bytes) *needed_bytes = bsplat_render_workspace_bytes(N, 4 * N + 1024, f.W, f.H, tile_size);
        return BSPLAT_E_WORKSPACE;
    }
    if (N == 0) {
        BSPLAT_CUDA_TRY(cudaMemsetAsync(image, 0, image_bytes, stream));
        return BSPLAT_OK;
    }
    StageEvents te;
    if (aux && aux->timing) {
        rc = te.create();
        if (rc != BSPLAT_OK) return rc;
    }
    rc = te.record(0, stream);
    if (rc != BSPLAT_OK) return rc;
    const bool want_aux = aux && (aux->means2d || aux->conics || aux->depths || aux->radii);
    // the reference's four projection outputs are only stored when somebody reads them
    const bool stage_outputs = !f.fast_raster || want_aux;
    float* d_means2d = (aux && aux->means2d) ? aux->means2d : w.means2d;
    float* d_conics = (aux && aux->conics) ? aux->conics : w.conics;
    float* d_depths = (aux && aux->depths) ? aux->depths : w.depths;
    int32_t* d_radii = (aux && aux->radii) ? aux->radii : w.radii;
    int32_t* d_ranges = (aux && aux->tile_ranges) ? aux->tile_ranges : w.tile_ranges;
    rc = frame_front(f, nullptr, f.fast_raster, stage_outputs ? d_means2d : nullptr, stage_outputs ? d_conics : nullptr,
                     stage_outputs ? d_depths : nullptr, stage_outputs ? d_radii : nullptr, w, stream,
                     te.on ? te.ev[1] : nullptr);
    if (rc != BSPLAT_OK) return rc;
    bsplat_bin_info info;
    BSPLAT_CUDA_TRY(cudaMemcpyAsync(&info, bin2_info_ptr(w.bin_ws, N), sizeof(info), cudaMemcpyDeviceToHost, stream));
    BSPLAT_CUDA_TRY(cudaStreamSynchronize(stream));  // the single read-back of the frame (M, key range)
    const int64_t M = (int64_t)info.n_isect;
    if (aux) { aux->n_isect = M; aux->n_launches = 6; }  // so far: project, 4 depth passes, count + scan
    if (M >= (1ll << 30)) return BSPLAT_E_OVERFLOW;
    if (M == 0) {
        // render.py:73-76: no overlaps => black image (not the background)
        BSPLAT_CUDA_TRY(cudaMemsetAsync(image, 0, image_bytes, stream));
        BSPLAT_CUDA_TRY(cudaMemsetAsync(d_ranges, 0, (size_t)f.tiles_w * f.tiles_h * 2 * sizeof(int32_t), stream));
        return BSPLAT_OK;
    }
    w = carve_render(workspace, N, M, f.W, f.H, tile_size);
    if (workspace_bytes < w.total) {
        if (needed_bytes) *needed_bytes = bsplat_render_workspace_bytes(N, M + M / 4, f.W, f.H, tile_size);
        return BSPLAT_E_WORKSPACE;
    }
    if (aux) {
        int tb = 1;
        while ((1 << tb) < f.tiles_w * f.tiles_h) ++tb;
        const int tile_passes = (tb + 7) / 8;
        aux->key_bits = 32 + tb;
        aux->sort_passes = 4 + tile_passes;  // 4 over N items, the rest over M items
        // project (+ epilogue), [compact,] 4 passes, count_scan | emit, tile passes, tile_finish | [long-list
        // pre-pass,] rasterizer
        aux->n_launches = 1 + ((flags & BSPLAT_FLAG_PACKED) ? 1 : 0) + 4 + 1 + 1 + tile_passes + 1 +
                          (f.fast_raster ? 1 : 0) + 1;
    }
    // stage_ms: [0] projection (+ epilogue), [1] depth sort + count/scan (+ the M read-back), [2] emit + tile sort +
    // ranges, [3] rasterizer (+ long-list pre-pass)
    rc = frame_back(f, w, M, /*device_m=*/false, d_means2d, d_conics, d_ranges, /*rec_ready=*/f.fast_raster, nullptr,
                    stream, stream, nullptr, nullptr, &te);
    if (rc != BSPLAT_OK) return rc;
    if (aux && aux->sorted_ids && aux->sorted_ids_capacity >= M)
        BSPLAT_CUDA_TRY(cudaMemcpyAsync(aux->sorted_ids, w.sorted_ids, (size_t)M * sizeof(int32_t),
                                        cudaMemcpyDeviceToDevice, stream));
    if (te.on) {
        rc = te.record(4, stream);
        if (rc != BSPLAT_OK) return rc;
        BSPLAT_CUDA_TRY(cudaEventSynchronize(te.ev[4]));
        for (int s = 0; s < 4; ++s) cudaEventElapsedTime(&aux->stage_ms[s], te.ev[s], te.ev[s + 1]);
    }
    return BSPLAT_OK;
}

// ------------------------------------------------------------------------------------------
// split-phase frame: begin = project + depth sort + count/scan (N-scale, latency-bound) and an async
// copy of M into pinned host memory; end = emit + tile sort + ranges + order + raster (M-scale).
// A two-stream pipeline overlaps begin(k+1) with end(k) (mojosplat_b200/pipeline.py).
// ------------------------------------------------------------------------------------------
extern "C" int bsplat_render_begin(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                                   const float* opacities, const bsplat_camera* cam, int32_t tile_size,
                                   int32_t semantics, void* workspace, size_t workspace_bytes,
                                   bsplat_bin_info* info_host_pinned, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    Frame f;
    int rc = make_frame(N, means3d, log_scales, quats, opacities, nullptr, 0, cam, nullptr, tile_size, semantics, 0,
                        nullptr, &f);
    if (rc != BSPLAT_OK) return rc;
    if (!info_host_pinned || N <= 0 || !means3d || !log_scales || !quats) return BSPLAT_E_ARG;
    RenderWs w = carve_render(workspace, N, 0, f.W, f.H, tile_size);
    if (!workspace || workspace_bytes < w.total) return BSPLAT_E_WORKSPACE;
    // (colours arrive with bsplat_render_end: the raster records are built there, from the stage outputs kept here)
    rc = frame_front(f, nullptr, false, w.means2d, w.conics, w.depths, w.radii, w, stream);
    if (rc != BSPLAT_OK) return rc;
    BSPLAT_CUDA_TRY(cudaMemcpyAsync(info_host_pinned, bin2_info_ptr(w.bin_ws, N), sizeof(bsplat_bin_info),
                                    cudaMemcpyDeviceToHost, stream));
    return BSPLAT_OK;
}

extern "C" int bsplat_render_end(int64_t N, int64_t M, const float* colors, const float* opacities, int32_t channels,
                                 const bsplat_camera* cam, const float* background, int32_t tile_size,
                                 int32_t semantics, int32_t flags, float* image, void* workspace,
                                 size_t workspace_bytes, size_t* needed_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    // bsplat_render_begin ran without BSPLAT_FLAG_PACKED: only the rasterizer mode of `flags` applies here
    Frame f;
    int rc = make_frame(N, nullptr, nullptr, nullptr, opacities, colors, channels, cam, background, tile_size,
                        semantics, flags & 0xff, image, &f);
    if (rc != BSPLAT_OK) return rc;
    if (!image || !background || channels <= 0 || N <= 0 || M < 0 || !colors || !opacities) return BSPLAT_E_ARG;
    if (M >= (1ll << 30)) return BSPLAT_E_OVERFLOW;
    if (M == 0) {
        BSPLAT_CUDA_TRY(cudaMemsetAsync(image, 0, (size_t)f.W * f.H * channels * sizeof(float), stream));
        return BSPLAT_OK;
    }
    RenderWs w = carve_render(workspace, N, M, f.W, f.H, tile_size);
    if (!workspace || workspace_bytes < w.total) {
        if (needed_bytes) *needed_bytes = w.total;
        return BSPLAT_E_WORKSPACE;
    }
    return frame_back(f, w, M, /*device_m=*/false, w.means2d, w.conics, w.tile_ranges, /*rec_ready=*/false, nullptr,
                      stream, stream, nullptr, nullptr, nullptr);
}

// ------------------------------------------------------------------------------------------
// sync-free frame: nothing in here waits for the GPU.  The pair buffers are sized by M_capacity, the
// real M stays on the device (bin info written by the count+scan kernel) and every M-scale kernel
// reads it there; a frame that produces more than M_capacity pairs raises info.reserved[1] and renders
// nothing useful -- the caller looks at the (asynchronously copied) info once the frame is done and
// re-renders with a larger workspace.  Binning and rasterization may go to different streams
// (priorities): with the binning stream at high priority, binning(k+1) fills the slots that
// rasterization(k) frees, which hides the latency-bound binning kernels behind the issue-bound rasterizer.
// Capturable into a CUDA graph (single stream or fork/join through event_bin_done).
// ------------------------------------------------------------------------------------------
extern "C" int bsplat_render_enqueue(int64_t N, const float* means3d, const float* log_scales, const float* quats,
                                     const float* opacities, const float* colors, int32_t channels,
                                     const bsplat_camera* cam, const float* background, int32_t tile_size,
                                     int32_t semantics, int32_t flags, float* image, void* workspace,
                                     size_t workspace_bytes, int64_t M_capacity, size_t* needed_bytes,
                                     bsplat_bin_info* info_host_pinned, void* stream_bin_, void* stream_raster_,
                                     void* event_bin_done) {
    return bsplat_render_enqueue_band(N, means3d, log_scales, quats, opacities, colors, channels, cam, background,
                                      tile_size, semantics, flags, 0, 1 << 30, image, workspace, workspace_bytes,
                                      M_capacity, needed_bytes, info_host_pinned, stream_bin_, stream_raster_,
                                      event_bin_done);
}

// The same frame restricted to tile rows [tile_row_begin, tile_row_end): every Gaussian is projected, only the
// band is binned and rasterized, only the band's rows of `image` are written (row-band multi-GPU split).
extern "C" int bsplat_render_enqueue_band(int64_t N, const float* means3d, const float* log_scales,
                                          const float* quats, const float* opacities, const float* colors,
                                          int32_t channels, const bsplat_camera* cam, const float* background,
                                          int32_t tile_size, int32_t semantics, int32_t flags,
                                          int32_t tile_row_begin, int32_t tile_row_end, float* image,
                                          void* workspace, size_t workspace_bytes, int64_t M_capacity,
                                          size_t* needed_bytes, bsplat_bin_info* info_host_pinned,
                                          void* stream_bin_, void* stream_raster_, void* event_bin_done) {
    return bsplat_render_enqueue_band_p2p(N, means3d, log_scales, quats, opacities, colors, channels, cam, background,
                                          tile_size, semantics, flags, tile_row_begin, tile_row_end, image, nullptr, 0,
                                          workspace, workspace_bytes, M_capacity, needed_bytes, info_host_pinned,
                                          stream_bin_, stream_raster_, event_bin_done);
}

// ... and with the band exchange fused into the rasterizer: every finished tile is also stored into the image
// buffers of the n_peers other ranks (peer-mapped pointers, e.g. torch symmetric memory over NVLink/NVSwitch).
// The caller follows the call with a cross-device barrier on the stream; no all-gather is needed.
extern "C" int bsplat_render_enqueue_band_p2p(int64_t N, const float* means3d, const float* log_scales,
                                              const float* quats, const float* opacities, const float* colors,
                                              int32_t channels, const bsplat_camera* cam, const float* background,
                                              int32_t tile_size, int32_t semantics, int32_t flags,
                                              int32_t tile_row_begin, int32_t tile_row_end, float* image,
                                              float* const* peer_images, int32_t n_peers, void* workspace,
                                              size_t workspace_bytes, int64_t M_capacity, size_t* needed_bytes,
                                              bsplat_bin_info* info_host_pinned, void* stream_bin_,
                                              void* stream_raster_, void* event_bin_done) {
    if (n_peers < 0 || n_peers > kMaxPeers || (n_peers > 0 && !peer_images)) return BSPLAT_E_ARG;
    PeerImages peers;
    peers.n = n_peers;
    for (int q = 0; q < n_peers; ++q) {
        if (!peer_images[q]) return BSPLAT_E_ARG;
        peers.p[q] = peer_images[q];
    }
    cudaStream_t sb = (cudaStream_t)stream_bin_;
    cudaStream_t sr = stream_raster_ ? (cudaStream_t)stream_raster_ : sb;
    Frame f;
    int rc = make_frame(N, means3d, log_scales, quats, opacities, colors, channels, cam, background, tile_size,
                        semantics, flags, image, &f);
    if (rc != BSPLAT_OK) return rc;
    if (!image || !background || channels <= 0 || N <= 0 || M_capacity <= 0) return BSPLAT_E_ARG;
    if (!means3d || !log_scales || !quats || !opacities || !colors) return BSPLAT_E_ARG;
    if (M_capacity >= (1ll << 30)) return BSPLAT_E_OVERFLOW;
    if (sr != sb && !event_bin_done) return BSPLAT_E_ARG;
    RenderWs w = carve_render(workspace, N, M_capacity, f.W, f.H, tile_size);
    if (!workspace || workspace_bytes < w.total) {
        if (needed_bytes) *needed_bytes = w.total;
        return BSPLAT_E_WORKSPACE;
    }
    f.row0 = tile_row_begin < 0 ? 0 : tile_row_begin;
    f.row1 = tile_row_end > f.tiles_h ? f.tiles_h : tile_row_end;
    if (f.row1 <= f.row0) {
        // empty band: nothing to write, but the caller's status protocol still holds -- a zeroed info and the event
        bsplat_bin_info* d_info = bin2_info_ptr(w.bin_ws, N);
        BSPLAT_CUDA_TRY(cudaMemsetAsync(d_info, 0, sizeof(bsplat_bin_info), sb));
        if (info_host_pinned)
            BSPLAT_CUDA_TRY(cudaMemcpyAsync(info_host_pinned, d_info, sizeof(bsplat_bin_info), cudaMemcpyDeviceToHost, sb));
        if (sr != sb) {
            BSPLAT_CUDA_TRY(cudaEventRecord((cudaEvent_t)event_bin_done, sb));
            BSPLAT_CUDA_TRY(cudaStreamWaitEvent(sr, (cudaEvent_t)event_bin_done, 0));
        }
        return BSPLAT_OK;
    }
    const bsplat_camera* cam_dev = nullptr;
    if (flags & BSPLAT_FLAG_CAMERA_INDIRECT) {
        // `cam` is pinned host (or managed) memory: copied when the stream gets here, i.e. at every replay
        BSPLAT_CUDA_TRY(cudaMemcpyAsync(w.cam_dev, cam, sizeof(bsplat_camera), cudaMemcpyDefault, sb));
        cam_dev = w.cam_dev;
    }
    const PdlScope pdl_scope(sr == sb);  // two streams = overlapped pipeline: plain launches (common.cuh)
    // the faithful rasterizer reads the stage outputs; the fast one only needs the records of the projection epilogue
    const bool stage_outputs = !f.fast_raster;
    rc = frame_front(f, cam_dev, f.fast_raster, stage_outputs ? w.means2d : nullptr, stage_outputs ? w.conics : nullptr,
                     stage_outputs ? w.depths : nullptr, stage_outputs ? w.radii : nullptr, w, sb);
    if (rc != BSPLAT_OK) return rc;
    return frame_back(f, w, M_capacity, /*device_m=*/true, w.means2d, w.conics, w.tile_ranges,
                      /*rec_ready=*/f.fast_raster, &peers, sb, sr, (cudaEvent_t)event_bin_done, info_host_pinned,
                      nullptr);
}

extern "C" size_t bsplat_render_host_scratch_bytes(int64_t N, int32_t channels, int32_t width, int32_t height) {
    const size_t n = (size_t)(N > 0 ? N : 1);
    size_t off = 0;
    off += align_up(n * 3 * sizeof(float)) * 2;        // means3d, log_scales
    off += align_up(n * 4 * sizeof(float));            // quats
    off += align_up(n * sizeof(float));                // opacities
    off += align_up(n * (size_t)channels * sizeof(float));
    off += align_up((size_t)channels * sizeof(float)); // background
    off += align_up((size_t)width * height * channels * sizeof(float));
    return off;
}

extern "C" int bsplat_render_fwd_host(int64_t N, const float* means3d, const float* log_scales,
                                      const float* quats, const float* opacities, const float* colors,
                                      int32_t channels, const bsplat_camera* cam, const float* background,
                                      int32_t tile_size, int32_t semantics, int32_t flags,
                                      float* image_host, void* device_scratch, size_t scratch_bytes,
                                      void* workspace, size_t workspace_bytes, size_t* needed_bytes,
                                      bsplat_render_aux* aux, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!cam || !image_host || !background || N < 0 || channels <= 0) return BSPLAT_E_ARG;
    const int W = cam->width, H = cam->height;
    if (W <= 0 || H <= 0) return BSPLAT_E_ARG;
    // the scratch size is a pure function of the arguments (bsplat_render_host_scratch_bytes): a short buffer is a
    // caller error; *needed_bytes / BSPLAT_E_WORKSPACE always refer to the render workspace
    if (!device_scratch || scratch_bytes < bsplat_render_host_scratch_bytes(N, channels, W, H)) return BSPLAT_E_ARG;
    const size_t n = (size_t)(N > 0 ? N : 1);
    char* p = static_cast<char*>(device_scratch);
    size_t off = 0;
    auto take = [&](size_t bytes) { void* r = p + off; off += align_up(bytes); return r; };
    float* d_means = (float*)take(n * 3 * sizeof(float));
    float* d_scales = (float*)take(n * 3 * sizeof(float));
    float* d_quats = (float*)take(n * 4 * sizeof(float));
    float* d_opac = (float*)take(n * sizeof(float));
    float* d_colors = (float*)take(n * (size_t)channels * sizeof(float));
    float* d_bg = (float*)take((size_t)channels * sizeof(float));
    float* d_image = (float*)take((size_t)W * H * channels * sizeof(float));
    if (N > 0) {
        BSPLAT_CUDA_TRY(cudaMemcpyAsync(d_means, means3d, (size_t)N * 3 * sizeof(float), cudaMemcpyHostToDevice, stream));
        BSPLAT_CUDA_TRY(cudaMemcpyAsync(d_scales, log_scales, (size_t)N * 3 * sizeof(float), cudaMemcpyHostToDevice, stream));
        BSPLAT_CUDA_TRY(cudaMemcpyAsync(d_quats, quats, (size_t)N * 4 * sizeof(float), cudaMemcpyHostToDevice, stream));
        BSPLAT_CUDA_TRY(cudaMemcpyAsync(d_opac, opacities, (size_t)N * sizeof(float), cudaMemcpyHostToDevice, stream));
        BSPLAT_CUDA_TRY(cudaMemcpyAsync(d_colors, colors, (size_t)N * channels * sizeof(float), cudaMemcpyHostToDevice, stream));
    }
    BSPLAT_CUDA_TRY(cudaMemcpyAsync(d_bg, background, (size_t)channels * sizeof(float), cudaMemcpyHostToDevice, stream));
    int rc = bsplat_render_fwd(N, d_means, d_scales, d_quats, d_opac, d_colors, channels, cam, d_bg, tile_size,
                               semantics, flags, d_image, workspace, workspace_bytes, needed_bytes, aux, stream);
    if (rc != BSPLAT_OK) return rc;
    BSPLAT_CUDA_TRY(cudaMemcpyAsync(image_host, d_image, (size_t)W * H * channels * sizeof(float),
                                    cudaMemcpyDeviceToHost, stream));
    BSPLAT_CUDA_TRY(cudaStreamSynchronize(stream));
    return BSPLAT_OK;
}
