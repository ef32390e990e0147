// bflk_api.cu -- the C ABI declared in include/bflk.h: host-side logic + kernel dispatch.
//
// Host work kept here on purpose (it is O(D) or O(C), one-time, and needs libm in double exactly like
// the reference): the direction grid of MIMOWorker::computeDelayLUT (src/dsp/mimo.cpp:20-43), the
// rotation-matrix entries of rotateZ / rotateY (src/geometry/geometry.cpp:219-233), create_antenna
// (src/geometry/antenna.cpp:60-87) and the median gate of AWProcessingUnit::calibrate
// (src/aw_processing_unit/aw_processing_unit.cpp:148-200).  Everything O(D*C) or larger runs on the GPU.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>

#include "bflk_internal.h"

using namespace bflk;

static thread_local std::string g_create_error;

static int create_fail(int code, const std::string &msg) {
    g_create_error = msg;
    return code;
}

bflk_handle::~bflk_handle() {
    for (const Stream *s : {&stream, &copy_stream, &lane[0], &lane[1]}) s->sync();
    comm_release(this);
}

extern "C" {

int bflk_version(void) { return BFLK_VERSION; }

void bflk_default_config(bflk_config *cfg) {
    if (!cfg) return;
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->n_channels = 64;
    cfg->frame_len = 256;
    cfg->history = 256;
    cfg->window_len = 1024;
    cfg->sample_rate = 48828.0;
    cfg->propagation_speed = 340.0;
    cfg->device = 0;
}

const char *bflk_last_error(const bflk_handle *h) { return h ? h->error.c_str() : g_create_error.c_str(); }

int bflk_create(const bflk_config *cfg, bflk_handle **out) {
    if (!cfg || !out) return create_fail(BFLK_ERR_INVALID, "bflk_create: null argument");
    *out = nullptr;
    if (cfg->n_channels <= 0 || cfg->frame_len < 3 || cfg->history < 0 || cfg->window_len < cfg->frame_len + 1 ||
        !(cfg->sample_rate > 0) || !(cfg->propagation_speed > 0))
        return create_fail(BFLK_ERR_INVALID, "bflk_create: invalid configuration");
    if (cfg->history + cfg->frame_len + 1 > cfg->window_len)
        return create_fail(BFLK_ERR_INVALID, "bflk_create: window_len must be >= history + frame_len + 1");
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev <= 0)
        return create_fail(BFLK_ERR_NO_DEVICE, std::string("bflk_create: no CUDA device (") + cudaGetErrorString(e) +
                                                   "); this library has no CPU fallback");
    if (cfg->device < 0 || cfg->device >= n_dev) return create_fail(BFLK_ERR_INVALID, "bflk_create: device ordinal out of range");
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, cfg->device)) != cudaSuccess)
        return create_fail(BFLK_ERR_CUDA, std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e));
    if (prop.major != 10)
        return create_fail(BFLK_ERR_NO_DEVICE, "bflk_create: device is not sm_100 (kernels are built for sm_100a only)");
    if ((e = cudaSetDevice(cfg->device)) != cudaSuccess)
        return create_fail(BFLK_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    cudaGetLastError();   // clear an earlier call's error: the check below is about the handle's streams and events
    std::unique_ptr<bflk_handle> h(new bflk_handle());
    if ((e = cudaGetLastError()) != cudaSuccess)
        return create_fail(BFLK_ERR_CUDA, std::string("bflk_create: cannot create the streams and events: ") + cudaGetErrorString(e));
    h->cfg = *cfg;
    h->sm_count = prop.multiProcessorCount;
    // tuning knobs: read once here, never on a call path (a worker thread calls bflk_power_map every 5 ms)
    auto env_int = [](const char *name, int dflt) { const char *v = getenv(name); return v && *v ? atoi(v) : dflt; };
    h->tuning.tile_nch = env_int("BFLK_TILE_NCH", 0);
    h->tuning.tile_warps = env_int("BFLK_TILE_WARPS", 0);
    h->tuning.tile_stages = env_int("BFLK_TILE_STAGES", 0);
    h->tuning.tile_pairs = env_int("BFLK_TILE_PAIRS", 0);
    h->tuning.tile_mode = env_int("BFLK_TILE_MODE", -1);
    h->tuning.no_ksplit = env_int("BFLK_NO_KSPLIT", 0);
    h->tuning.lat_warps = env_int("BFLK_LAT_WARPS", 0);
    h->tuning.lat_split = env_int("BFLK_LAT_SPLIT", 0);
    h->tuning.chunk_mib = env_int("BFLK_CHUNK_MIB", 0);
    *out = h.release();
    return BFLK_OK;
}

int bflk_destroy(bflk_handle *h) {
    if (!h) return BFLK_ERR_INVALID;
    cudaSetDevice(h->cfg.device);
    delete h;
    return BFLK_OK;
}

// ---- geometry -----------------------------------------------------------------------------------------
static void invalidate_tables(bflk_handle *h) {
    h->have_grid = false;
    h->drop_kernel_tables();
    h->n_dir = 0;
    h->dir_first = h->dir_count = 0;
    h->last_map_on_device = false;
}

int bflk_set_geometry(bflk_handle *h, const float *xyz, int32_t n_channels) {
    if (!h) return BFLK_ERR_INVALID;
    if (!xyz || n_channels != h->cfg.n_channels)
        return h->fail(BFLK_ERR_INVALID, "bflk_set_geometry: expected %d channels, got %d", h->cfg.n_channels, n_channels);
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    h->xyz.assign(xyz, xyz + 3 * (size_t)n_channels);
    h->max_radius = 0.0;
    for (int c = 0; c < n_channels; c++) {
        const double x = xyz[3 * c], y = xyz[3 * c + 1], z = xyz[3 * c + 2];
        h->max_radius = std::max(h->max_radius, std::sqrt((x * x + y * y) + z * z));
    }
    BFLK_CUDA(h, h->d_xyz.reserve(3 * (size_t)n_channels));
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_xyz.p, h->xyz.data(), h->xyz.size() * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    h->have_geometry = true;
    invalidate_tables(h);
    if (h->index.empty()) return bflk_set_channel_mask(h, nullptr, 0);
    return BFLK_OK;
}

int bflk_set_tiled_geometry(bflk_handle *h, int32_t n_tiles, const float *origins) {
    if (!h) return BFLK_ERR_INVALID;
    if (n_tiles <= 0 || !origins || n_tiles * 64 != h->cfg.n_channels)
        return h->fail(BFLK_ERR_INVALID, "bflk_set_tiled_geometry: n_tiles*64 must equal n_channels (%d)", h->cfg.n_channels);
    // create_antenna(position, COLUMNS = 8, ROWS = 8, DISTANCE = 0.02f), antenna.cpp:60-76
    const int columns = 8, rows = 8;
    const float distance = 0.02f;
    const float half = distance / 2;
    std::vector<float> xyz(3 * (size_t)h->cfg.n_channels);
    for (int a = 0; a < n_tiles; a++) {
        int i = 0;
        for (int r = 0; r < rows; r++)
            for (int c = 0; c < columns; c++, i++) {
                float *p = &xyz[3 * ((size_t)a * 64 + i)];
                p[0] = (static_cast<float>(c) * distance - rows * half + half) + origins[3 * a + 0];
                p[1] = (static_cast<float>(r) * distance - columns * half + half) + origins[3 * a + 1];
                p[2] = 0.f + origins[3 * a + 2];
            }
    }
    return bflk_set_geometry(h, xyz.data(), h->cfg.n_channels);
}

int bflk_get_geometry(const bflk_handle *h, float *xyz) {
    if (!h || !xyz || !h->have_geometry) return BFLK_ERR_STATE;
    std::memcpy(xyz, h->xyz.data(), h->xyz.size() * sizeof(float));
    return BFLK_OK;
}

int bflk_set_channel_mask(bflk_handle *h, const int32_t *index, int32_t usable) {
    if (!h) return BFLK_ERR_INVALID;
    const int C = h->cfg.n_channels;
    std::vector<int32_t> idx;
    if (!index) {
        idx.resize(C);
        for (int c = 0; c < C; c++) idx[c] = c;
    } else {
        if (usable <= 0 || usable > C) return h->fail(BFLK_ERR_INVALID, "bflk_set_channel_mask: usable=%d out of range", usable);
        idx.assign(index, index + usable);
        for (int v : idx)
            if (v < 0 || v >= C) return h->fail(BFLK_ERR_INVALID, "bflk_set_channel_mask: channel %d out of range", v);
    }
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    h->index = idx;
    h->drop_kernel_tables();
    BFLK_CUDA(h, h->d_index.reserve(idx.size()));
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_index.p, h->index.data(), idx.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    return BFLK_OK;
}

// ---- steering tables ------------------------------------------------------------------------------------
static DirTrig make_trig(double theta, double phi) {
    // steer(): rotateY(-static_cast<float>(theta)) * (rotateZ(static_cast<float>(phi)) * points), antenna.cpp:103
    const float az = static_cast<float>(phi);
    const float ay = -static_cast<float>(theta);
    DirTrig t;
    t.cz = static_cast<float>(std::cos((double)az));
    t.sz = static_cast<float>(std::sin((double)az));
    t.cy = static_cast<float>(std::cos((double)ay));
    t.sy = static_cast<float>(std::sin((double)ay));
    return t;
}

static float delay_scale(const bflk_handle *h) { return (float)(h->cfg.sample_rate / h->cfg.propagation_speed); }

// Runs the device table kernel for n directions, focused at `focus` (0: far field); results land in d_off/d_frac;
// *max_delay updated.
static int run_steer_tables(bflk_handle *h, const double *theta, const double *phi, int n, int32_t *d_off, float *d_frac,
                            int32_t *max_delay, double focus) {
    BFLK_CUDA(h, h->p_trig.reserve(n));
    BFLK_CUDA(h, h->d_trig.reserve(n));
    BFLK_CUDA(h, h->d_misc.reserve(4));
    BFLK_CUDA(h, h->p_misc.reserve(4));
    for (int i = 0; i < n; i++) h->p_trig.p[i] = make_trig(theta[i], phi[i]);
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_trig.p, h->p_trig.p, n * sizeof(DirTrig), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, cudaMemsetAsync(h->d_misc.p, 0, 4 * sizeof(int32_t), h->stream));
    BFLK_CUDA(h, launch_steer_tables(h->d_trig.p, n, h->d_xyz.p, h->cfg.n_channels, delay_scale(h), h->cfg.history, d_off,
                                     d_frac, h->d_misc.p, focus, h->stream));
    h->launches++;
    BFLK_CUDA(h, cudaMemcpyAsync(h->p_misc.p, h->d_misc.p, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    *max_delay = h->p_misc.p[0];
    return BFLK_OK;
}

static int check_delay_range(bflk_handle *h, int max_delay, const char *who) {
    if (max_delay > h->cfg.history)
        return h->fail(BFLK_ERR_RANGE, "%s: largest delay %d samples exceeds history %d", who, max_delay, h->cfg.history);
    return BFLK_OK;
}

// A focus point must lie outside the array: every element nearer to the origin than `focus` (0: far field, always fine).
static int check_focus(bflk_handle *h, double focus, const char *who) {
    if (focus > 0.0 && h->have_geometry && !(focus > h->max_radius))
        return h->fail(BFLK_ERR_INVALID, "%s: focus distance %g m is not beyond the array (an element lies %g m from the origin)",
                       who, focus, h->max_radius);
    return BFLK_OK;
}

int bflk_set_grid_fov(bflk_handle *h, int32_t rows, int32_t cols, float fov_deg) {
    if (!h) return BFLK_ERR_INVALID;
    if (!h->have_geometry) return h->fail(BFLK_ERR_STATE, "bflk_set_grid_fov: set the geometry first");
    if (rows <= 0 || cols <= 0 || !(fov_deg > 0.f) || fov_deg > 180.f)
        return h->fail(BFLK_ERR_INVALID, "bflk_set_grid_fov: invalid grid %d x %d fov %g", rows, cols, (double)fov_deg);
    if (int rc = check_focus(h, h->focus, "bflk_set_grid_fov")) return rc;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const int D = rows * cols;
    std::vector<double> theta(D), phi(D);
    // MIMOWorker::computeDelayLUT grid, mimo.cpp:21-43 (all double)
    const double fovRadian = (double)fov_deg * (M_PI / 180.0);
    const double separationRows = std::sin(fovRadian / 2.0) / (static_cast<double>(rows) / 2.0);
    const double separationColumns = std::sin(fovRadian / 2.0) / (static_cast<double>(cols) / 2.0);
    int k = 0;
    for (int r = 0; r < rows; r++) {
        for (int c = 0; c < cols; c++, k++) {
            double y = static_cast<double>(r) * separationRows - static_cast<double>(rows) * separationRows / 2.0 + separationRows / 2.0;
            double x = static_cast<double>(c) * separationColumns - static_cast<double>(cols) * separationColumns / 2.0 + separationColumns / 2.0;
            double norm = std::sqrt(std::pow(x, 2) + std::pow(y, 2));
            if (norm == 0.0) {  // centre cell of an odd grid: the reference divides by zero; defined as boresight
                theta[k] = 0.0;
                phi[k] = 0.0;
                continue;
            }
            x /= norm;
            y /= norm;
            if (norm > 1.0) norm = 1.0;
            theta[k] = std::asin(norm);
            phi[k] = std::atan2(y, x);
        }
    }
    const size_t DC = (size_t)D * h->cfg.n_channels;
    BFLK_CUDA(h, h->d_off.reserve(DC));
    BFLK_CUDA(h, h->d_frac.reserve(DC));
    int32_t max_delay = 0;
    int rc = run_steer_tables(h, theta.data(), phi.data(), D, h->d_off.p, h->d_frac.p, &max_delay, h->focus);
    if (rc) return rc;
    invalidate_tables(h);
    if ((rc = check_delay_range(h, max_delay, "bflk_set_grid_fov"))) return rc;
    // the angles of the Targets records, on the device
    BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));   // a caller's stream may still read the old ones
    BFLK_CUDA(h, h->d_theta.reserve(D));
    BFLK_CUDA(h, h->d_phi.reserve(D));
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_theta.p, theta.data(), D * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_phi.p, phi.data(), D * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    h->theta.swap(theta);
    h->phi.swap(phi);
    h->rows = rows;
    h->cols = cols;
    h->n_dir = D;
    h->dir_first = 0;
    h->dir_count = D;
    h->max_delay = max_delay;
    h->have_grid = true;
    return BFLK_OK;
}

int bflk_set_grid_tables(bflk_handle *h, const int32_t *offsets, const float *fractions, int32_t n_directions) {
    if (!h) return BFLK_ERR_INVALID;
    if (!offsets || !fractions || n_directions <= 0) return h->fail(BFLK_ERR_INVALID, "bflk_set_grid_tables: null / empty tables");
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const size_t DC = (size_t)n_directions * h->cfg.n_channels;
    BFLK_CUDA(h, h->d_off.reserve(DC));
    BFLK_CUDA(h, h->d_frac.reserve(DC));
    BFLK_CUDA(h, h->d_misc.reserve(4));
    BFLK_CUDA(h, h->p_misc.reserve(4));
    invalidate_tables(h);
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_off.p, offsets, DC * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_frac.p, fractions, DC * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    h->p_misc.p[0] = INT32_MIN;
    h->p_misc.p[1] = INT32_MAX;
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_misc.p, h->p_misc.p, 2 * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, launch_offset_range(h->d_off.p, DC, h->d_misc.p, h->d_misc.p + 1, h->stream));
    h->launches++;
    BFLK_CUDA(h, cudaMemcpyAsync(h->p_misc.p, h->d_misc.p, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    const int max_off = h->p_misc.p[0], min_off = h->p_misc.p[1];
    if (min_off < 0 || max_off > h->cfg.history)
        return h->fail(BFLK_ERR_RANGE, "bflk_set_grid_tables: offsets must lie in [0, history = %d]; got [%d, %d]",
                       h->cfg.history, min_off, max_off);
    const int max_delay = h->cfg.history - min_off;
    h->theta.clear();   // no angles: the Targets calls refuse these tables
    h->phi.clear();
    h->rows = h->cols = 0;
    h->n_dir = n_directions;
    h->dir_first = 0;
    h->dir_count = n_directions;
    h->max_delay = max_delay;
    h->have_grid = true;
    return BFLK_OK;
}

int bflk_set_grid_shape(bflk_handle *h, int32_t rows, int32_t cols) {
    if (!h) return BFLK_ERR_INVALID;
    if (!h->have_grid) return h->fail(BFLK_ERR_STATE, "bflk_set_grid_shape: set the tables first");
    if (rows <= 0 || cols <= 0 || (int64_t)rows * cols != h->n_dir)
        return h->fail(BFLK_ERR_INVALID, "bflk_set_grid_shape: %d x %d is not the %d directions of the tables", rows, cols, h->n_dir);
    h->rows = rows;
    h->cols = cols;
    h->drop_kernel_tables();
    return BFLK_OK;
}

int bflk_set_direction_range(bflk_handle *h, int32_t first, int32_t count) {
    if (!h) return BFLK_ERR_INVALID;
    if (!h->have_grid) return h->fail(BFLK_ERR_STATE, "bflk_set_direction_range: set the grid first");
    if (first < 0 || count <= 0 || first + count > h->n_dir)
        return h->fail(BFLK_ERR_INVALID, "bflk_set_direction_range: [%d, %d) outside grid of %d", first, first + count, h->n_dir);
    h->dir_first = first;
    h->dir_count = count;
    h->drop_kernel_tables();
    h->last_map_on_device = false;   // the map left on the device covers the old range
    return BFLK_OK;
}

int bflk_get_n_directions(const bflk_handle *h, int32_t *total, int32_t *first, int32_t *count) {
    if (!h || !h->have_grid) return BFLK_ERR_STATE;
    if (total) *total = h->n_dir;
    if (first) *first = h->dir_first;
    if (count) *count = h->dir_count;
    return BFLK_OK;
}

int bflk_get_grid(const bflk_handle *h, double *theta, double *phi) {
    if (!h || !h->have_grid || h->theta.empty()) return BFLK_ERR_STATE;
    if (theta) std::memcpy(theta, h->theta.data(), h->theta.size() * sizeof(double));
    if (phi) std::memcpy(phi, h->phi.data(), h->phi.size() * sizeof(double));
    return BFLK_OK;
}

int bflk_get_tables(const bflk_handle *hc, int32_t *offsets, float *fractions) {
    bflk_handle *h = const_cast<bflk_handle *>(hc);
    if (!h) return BFLK_ERR_INVALID;
    if (!h->have_grid) return h->fail(BFLK_ERR_STATE, "bflk_get_tables: no grid");
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const size_t DC = (size_t)h->n_dir * h->cfg.n_channels;
    if (offsets) BFLK_CUDA(h, cudaMemcpyAsync(offsets, h->d_off.p, DC * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (fractions) BFLK_CUDA(h, cudaMemcpyAsync(fractions, h->d_frac.p, DC * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    return BFLK_OK;
}

int bflk_steer_tables(bflk_handle *h, const double *theta, const double *phi, int32_t n_targets, int32_t *offsets,
                      float *fractions) {
    if (!h) return BFLK_ERR_INVALID;
    if (!h->have_geometry) return h->fail(BFLK_ERR_STATE, "bflk_steer_tables: set the geometry first");
    if (!theta || !phi || n_targets <= 0) return h->fail(BFLK_ERR_INVALID, "bflk_steer_tables: null / empty direction list");
    if (int rc = check_focus(h, h->focus, "bflk_steer_tables")) return rc;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const size_t TC = (size_t)n_targets * h->cfg.n_channels;
    BFLK_CUDA(h, h->d_soff.reserve(TC));
    BFLK_CUDA(h, h->d_sfrac.reserve(TC));
    int32_t max_delay = 0;
    int rc = run_steer_tables(h, theta, phi, n_targets, h->d_soff.p, h->d_sfrac.p, &max_delay, h->focus);
    if (rc) return rc;
    if (offsets) BFLK_CUDA(h, cudaMemcpyAsync(offsets, h->d_soff.p, TC * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (fractions) BFLK_CUDA(h, cudaMemcpyAsync(fractions, h->d_sfrac.p, TC * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    return check_delay_range(h, max_delay, "bflk_steer_tables");
}

int bflk_set_focus(bflk_handle *h, double distance_m) {
    if (!h) return BFLK_ERR_INVALID;
    if (!(distance_m >= 0.0) || std::isinf(distance_m))
        return h->fail(BFLK_ERR_INVALID, "bflk_set_focus: distance %g m (0 = far field, else a finite distance)", distance_m);
    if (int rc = check_focus(h, distance_m, "bflk_set_focus")) return rc;
    if (h->have_grid && !h->theta.empty()) {
        // a bflk_set_grid_fov grid: its tables again, at the new focus, built aside so that a refusal leaves the old ones
        BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
        const size_t DC = (size_t)h->n_dir * h->cfg.n_channels;
        DevBuf<int32_t> off;
        DevBuf<float> frac;
        BFLK_CUDA(h, off.reserve(DC));
        BFLK_CUDA(h, frac.reserve(DC));
        int32_t max_delay = 0;
        int rc = run_steer_tables(h, h->theta.data(), h->phi.data(), h->n_dir, off.p, frac.p, &max_delay, distance_m);
        if (rc) return rc;
        if ((rc = check_delay_range(h, max_delay, "bflk_set_focus"))) return rc;
        BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));   // a caller's stream may still read the old tables
        std::swap(h->d_off, off);
        std::swap(h->d_frac, frac);
        h->max_delay = max_delay;
        h->drop_kernel_tables();
        h->last_map_on_device = false;
    }
    h->focus = distance_m;
    return BFLK_OK;
}

// ---- power map ---------------------------------------------------------------------------------------------
int bflk_set_kernel(bflk_handle *h, int32_t which) {
    if (!h) return BFLK_ERR_INVALID;
    if (which < kAuto || which > kTiledFma2) return h->fail(BFLK_ERR_INVALID, "bflk_set_kernel: %d", which);
    h->kernel_choice = (Kernel)which;
    return BFLK_OK;
}

int bflk_set_channel_split(bflk_handle *h, int32_t on) {
    if (!h) return BFLK_ERR_INVALID;
    h->allow_ksplit = on != 0;
    return BFLK_OK;
}

int bflk_launch_shape(int32_t rows, int32_t cols, int32_t n_channels, int32_t frame_len, int32_t n_frames, int32_t n_sms,
                      int32_t channel_split, int32_t *warps, int32_t *split) {
    if (rows <= 0 || cols <= 0 || n_channels <= 0 || frame_len < 256 || n_frames <= 0 || n_sms <= 0 || !warps || !split) return BFLK_ERR_INVALID;
    int w = 0, sp = 1;
    bflk::latency_shape((long long)((rows + 1) / 2) * ((cols + 1) / 2), n_frames, frame_len, n_channels,
                        block_pairs_per_cta(0, n_channels), n_sms, channel_split != 0, &w, &sp);
    *warps = w;
    *split = sp;
    return BFLK_OK;
}

int64_t bflk_launch_count(const bflk_handle *h) { return h ? h->launches : 0; }

int bflk_get_kernel(const bflk_handle *h, int32_t *last_used, int32_t *tile_span, int32_t *window_chunks) {
    if (!h) return BFLK_ERR_INVALID;
    if (last_used) *last_used = h->kernel_last;
    if (tile_span) *tile_span = h->tiles.valid ? h->tiles.smax : -1;
    if (window_chunks) *window_chunks = (h->tiles.valid && h->tiles.usable) ? h->tiles.geom.nch : 0;
    return BFLK_OK;
}

static void timing_hook(void *ctx, int kind, bool begin, cudaStream_t st) {
    bflk_handle *h = static_cast<bflk_handle *>(ctx);
    if (!h->timing) return;
    if (begin) {
        h->timed.emplace_back();
        h->timed.back().kind = kind;
        cudaEventRecord(h->timed.back().e0, st);
    } else if (!h->timed.empty()) {
        cudaEventRecord(h->timed.back().e1, st);
    }
}

int bflk_fp32_peak_tflops(bflk_handle *h, float *tflops) {
    if (!h || !tflops) return BFLK_ERR_INVALID;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const int blocks = h->sm_count, iters = 8192;
    DevBuf<float> d_out;
    BFLK_CUDA(h, d_out.reserve((size_t)blocks * 512));
    Event e0(cudaEventDefault), e1(cudaEventDefault);
    if (!e0 || !e1) return h->fail(BFLK_ERR_CUDA, "bflk_fp32_peak_tflops: cannot create events: %s", cudaGetErrorString(cudaGetLastError()));
    float best = 0.f;
    for (int rep = 0; rep < 4; rep++) {   // first launch warms up; best of the rest
        BFLK_CUDA(h, cudaEventRecord(e0, h->stream));
        BFLK_CUDA(h, launch_ffma2_peak(d_out.p, blocks, iters, h->stream));
        BFLK_CUDA(h, cudaEventRecord(e1, h->stream));
        BFLK_CUDA(h, cudaEventSynchronize(e1));
        float ms = 0.f;
        BFLK_CUDA(h, cudaEventElapsedTime(&ms, e0, e1));
        h->launches++;
        const double flop = (double)blocks * 512 * iters * 16 * 4;   // a packed FMA = 2 lanes x 2 FLOP
        if (rep > 0) best = std::max(best, (float)(flop / (ms * 1e-3) / 1e12));
    }
    *tflops = best;
    return BFLK_OK;
}

int bflk_enable_timing(bflk_handle *h, int32_t on) {
    if (!h) return BFLK_ERR_INVALID;
    h->timing = on != 0;
    return BFLK_OK;
}

int bflk_kernel_time_ms(bflk_handle *h, float *das_ms, int32_t *das_launches, float *pack_ms, int32_t *pack_launches) {
    if (!h) return BFLK_ERR_INVALID;
    float ms[2] = {0.f, 0.f};
    int32_t n[2] = {0, 0};
    for (auto &t : h->timed) {
        float v = 0.f;
        BFLK_CUDA(h, cudaEventSynchronize(t.e1));
        BFLK_CUDA(h, cudaEventElapsedTime(&v, t.e0, t.e1));
        ms[t.kind] += v;
        n[t.kind]++;
    }
    h->timed.clear();
    if (das_ms) *das_ms = ms[0];
    if (das_launches) *das_launches = n[0];
    if (pack_ms) *pack_ms = ms[1];
    if (pack_launches) *pack_launches = n[1];
    return BFLK_OK;
}

}  // extern "C"

namespace bflk {

static int64_t min_stream_samples(const bflk_handle *h, int n_frames) {
    return (int64_t)(n_frames - 1) * h->cfg.frame_len + h->cfg.history + h->cfg.frame_len + 1;
}

int check_frames(bflk_handle *h, int64_t n_samples, int n_frames, const char *who) {
    const int64_t need = min_stream_samples(h, n_frames);
    if (n_samples < need)
        return h->fail(BFLK_ERR_INVALID, "%s: %lld samples per channel cannot hold %d frames (need %lld)", who, (long long)n_samples, n_frames, (long long)need);
    if (h->fir_phases > 0 && n_samples < need + h->fir_taps - 2)
        return h->fail(BFLK_ERR_INVALID, "%s: the FIR reads %d samples past a frame's last tap", who, h->fir_taps - 2);
    return BFLK_OK;
}

// 2x2 direction tiles of the handle's direction range (whole rows of the grid; the first is even)
static int tile_count(const bflk_handle *h) {
    const int row0 = (h->dir_first / h->cols) & ~1;
    const int row1 = (h->dir_first + h->dir_count - 1) / h->cols;  // inclusive
    return ((row1 - row0) / 2 + 1) * ((h->cols + 1) / 2);
}

// Builds (once per grid / mask / range) the packed tables of the register-tiled kernel.  tiles.valid is set only after
// the last step has succeeded, so a failed build is retried (and reported again) by the next call.
static int ensure_tiles(bflk_handle *h, int fast, int want_warps) {
    bflk_handle::TileTables &t = h->tiles;
    if (t.valid && t.fast == fast && t.want_warps == want_warps) return BFLK_OK;
    BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));   // a queued kernel may still read the old tables
    t.valid = false;
    t.fast = fast;
    t.want_warps = want_warps;
    t.usable = false;
    if (h->rows <= 0 || h->cols <= 0) {  // caller-supplied LUT without a declared grid shape: nothing to tile
        t.valid = true;
        return BFLK_OK;
    }
    const int cols = h->cols;
    const int n_tiles = tile_count(h);
    const int usable = (int)h->index.size();
    BFLK_CUDA(h, t.d_dirs.reserve((size_t)n_tiles * 4));
    BFLK_CUDA(h, h->d_misc.reserve(4));
    BFLK_CUDA(h, h->p_misc.reserve(4));
    const int stage_off = das_tile_geometry(h->cfg.history, h->max_delay, 0).stage_off;
    // pass 1: largest offset spread per tiling mode -> which kernel variant (window chunks, warps per CTA).
    // mode 0 shares one window among the 2x2 tile; modes 1 / 2 share one window per direction pair (coarse grids).
    BFLK_CUDA(h, cudaMemsetAsync(h->d_misc.p, 0, 4 * sizeof(int32_t), h->stream));
    for (int mode = 0; mode < 3; mode++) {
        BFLK_CUDA(h, launch_build_tiles(h->d_off.p, h->d_frac.p, h->cfg.n_channels, h->d_index.p, usable, h->rows, cols,
                                        h->dir_first, h->dir_count, stage_off, 0, 1, mode, -1, 0, nullptr, nullptr, n_tiles,
                                        h->d_misc.p, h->stream));
        h->launches++;
    }
    BFLK_CUDA(h, cudaMemcpyAsync(h->p_misc.p, h->d_misc.p, 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    const int span0 = h->p_misc.p[0], span1 = h->p_misc.p[1], span2 = h->p_misc.p[2];
    // one shared window while the 2x2 spread fits the 6- or 8-chunk variant; beyond that (coarse grid, long array) the
    // direction pairs along the array's short axis still fit a 6- / 7-chunk window each: measured faster than one wide
    // window (fewer dispatch cases, smaller code, more resident warps; two-FMA form: cfg2 0.576 vs 0.568, cfg3 0.539 vs
    // 0.455 of the FP32 peak)
    int mode = 0;
    const int pair_span = std::min(span1, span2), pair_mode = span1 <= span2 ? 1 : 2;
    if (span0 > 3 && pair_span <= 3) mode = pair_mode;        // two 6-chunk windows, 16 warps
    else if (span0 > 7 && pair_span <= 5) mode = pair_mode;   // two 7-chunk windows instead of one 10-chunk window
    const int forced = h->tuning.tile_mode;
    if (forced == 0 || ((forced == 1 || forced == 2) && h->p_misc.p[forced] <= 5)) mode = forced;
    t.n_tiles = n_tiles;
    t.smax = h->p_misc.p[mode];
    t.geom = das_tile_geometry(h->cfg.history, h->max_delay, t.smax, n_tiles, mode, fast, &h->tuning, want_warps);
    // usable: the spread fits a compiled variant, frames are whole blocks, AND the stage ring of some CTA shape fits
    // shared memory (packed rows grow with the largest delay: long arrays fall through to the other kernels)
    t.usable = t.smax <= das_tile_max_span() && h->cfg.frame_len >= 256 && h->cfg.frame_len % 2 == 0 && t.geom.stages >= 3;
    if (!t.usable) {
        t.valid = true;
        return BFLK_OK;
    }
    // pass 2: the packed per-(tile, channel) entries, grouped for that variant's CTA shape
    const size_t entries = tile_table_entries(n_tiles, usable, t.geom.warps);
    const size_t ent_bytes = das_tile_entry_bytes(t.geom);
    BFLK_CUDA(h, t.d_tiles.reserve(entries * ent_bytes));
    BFLK_CUDA(h, cudaMemsetAsync(t.d_tiles.p, 0, entries * ent_bytes, h->stream));
    BFLK_CUDA(h, launch_build_tiles(h->d_off.p, h->d_frac.p, h->cfg.n_channels, h->d_index.p, usable, h->rows, cols,
                                    h->dir_first, h->dir_count, stage_off, t.geom.copy_bytes, t.geom.warps, mode,
                                    2 * t.geom.nch - 9, fast, t.d_tiles.p, t.d_dirs.p, n_tiles, h->d_misc.p, h->stream));
    h->launches++;
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    t.valid = true;
    return BFLK_OK;
}

// Builds (once per grid / mask / range) the direction tiles and per-lane tables of the lane-broadcast kernel.
static int ensure_bcast(bflk_handle *h) {
    if (h->bcast.valid) return BFLK_OK;
    BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));   // a queued kernel may still read the old tables
    const int first = h->dir_first, count = h->dir_count;
    std::vector<int32_t> globals;
    if (h->rows > 0 && h->cols > 0) {
        // 32 directions per tile; the narrow tile side runs along the array's longer axis, where
        // neighbouring directions differ most in delay
        float minx = 1e30f, maxx = -1e30f, miny = 1e30f, maxy = -1e30f;
        for (size_t c = 0; c < h->xyz.size() / 3; c++) {
            minx = std::min(minx, h->xyz[3 * c]); maxx = std::max(maxx, h->xyz[3 * c]);
            miny = std::min(miny, h->xyz[3 * c + 1]); maxy = std::max(maxy, h->xyz[3 * c + 1]);
        }
        const int TR = (maxx - minx >= maxy - miny) ? 8 : 4, TC = 32 / TR;
        const int cols = h->cols, r0 = first / cols, r1 = (first + count - 1) / cols;
        for (int r = r0; r <= r1; r += TR)
            for (int c = 0; c < cols; c += TC) {
                int32_t t[32];
                bool any = false;
                for (int q = 0; q < 32; q++) {
                    const int rr = r + q / TC, cc = c + q % TC;
                    const int g = (rr < h->rows && cc < cols) ? rr * cols + cc : -1;
                    t[q] = (g >= first && g < first + count) ? g : -1;
                    any |= t[q] >= 0;
                }
                if (!any) continue;
                std::stable_partition(t, t + 32, [](int32_t v) { return v >= 0; });  // valid directions first
                globals.insert(globals.end(), t, t + 32);
            }
    } else {
        for (int g0 = first; g0 < first + count; g0 += 32)
            for (int q = 0; q < 32; q++) globals.push_back(g0 + q < first + count ? g0 + q : -1);
    }
    const int n_tiles = (int)(globals.size() / 32);
    std::vector<int32_t> locals(globals.size());
    for (size_t i = 0; i < globals.size(); i++) locals[i] = globals[i] >= 0 ? globals[i] - first : -1;
    const int usable = (int)h->index.size();
    h->bcast.geom = das_bcast_geometry(h->cfg.history, h->max_delay);
    BFLK_CUDA(h, h->bcast.d_globals.reserve(globals.size()));
    BFLK_CUDA(h, h->bcast.d_dirs.reserve(globals.size()));
    BFLK_CUDA(h, h->bcast.d_table.reserve(das_bcast_table_entries(n_tiles, usable)));
    BFLK_CUDA(h, cudaMemcpyAsync(h->bcast.d_globals.p, globals.data(), globals.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, cudaMemcpyAsync(h->bcast.d_dirs.p, locals.data(), locals.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, launch_bcast_table(h->d_off.p, h->d_frac.p, h->cfg.n_channels, h->d_index.p, usable, h->bcast.d_globals.p,
                                    n_tiles, h->bcast.geom, h->bcast.d_table.p, h->stream));
    h->launches++;
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));  // the host vectors above go out of scope
    h->bcast.n_tiles = n_tiles;
    h->bcast.valid = true;
    return BFLK_OK;
}

}  // namespace bflk

// CTA shape of a call that cannot fill two waves of 16-warp CTAs (a live worker's single frame).  One CTA per SM (the stage
// ring takes the shared memory), so the call takes waves x the time of one CTA = a fixed cost (launch, barrier set-up, first
// bulk copies, epilogue) + its channels x the time of a channel step, which depends on the warps that share a scheduler.
// The two-FMA variants can also split the channels of a block pair across a thread-block cluster of 2 or 4 CTAs (das_tile.cu,
// KSPLIT; opt-in, bflk_set_channel_split): the serial channel loop gets shorter by the cluster size for the price of the
// exchange.  Constants fitted to cfg3 / cfg2 / cfg1 single-frame launches on B200 (profiles/r2c_latency_shapes.txt): cycles
// per channel step with 1 / 2 / 3 / 4 / 5 warps per scheduler (a lone warp is bound by its own load -> FFMA2 -> branch
// latencies, four by the issue port); clusters of 8 are not used (16 warps x 8 ranks: 82 us where 16 x 4 takes 76 -- they
// do not all fit at once next to 200 KB of shared memory per CTA).
// Returns warps = 0 (throughput shape) for larger calls; otherwise the shape with the smallest estimate -- the larger CTA
// (fewer copies of the rows staged) on ties, no split unless it wins by 10 %.
void bflk::latency_shape(long long n_tiles, int n_frames, int frame_len, int usable, int pairs_per_cta, int sms, bool may_split,
                         int *warps, int *split) {
    *warps = 0;
    *split = 1;
    const long long pairs = ((long long)n_frames * blocks_per_frame(frame_len) + 1) / 2;
    const long long pair_ctas = (pairs + pairs_per_cta - 1) / pairs_per_cta;
    const int n_stage = (usable + kTileCC - 1) / kTileCC;
    if (((n_tiles + 15) / 16) * pair_ctas >= 2LL * sms) return;
    static const double step[6] = {0, 455, 538, 658, 880, 1100};
    const double fixed = 19650, exchange = 6000;
    double best_t = 0;
    for (int sp = 1; sp <= (may_split ? 4 : 1); sp *= 2) {
        if (sp > 1 && n_stage / sp < 4) break;
        for (int w = 16; w >= 2; w--) {
            const long long ctas = ((n_tiles + w - 1) / w) * pair_ctas * sp;
            const double chans = 8.0 * ((n_stage + sp - 1) / sp);
            const double t = (double)((ctas + sms - 1) / sms) * (chans * step[(w + 3) / 4] + fixed + (sp > 1 ? exchange : 0));
            if (!*warps || t < best_t * (sp > *split ? 0.9 : 1.0) - 1e-9) { *warps = w; *split = sp; best_t = t; }
        }
    }
    if (*warps == 16 && *split == 1) *warps = 0;
}

// *serve (serve may be null): the register-tiled kernels serve calls in the CTA shape of want_warps (0: throughput) from float
// rows row_stride apart, or from wire rows (rows = nullptr).  Builds their tables for it unless FIR or kernel 1 / 3 rule them out.
static int tiles_serve(bflk_handle *h, bool *serve, int want_warps = 0, const float *rows = nullptr, int64_t row_stride = 0) {
    const bool form_ok = h->fir_phases == 0 && h->kernel_choice != kGeneric && h->kernel_choice != kBcast;
    const int rc = form_ok ? ensure_tiles(h, h->kernel_choice != kTiledExact, want_warps) : BFLK_OK;
    // the tiled kernels pack float rows with 8-byte loads: an even row stride from an 8-byte aligned start
    if (serve) *serve = form_ok && rc == BFLK_OK && h->tiles.usable && (!rows || (!(row_stride & 1) && !((uintptr_t)rows & 7)));
    return rc;
}

int bflk::note_use(bflk_handle *h, cudaStream_t st, bool overlapped) {
    BFLK_CUDA(h, cudaEventRecord(h->caller_event, st));
    h->last_stream = st;
    h->caller_event_is_overlapped = overlapped;
    return BFLK_OK;
}

int bflk::lanes_fork(bflk_handle *h, cudaEvent_t after, int only) {
    // tables first (ensure_tiles synchronises the handle's stream when it has to build them), before anything is queued
    int rc = tiles_serve(h, nullptr);
    if (rc) return rc;
    const bool wait_caller = !(only >= 0 && h->caller_event_is_overlapped);
    for (int i = 0; i < 2; i++) {
        if (only >= 0 && i != only) continue;
        if (after) BFLK_CUDA(h, cudaStreamWaitEvent(h->lane[i], after, 0));
        if (wait_caller) BFLK_CUDA(h, cudaStreamWaitEvent(h->lane[i], h->caller_event, 0));
    }
    return BFLK_OK;
}

int bflk::lanes_join(bflk_handle *h, int only) {
    for (int i = 0; i < 2; i++) {
        if (only >= 0 && i != only) continue;
        BFLK_CUDA(h, cudaEventRecord(h->lane_done[i], h->lane[i]));
        BFLK_CUDA(h, cudaStreamWaitEvent(h->stream, h->lane_done[i], 0));
    }
    return note_use(h, h->stream, only >= 0);
}

// route: the kernel of a call of n_frames frames from launch.wire or float rows (stream_dev, row_stride), the tiled kernels'
// channel split (their warps are in the tables route builds), and whether wire samples go through ingest_kernel first.  A
// chosen kernel that cannot serve the call is refused with BFLK_ERR_STATE.
struct Route { Kernel kernel = kGeneric; int split = 1; bool ingest = false; };
static int route(bflk_handle *h, const float *stream_dev, int64_t row_stride, int n_frames, const Launch &launch, Route *r) {
    const int N = h->cfg.frame_len, usable = (int)h->index.size();
    const bool fir = h->fir_phases > 0;   // FIR interpolation runs through the generic kernel only
    if (fir && h->kernel_choice > kGeneric) return h->fail(BFLK_ERR_STATE, "bflk_power_map: FIR interpolation needs kernel 0 or 1");
    // automatic choice = the two-FMA variant (power within the 1e-4 bar); 2 asks for bit-identical delayed sums
    // a call with few block pairs cannot fill the SMs with 16-warp CTAs (one cfg3 frame: 16 CTAs, each walking 512
    // channels with four warps per scheduler): smaller CTAs trade per-SM efficiency for latency.  The shape is part of
    // the table layout, so a handle that alternates between single frames and large batches rebuilds its tables.
    int want_warps = 0, want_split = 1;
    if (h->rows > 0 && h->cols > 0 && h->tuning.tile_warps == 0)
        latency_shape(tile_count(h), n_frames, N, usable, block_pairs_per_cta(h->tuning.tile_pairs, usable), h->sm_count,
                      h->kernel_choice != kTiledExact && h->allow_ksplit && !h->tuning.no_ksplit, &want_warps, &want_split);
    if (want_warps > 0 && h->tuning.lat_warps >= 2 && h->tuning.lat_warps <= 16) want_warps = h->tuning.lat_warps;   // experiments
    if (want_warps > 0 && h->tuning.lat_split >= 1 && h->allow_ksplit) want_split = h->tuning.lat_split;
    if (launch.pipelined) { want_warps = 0; want_split = 1; }   // lanes_fork built the throughput-shape tables
    bool tiled;
    int rc = tiles_serve(h, &tiled, want_warps, launch.wire ? nullptr : stream_dev, row_stride);
    if (rc) return rc;
    if ((h->kernel_choice == kTiledExact || h->kernel_choice == kTiledFma2) && !tiled)
        return h->fail(BFLK_ERR_STATE, "bflk_power_map: the register-tiled kernel does not fit this grid (offset spread %d of at most %d, %d stage buffers fit shared memory)",
                       h->tiles.smax, das_tile_max_span(), h->tiles.geom.stages);
    const bool bcast_ok = N >= 256 && das_bcast_fits(das_bcast_geometry(h->cfg.history, h->max_delay));
    if (h->kernel_choice == kBcast && !bcast_ok)
        return h->fail(BFLK_ERR_STATE, "bflk_power_map: the lane-broadcast kernel needs frame_len >= 256 and a stage ring that fits shared memory");
    r->split = tiled && das_tile_ksplit_ok(h->tiles.geom, want_split) ? want_split : 1;
    r->ingest = launch.wire && !tiled;
    if (tiled) r->kernel = h->tiles.geom.fast ? kTiledFma2 : kTiledExact;
    else if (!fir && (h->kernel_choice == kAuto || h->kernel_choice == kBcast) && bcast_ok) r->kernel = kBcast;
    return r->kernel == kBcast ? ensure_bcast(h) : BFLK_OK;
}

int bflk::power_map_dev(bflk_handle *h, const float *stream_dev, int64_t row_stride, int64_t n_samples, int32_t n_frames,
                        float *power_dev, const Launch &launch, float *beams_dev) {
    if (!h) return BFLK_ERR_INVALID;
    if (!h->have_grid) return h->fail(BFLK_ERR_STATE, "bflk_power_map: set geometry and grid first");
    const int32_t *wire = launch.wire;   // wire-format call: stream_dev is null, the samples are wire[n_samples][C]
    if ((!stream_dev && !wire) || !power_dev || n_frames <= 0) return h->fail(BFLK_ERR_INVALID, "bflk_power_map: null buffer or no frames");
    int rc = check_frames(h, n_samples, n_frames, "bflk_power_map");
    if (rc) return rc;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = launch.st ? launch.st : h->stream;
    // the packed rows, partial sums and tables are the handle's: a call on another stream than the previous one waits for it
    if (!launch.pipelined && h->last_stream != st) BFLK_CUDA(h, cudaStreamWaitEvent(st, h->caller_event, 0));
    struct Mark {   // every exit after this point leaves an event behind on the stream the call used
        bflk_handle *h;
        cudaStream_t st;
        bool on;
        ~Mark() { if (on) note_use(h, st, false); }
    } mark{h, st, !launch.pipelined};
    DevBuf<char> &d_packed = h->scratch[launch.scratch].packed;
    DevBuf<float> &d_partial = h->scratch[launch.scratch].partial;
    const int N = h->cfg.frame_len, C = h->cfg.n_channels, usable = (int)h->index.size();
    const float norm = static_cast<float>(N * usable);  // power /= float(N_SAMPLES * count), mimo.cpp:137
    // automatic choice: register-tiled kernel when the grid tiles (2x2 direction tiles with small offset
    // spread), else the lane-broadcast kernel (any direction list), else the generic kernel (any frame length)
    Route r;
    if ((rc = route(h, stream_dev, row_stride, n_frames, launch, &r))) return rc;
    if (r.ingest) {
        // the other kernels read channel-major float rows: convert the wire samples first (ingest_kernel), then carry on
        BFLK_CUDA(h, h->d_window.reserve((size_t)C * (n_samples + 1)));
        BFLK_CUDA(h, launch_ingest(wire, n_samples, C, h->d_window.p, st));
        h->launches++;
        stream_dev = h->d_window.p;
        row_stride = n_samples;
    }
    if (r.kernel == kGeneric) {
        GenericArgs a{};
        a.stream = stream_dev;
        a.row_stride = row_stride;
        a.n_frames = n_frames;
        a.frame_len = N;
        a.frame_stride = N;
        a.off = h->d_off.p + (size_t)h->dir_first * C;
        a.frac = h->d_frac.p + (size_t)h->dir_first * C;
        a.C = C;
        a.index = h->d_index.p;
        a.usable = usable;
        a.n_dir = h->dir_count;
        a.power = power_dev;
        a.audio = beams_dev;
        a.norm = norm;
        if (h->fir_phases > 0) { a.fir = h->d_fir.p; a.fir_phases = h->fir_phases; a.fir_taps = h->fir_taps; }
        timing_hook(h, 0, true, st);
        BFLK_CUDA(h, launch_das_generic(a, st));
        timing_hook(h, 0, false, st);
        h->launches++;
        h->kernel_last = r.kernel;
        return BFLK_OK;
    }
    // the staged kernels: pack pre-pass, delay-and-sum, and for frames longer than one block finalize_kernel
    FrameArgs f;
    f.stream = stream_dev;
    f.row_stride = row_stride;
    f.row_len = n_samples;
    f.n_frames = n_frames;
    f.frame_len = N;
    f.frame_stride = N;
    f.usable = usable;
    f.n_dir = h->dir_count;
    f.index = h->d_index.p;
    f.power = power_dev;
    f.beams = beams_dev;
    f.norm = norm;
    BFLK_CUDA(h, d_packed.reserve(packed_bytes(f, r.kernel == kBcast ? h->bcast.geom.row_bytes : h->tiles.geom.row_bytes)));
    f.packed = d_packed.p;
    if (blocks_per_frame(N) > 1) {
        BFLK_CUDA(h, d_partial.reserve((size_t)n_frames * blocks_per_frame(N) * h->dir_count));
        f.partial = d_partial.p;
    }
    int launches = 0;
    if (r.kernel != kBcast) {
        TileArgs a;
        a.f = f;
        a.wire = wire;
        a.wire_cols = C;
        a.tiles = h->tiles.d_tiles.p;
        a.tile_dirs = h->tiles.d_dirs.p;
        a.n_tiles = h->tiles.n_tiles;
        a.geom = h->tiles.geom;
        a.geom.ksplit = r.split;
        BFLK_CUDA(h, launch_das_tile(a, h->sm_count, st, &launches, timing_hook, h));
    } else {
        BcastArgs a;
        a.f = f;
        a.table = h->bcast.d_table.p;
        a.tile_dirs = h->bcast.d_dirs.p;
        a.n_tiles = h->bcast.n_tiles;
        a.geom = h->bcast.geom;
        BFLK_CUDA(h, launch_das_bcast(a, st, &launches, timing_hook, h));
    }
    h->launches += launches;
    h->kernel_last = r.kernel;
    return BFLK_OK;
}

int bflk::power_map_dev_overlapped(bflk_handle *h, const float *stream_dev, int64_t row_stride, int64_t n_samples, int32_t n_frames,
                                   float *power_dev, cudaStream_t caller, cudaStream_t *used) {
    *used = caller;
    if (!h->have_grid) return h->fail(BFLK_ERR_STATE, "bflk_power_map: set geometry and grid first");
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    bool tiled;
    int rc = tiles_serve(h, &tiled, 0, stream_dev, row_stride);
    if (rc) return rc;
    if (!tiled) return power_map_dev(h, stream_dev, row_stride, n_samples, n_frames, power_dev, Launch{caller});
    const int slot = (int)(h->dev_seq++ & 1);
    // this batch's kernels wait for (a) the caller's stream having reached this call (its inputs), (b) whatever used the handle's
    // scratch on another stream before the overlapped batches began.  Earlier overlapped batches need no wait: the same
    // set's previous batch ran on this very lane, the other set's batch shares nothing with this one.
    BFLK_CUDA(h, cudaEventRecord(h->dev_in[slot], caller));
    if ((rc = lanes_fork(h, h->dev_in[slot], slot))) return rc;
    if ((rc = power_map_dev(h, stream_dev, row_stride, n_samples, n_frames, power_dev, Launch{h->lane[slot], slot, true})))
        return rc;
    // the handle's own stream collects the ends of all overlapped batches: caller_event then covers everything enqueued so far
    if ((rc = lanes_join(h, slot))) return rc;
    *used = h->lane[slot];
    return BFLK_OK;
}

extern "C" {

int bflk_power_map_batch_dev(bflk_handle *h, const float *stream_dev, int64_t n_samples, int32_t n_frames,
                             float *power_dev, void *cuda_stream) {
    return power_map_dev(h, stream_dev, n_samples, n_samples, n_frames, power_dev, Launch{(cudaStream_t)cuda_stream});
}

int bflk_beams_batch_dev(bflk_handle *h, const float *stream_dev, int64_t n_samples, int32_t n_frames, float *beams_dev,
                         float *power_dev, void *cuda_stream) {
    if (!h) return BFLK_ERR_INVALID;
    if (!beams_dev || ((uintptr_t)beams_dev & 7)) return h->fail(BFLK_ERR_INVALID, "bflk_beams_batch_dev: beams_dev is null or not 8-byte aligned");
    return power_map_dev(h, stream_dev, n_samples, n_samples, n_frames, power_dev, Launch{(cudaStream_t)cuda_stream}, beams_dev);
}

int bflk_power_map_batch_dev_submit(bflk_handle *h, const float *stream_dev, int64_t n_samples, int32_t n_frames,
                                    float *power_dev, void *cuda_stream) {
    if (!h) return BFLK_ERR_INVALID;
    if (!stream_dev || !power_dev || n_frames <= 0) return h->fail(BFLK_ERR_INVALID, "bflk_power_map_batch_dev_submit: null buffer or no frames");
    cudaStream_t used;
    return power_map_dev_overlapped(h, stream_dev, n_samples, n_samples, n_frames, power_dev, cuda_stream ? (cudaStream_t)cuda_stream : h->stream, &used);
}

int bflk_power_map_batch_dev_join(bflk_handle *h, void *cuda_stream) {
    if (!h) return BFLK_ERR_INVALID;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : h->stream;
    if (h->last_stream != st) BFLK_CUDA(h, cudaStreamWaitEvent(st, h->caller_event, 0));
    return BFLK_OK;
}

}  // extern "C"

namespace bflk {

// samples a frame needs beyond its own N (the FIR interpolation reads taps - 2 more)
int64_t frame_tail_samples(const bflk_handle *h) {
    return min_stream_samples(h, 1) - h->cfg.frame_len + (h->fir_phases > 0 ? h->fir_taps - 2 : 0);
}

// Host batches go up in chunks of frames: the H2D copy of chunk k+1 (copy stream) overlaps the kernels of chunk k.
// A chunk is ~32 MiB of new samples (measured on B200 / PCIe 5 at cfg3 with wave-aligned chunks: 32 MiB 64.7 k maps/s,
// 64 MiB 61.6 k, 96 MiB 56.9 k), rounded to whole CTA waves of the tiled kernel so PCIe and the SMs both stay busy;
// small batches are one chunk.
int host_chunk_frames(bflk_handle *h, int n_frames, int *chunk_frames_out) {
    const int C = h->cfg.n_channels, N = h->cfg.frame_len;
    const int64_t chunk_bytes = (int64_t)(h->tuning.chunk_mib > 0 ? h->tuning.chunk_mib : 32) << 20;
    const int64_t frame_bytes = (int64_t)C * N * sizeof(float);
    int n_chunks = (int)std::max<int64_t>(1, ((int64_t)n_frames * frame_bytes + chunk_bytes / 2) / chunk_bytes);
    int chunk_frames = (n_frames + n_chunks - 1) / n_chunks;  // even split
    if (n_chunks > 1 && N == 256 && h->sm_count > 0) {
        // the tiled kernel runs one CTA per (tile group, block pair): round the chunk to a whole number of CTA waves
        bool tiled;
        int rc = tiles_serve(h, &tiled);
        if (rc) return rc;
        if (tiled) {
            const int ctas_per_pair = (h->tiles.n_tiles + h->tiles.geom.warps - 1) / h->tiles.geom.warps;
            int g = h->sm_count, b = ctas_per_pair;
            while (b) { const int t = g % b; g = b; b = t; }          // gcd
            const int quantum = 2 * (h->sm_count / g);                // frames per whole wave set
            const int k = std::max(1, (chunk_frames + quantum / 2) / quantum);
            if (k * quantum < n_frames) chunk_frames = k * quantum;
        }
    }
    chunk_frames += chunk_frames & 1;                                 // block pairs
    *chunk_frames_out = std::max(2, chunk_frames);
    return BFLK_OK;
}

}  // namespace bflk

extern "C" {

// A host batch's samples as the chunk loop moves them: what differs between channel-major float rows and sample-major wire
// rows is data here, plus the copy.
struct HostSamples {
    const float *dev = nullptr;       // device copy: channel-major float rows [C][n_samples] ...
    const int32_t *wire = nullptr;    // ... or sample-major wire rows [n_samples][C]
    int64_t frame_elems = 0;          // elements from one frame's first sample to the next's: N, or N * C (wire)
    int64_t first = 0, last = 0;      // samples [first, last) of each channel travel; the frames read nothing outside them
    bool lanes = false;               // several chunks may alternate between the two lanes
    bool sync_upload_on_compute = false;   // a synchronous single-chunk batch uploads on the compute stream itself
    std::function<cudaError_t(int64_t t0, int64_t t1, cudaStream_t st)> upload;   // samples [t0, t1) of every channel
};

// Enqueues a host batch chunk by chunk: the samples of chunk k go up on the copy stream while chunk k - 1 is packed and
// beamformed, and each chunk's maps come back on its compute stream.  Several chunks alternate between the two lanes (each
// with its own scratch set), so the CTAs of chunk k + 1 fill the SMs that the last CTAs of chunk k leave idle one by one;
// the lanes wait for reuse_after (the batch that used these device buffers before), and everything ordered after the
// handle's stream sees the whole batch.  Does not synchronise.
static int host_chunks(bflk_handle *h, const HostSamples &in, int64_t n_samples, int32_t n_frames, int chunk_frames,
                       float *d_out, float *power_out, cudaEvent_t reuse_after) {
    const int N = h->cfg.frame_len;
    const int n_chunks = (n_frames + chunk_frames - 1) / chunk_frames;
    const int64_t tail = frame_tail_samples(h);
    while ((int)h->chunk_events.size() < n_chunks) {
        Event e;
        if (!e) return h->fail(BFLK_ERR_CUDA, "cannot create the chunk events: %s", cudaGetErrorString(cudaGetLastError()));
        h->chunk_events.push_back(std::move(e));
    }
    if (reuse_after) BFLK_CUDA(h, cudaStreamWaitEvent(h->copy_stream, reuse_after, 0));
    const bool lanes = in.lanes && n_chunks > 1;
    if (lanes) {
        int rc = lanes_fork(h, reuse_after);
        if (rc) return rc;
    }
    int64_t copied = in.first;
    for (int k = 0; k < n_chunks; k++) {
        const int f0 = k * chunk_frames, nf = std::min(chunk_frames, n_frames - f0);
        const int64_t need = k == n_chunks - 1 ? in.last : std::min<int64_t>(in.last, (int64_t)(f0 + nf) * N + tail);
        cudaStream_t cs = lanes ? h->lane[k & 1] : h->stream;
        // a synchronous single-chunk call (one live frame) has nothing to overlap: no event hop between two streams
        cudaStream_t up = (n_chunks == 1 && !reuse_after && in.sync_upload_on_compute) ? cs : h->copy_stream;
        if (need > copied) {
            BFLK_CUDA(h, in.upload(copied, need, up));
            copied = need;
        }
        if (up != cs) {
            BFLK_CUDA(h, cudaEventRecord(h->chunk_events[k], h->copy_stream));
            BFLK_CUDA(h, cudaStreamWaitEvent(cs, h->chunk_events[k], 0));
        }
        const int64_t off = (int64_t)f0 * in.frame_elems;
        float *pk = d_out + (size_t)f0 * h->dir_count;
        int rc = power_map_dev(h, in.dev ? in.dev + off : nullptr, n_samples, copied - (int64_t)f0 * N, nf, pk,
                               Launch{cs, lanes ? (k & 1) : 0, lanes, in.wire ? in.wire + off : nullptr});
        if (rc) return rc;
        BFLK_CUDA(h, cudaMemcpyAsync(power_out + (size_t)f0 * h->dir_count, pk, (size_t)nf * h->dir_count * sizeof(float),
                                     cudaMemcpyDeviceToHost, cs));
    }
    return lanes ? lanes_join(h) : BFLK_OK;
}

// One float host batch into the device buffers d_in / d_out of this batch.  Does not synchronise.
static int host_batch_enqueue(bflk_handle *h, const float *stream, int64_t n_samples, int32_t n_frames, float *power_out,
                              DevBuf<float> &d_in, DevBuf<float> &d_out, cudaEvent_t reuse_after) {
    const int C = h->cfg.n_channels, N = h->cfg.frame_len;
    const size_t n_in = (size_t)C * n_samples, n_out = (size_t)n_frames * h->dir_count;
    BFLK_CUDA(h, d_in.reserve(n_in));
    BFLK_CUDA(h, d_out.reserve(n_out));
    int chunk_frames = n_frames;
    int rc = host_chunk_frames(h, n_frames, &chunk_frames);
    if (rc) return rc;
    // only the samples a frame can touch travel: [history - largest delay, last frame's last tap] -- a third of the
    // reference's 1024-sample window for a single frame (the rest of d_in is never read)
    // (a strided copy out of PAGEABLE memory is staged row by row by the driver and loses more than it saves -- measured
    // cfg3: 289 -> 402 us; pageable single-chunk batches go up as one contiguous copy instead)
    cudaPointerAttributes attr{};
    const bool pageable = cudaPointerGetAttributes(&attr, stream) != cudaSuccess || attr.type == cudaMemoryTypeUnregistered;
    cudaGetLastError();
    if (pageable && chunk_frames >= n_frames) {
        if (reuse_after) BFLK_CUDA(h, cudaStreamWaitEvent(h->stream, reuse_after, 0));
        BFLK_CUDA(h, cudaMemcpyAsync(d_in.p, stream, n_in * sizeof(float), cudaMemcpyHostToDevice, h->stream));
        rc = power_map_dev(h, d_in.p, n_samples, n_samples, n_frames, d_out.p, Launch{h->stream});
        if (rc) return rc;
        BFLK_CUDA(h, cudaMemcpyAsync(power_out, d_out.p, n_out * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
        return BFLK_OK;
    }
    HostSamples in;
    in.dev = d_in.p;
    in.frame_elems = N;
    in.first = pageable ? 0 : std::max<int64_t>(0, (int64_t)(h->cfg.history - h->max_delay) & ~(int64_t)3);
    in.last = std::min<int64_t>(n_samples, (int64_t)(n_frames - 1) * N + frame_tail_samples(h) + N);
    in.lanes = true;
    in.sync_upload_on_compute = true;
    float *dev = d_in.p;
    in.upload = [=](int64_t t0, int64_t t1, cudaStream_t st) {
        return cudaMemcpy2DAsync(dev + t0, n_samples * sizeof(float), stream + t0, n_samples * sizeof(float),
                                 (t1 - t0) * sizeof(float), C, cudaMemcpyHostToDevice, st);
    };
    return host_chunks(h, in, n_samples, n_frames, chunk_frames, d_out.p, power_out, reuse_after);
}

static int host_batch_check(bflk_handle *h, const float *stream, int64_t n_samples, int32_t n_frames, const float *power_out) {
    if (!h->have_grid) return h->fail(BFLK_ERR_STATE, "bflk_power_map: set geometry and grid first");
    if (!stream || !power_out || n_frames <= 0 || n_samples <= 0) return h->fail(BFLK_ERR_INVALID, "bflk_power_map: null buffer or no frames");
    return check_frames(h, n_samples, n_frames, "bflk_power_map");
}

int bflk_power_map_batch_wait(bflk_handle *h) {
    if (!h) return BFLK_ERR_INVALID;
    if (h->async_pending == 0) return BFLK_OK;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const int slot = (int)((h->async_seq - h->async_pending) & 1);   // the oldest batch in flight
    BFLK_CUDA(h, cudaEventSynchronize(h->async_done[slot]));
    h->async_pending--;
    return BFLK_OK;
}

// Asynchronous flavour for continuous operation: returns once the batch is enqueued; at most two batches are in flight
// (a third submit first waits for the oldest).  The upload of batch i + 1 overlaps the kernels of batch i.
int bflk_power_map_batch_submit(bflk_handle *h, const float *stream, int64_t n_samples, int32_t n_frames, float *power_out) {
    if (!h) return BFLK_ERR_INVALID;
    int rc = host_batch_check(h, stream, n_samples, n_frames, power_out);
    if (rc) return rc;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    while (h->async_pending >= 2)
        if ((rc = bflk_power_map_batch_wait(h))) return rc;
    const int slot = (int)(h->async_seq & 1);
    rc = host_batch_enqueue(h, stream, n_samples, n_frames, power_out, h->d_async_in[slot], h->d_async_out[slot],
                            h->async_seq >= 2 ? (cudaEvent_t)h->async_done[slot] : nullptr);
    if (rc) return rc;
    BFLK_CUDA(h, cudaEventRecord(h->async_done[slot], h->stream));
    h->async_seq++;
    h->async_pending++;
    h->last_map_on_device = false;
    return BFLK_OK;
}

int bflk_power_map_batch(bflk_handle *h, const float *stream, int64_t n_samples, int32_t n_frames, float *power_out) {
    if (!h) return BFLK_ERR_INVALID;
    int rc = host_batch_check(h, stream, n_samples, n_frames, power_out);
    if (rc) return rc;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    h->last_map_on_device = false;
    rc = host_batch_enqueue(h, stream, n_samples, n_frames, power_out, h->d_window, h->d_maps, nullptr);
    if (rc) return rc;
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    h->async_pending = 0;                    // everything queued on the stream before this call has completed too
    h->last_map_on_device = n_frames == 1;   // d_maps[0 .. count) is the map: bflk_targets(NULL) / bflk_heatmap(NULL) use it
    return BFLK_OK;
}

static int wire_check(bflk_handle *h, int64_t n_samples) {
    if (h->cfg.n_channels % 8) return h->fail(BFLK_ERR_INVALID, "bflk_power_map_batch_i32: n_channels must be a multiple of 8 (serpentine rows)");
    if (n_samples > 0x7fffffff) return h->fail(BFLK_ERR_INVALID, "bflk_power_map_batch_i32: more than 2^31 samples per call");
    return BFLK_OK;
}

// frames[n_samples][C] int32 on the DEVICE, frame b = rows [b * N, b * N + H + N + 1): asynchronous on cuda_stream
int bflk_power_map_batch_i32_dev(bflk_handle *h, const int32_t *frames_dev, int64_t n_samples, int32_t n_frames,
                                 float *power_dev, void *cuda_stream) {
    if (!h) return BFLK_ERR_INVALID;
    if (!frames_dev) return h->fail(BFLK_ERR_INVALID, "bflk_power_map_batch_i32: null buffer");
    int rc = wire_check(h, n_samples);
    if (rc) return rc;
    return power_map_dev(h, nullptr, n_samples, n_samples, n_frames, power_dev, Launch{(cudaStream_t)cuda_stream, 0, false, frames_dev});
}

// Host buffers: the wire samples go up in chunks of frames (contiguous rows of the sample-major layout) on the copy
// stream while the previous chunk is packed and beamformed.
int bflk_power_map_batch_i32(bflk_handle *h, const int32_t *frames, int64_t n_samples, int32_t n_frames, float *power_out) {
    if (!h) return BFLK_ERR_INVALID;
    if (!h->have_grid) return h->fail(BFLK_ERR_STATE, "bflk_power_map_batch_i32: set geometry and grid first");
    if (!frames || !power_out || n_frames <= 0) return h->fail(BFLK_ERR_INVALID, "bflk_power_map_batch_i32: null buffer or no frames");
    int rc = check_frames(h, n_samples, n_frames, "bflk_power_map_batch_i32");
    if (rc) return rc;
    if ((rc = wire_check(h, n_samples))) return rc;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const int C = h->cfg.n_channels, N = h->cfg.frame_len;
    BFLK_CUDA(h, h->d_wire.reserve((size_t)C * n_samples));
    h->last_map_on_device = false;
    BFLK_CUDA(h, h->d_maps.reserve((size_t)n_frames * h->dir_count));
    int chunk_frames = n_frames;
    if ((rc = host_chunk_frames(h, n_frames, &chunk_frames))) return rc;
    HostSamples in;
    in.wire = h->d_wire.p;
    in.frame_elems = (int64_t)N * C;
    in.last = n_samples;
    // two lanes only when the register-tiled kernel takes the wire samples directly: the other kernels convert them into
    // the handle's one float window first (ingest_kernel)
    if (chunk_frames < n_frames && (rc = tiles_serve(h, &in.lanes))) return rc;
    int32_t *dev = h->d_wire.p;
    in.upload = [=](int64_t t0, int64_t t1, cudaStream_t st) {
        return cudaMemcpyAsync(dev + (size_t)t0 * C, frames + (size_t)t0 * C, (size_t)(t1 - t0) * C * sizeof(int32_t),
                               cudaMemcpyHostToDevice, st);
    };
    if ((rc = host_chunks(h, in, n_samples, n_frames, chunk_frames, h->d_maps.p, power_out, nullptr))) return rc;
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    h->last_map_on_device = n_frames == 1;
    return BFLK_OK;
}

int bflk_power_map_i32(bflk_handle *h, const int32_t *frames, float *power_out) {
    if (!h) return BFLK_ERR_INVALID;
    return bflk_power_map_batch_i32(h, frames, h->cfg.window_len, 1, power_out);
}

int bflk_power_map(bflk_handle *h, const float *window, float *power_out) {
    if (!h) return BFLK_ERR_INVALID;
    return bflk_power_map_batch(h, window, h->cfg.window_len, 1, power_out);
}

// ---- MISO ---------------------------------------------------------------------------------------------------
// The window can live on the device across calls (the tracker evaluates many steps on one frame,
// src/dsp/gradient_ascend.cpp:301-409): bflk_set_window uploads it once, bflk_set_window_dev borrows a device buffer,
// bflk_stream_window points at a frame in the session's ring.  Its rows are `stride` floats apart; frame >= 0: that
// session frame.
static void set_resident(bflk_handle *h, const float *window_dev, int64_t stride, int64_t frame = -1) {
    h->resident_window = window_dev;
    h->resident_stride = stride;
    if (h->session) h->session->window_frame = window_dev ? frame : -1;
}

// samples per channel the resident window holds from its first one: window_len, or what the ring has received from the
// session frame on
static int64_t resident_len(const bflk_handle *h) {
    const Session *s = h->session.get();
    return s && s->window_frame >= 0 ? s->pushed - s->window_frame * h->cfg.frame_len : h->cfg.window_len;
}

int bflk_set_window(bflk_handle *h, const float *window) {
    if (!h) return BFLK_ERR_INVALID;
    if (!window) {
        set_resident(h, nullptr, 0);
        return BFLK_OK;
    }
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const size_t n_in = (size_t)h->cfg.n_channels * h->cfg.window_len;
    BFLK_CUDA(h, h->d_resident.reserve(n_in));
    BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));   // a caller's stream may still read the old one
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_resident.p, window, n_in * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    set_resident(h, h->d_resident.p, h->cfg.window_len);
    return BFLK_OK;
}

int bflk_set_window_dev(bflk_handle *h, const float *window_dev) {
    if (!h) return BFLK_ERR_INVALID;
    set_resident(h, window_dev, h->cfg.window_len);
    return BFLK_OK;
}

// One launch on `st`.  Up to kMisoInline directions travel in the kernel's parameter space; more go through the pinned
// trig staging, whose reuse (and that of the device scratch) is ordered against a caller's stream by caller_event.
// flag_dev receives the call's epoch if a delay exceeds the history.  The window's rows are row_stride floats apart.
static int miso_launch(bflk_handle *h, const double *theta, const double *phi, int n_targets, const float *window_dev,
                       int64_t row_stride, float *audio_dev, float *power_dev, int32_t *flag_dev, cudaStream_t st) {
    const int C = h->cfg.n_channels, N = h->cfg.frame_len;
    // the partial sums, counters and range flag are the handle's: a call on another stream than the previous one waits for it
    if (h->last_stream != st) BFLK_CUDA(h, cudaStreamWaitEvent(st, h->caller_event, 0));
    MisoArgs a{};
    if (n_targets <= kMisoInline) {
        for (int i = 0; i < n_targets; i++) a.trig_inline[i] = make_trig(theta[i], phi[i]);
        a.n_inline = n_targets;
    } else {
        BFLK_CUDA(h, h->p_trig.reserve(n_targets));
        BFLK_CUDA(h, h->d_trig.reserve(n_targets));
        BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));   // the previous call's copy is done with the staging
        for (int i = 0; i < n_targets; i++) h->p_trig.p[i] = make_trig(theta[i], phi[i]);
        BFLK_CUDA(h, cudaMemcpyAsync(h->d_trig.p, h->p_trig.p, n_targets * sizeof(DirTrig), cudaMemcpyHostToDevice, st));
        a.trig = h->d_trig.p;
    }
    if (power_dev) {
        const size_t slots = (size_t)n_targets * das_miso_slices(N);
        if (slots > h->d_miso_partial.n || (size_t)n_targets > h->d_miso_counters.n) {
            BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));
            BFLK_CUDA(h, h->d_miso_partial.reserve(slots));
            const size_t had = h->d_miso_counters.n;
            BFLK_CUDA(h, h->d_miso_counters.reserve(std::max<size_t>(n_targets, 256)));
            if (h->d_miso_counters.n != had) BFLK_CUDA(h, cudaMemsetAsync(h->d_miso_counters.p, 0, h->d_miso_counters.n * sizeof(unsigned), st));
        }
        a.partial = h->d_miso_partial.p;
        a.counters = h->d_miso_counters.p;
    }
    a.window = window_dev;
    a.row_stride = row_stride;
    a.n_frames = 1;
    a.frame_len = N;
    a.frame_stride = N;
    a.xyz = h->d_xyz.p;
    a.C = C;
    a.index = h->d_index.p;
    a.usable = (int)h->index.size();
    a.k_scale = delay_scale(h);
    a.history = h->cfg.history;
    a.n_targets = n_targets;
    a.audio = audio_dev;
    a.power = power_dev;
    a.norm = static_cast<float>(N);  // Particle::beam: power_accumulator /= N_SAMPLES, particle.cpp:79
    a.error_flag = flag_dev;
    a.focus = h->focus;
    a.epoch = ++h->miso_epoch;
    if (h->miso_epoch == 0x7fffffff) h->miso_epoch = 0;
    BFLK_CUDA(h, launch_das_miso(a, st));
    h->launches++;
    return note_use(h, st, false);
}

// window_dev: rows row_stride floats apart, each holding n_samples samples
static int miso_dev(bflk_handle *h, const double *theta, const double *phi, int32_t n_targets, const float *window_dev,
                    int64_t row_stride, int64_t n_samples, float *audio_dev, float *power_dev, cudaStream_t st) {
    if (h->fir_phases == 0) {
        if (h->d_miso_out.n == 0) {
            BFLK_CUDA(h, h->d_miso_out.reserve(1));
            BFLK_CUDA(h, cudaMemsetAsync(h->d_miso_out.p, 0, sizeof(float), st));
        }
        return miso_launch(h, theta, phi, n_targets, window_dev, row_stride, audio_dev, power_dev,
                           reinterpret_cast<int32_t *>(h->d_miso_out.p), st);
    }
    // FIR interpolation (bflk_set_fir): tables through the table kernel, then the generic kernel
    const int C = h->cfg.n_channels, N = h->cfg.frame_len;
    const size_t TC = (size_t)n_targets * C;
    BFLK_CUDA(h, h->d_soff.reserve(TC));
    BFLK_CUDA(h, h->d_sfrac.reserve(TC));
    BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));
    int32_t max_delay = 0;
    int rc = run_steer_tables(h, theta, phi, n_targets, h->d_soff.p, h->d_sfrac.p, &max_delay, h->focus);  // Particle::steer
    if (rc) return rc;
    if ((rc = check_delay_range(h, max_delay, "bflk_miso"))) return rc;
    if (n_samples < h->cfg.history + N + h->fir_taps - 1)
        return h->fail(BFLK_ERR_INVALID, "bflk_miso: the window is too short for the FIR taps");
    GenericArgs a{};
    a.stream = window_dev;
    a.row_stride = row_stride;
    a.n_frames = 1;
    a.frame_len = N;
    a.frame_stride = N;
    a.off = h->d_soff.p;
    a.frac = h->d_sfrac.p;
    a.C = C;
    a.index = h->d_index.p;
    a.usable = (int)h->index.size();
    a.n_dir = n_targets;
    a.power = power_dev;
    a.audio = audio_dev;
    a.norm = static_cast<float>(N);
    a.fir = h->d_fir.p; a.fir_phases = h->fir_phases; a.fir_taps = h->fir_taps;
    if (h->last_stream != st) BFLK_CUDA(h, cudaStreamWaitEvent(st, h->caller_event, 0));
    BFLK_CUDA(h, launch_das_generic(a, st));
    h->launches++;
    return note_use(h, st, false);
}

int bflk_miso_dev(bflk_handle *h, const double *theta, const double *phi, int32_t n_targets, const float *window_dev,
                  float *audio_dev, float *power_dev, void *cuda_stream) {
    if (!h) return BFLK_ERR_INVALID;
    if (!h->have_geometry) return h->fail(BFLK_ERR_STATE, "bflk_miso: set the geometry first");
    if (!theta || !phi || n_targets <= 0 || (!window_dev && !h->resident_window))
        return h->fail(BFLK_ERR_INVALID, "bflk_miso: null / empty arguments (no window given and none resident)");
    if (int rc = check_focus(h, h->focus, "bflk_miso")) return rc;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : h->stream;
    if (window_dev) return miso_dev(h, theta, phi, n_targets, window_dev, h->cfg.window_len, h->cfg.window_len, audio_dev, power_dev, st);
    return miso_dev(h, theta, phi, n_targets, h->resident_window, h->resident_stride, resident_len(h), audio_dev, power_dev, st);
}

int bflk_miso(bflk_handle *h, const double *theta, const double *phi, int32_t n_targets, const float *window,
              float *audio_out, float *power_out) {
    if (!h) return BFLK_ERR_INVALID;
    if (!h->have_geometry) return h->fail(BFLK_ERR_STATE, "bflk_miso: set the geometry first");
    if (!theta || !phi || n_targets <= 0 || (!window && !h->resident_window))
        return h->fail(BFLK_ERR_INVALID, "bflk_miso: null / empty arguments (no window given and none resident)");
    if (int rc = check_focus(h, h->focus, "bflk_miso")) return rc;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const int N = h->cfg.frame_len;
    const size_t n_in = (size_t)h->cfg.n_channels * h->cfg.window_len;
    const float *wdev = h->resident_window;
    int64_t stride = h->resident_stride, len = resident_len(h);
    if (window) {
        BFLK_CUDA(h, h->d_window.reserve(n_in));
        BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));
        BFLK_CUDA(h, cudaMemcpyAsync(h->d_window.p, window, n_in * sizeof(float), cudaMemcpyHostToDevice, h->stream));
        wdev = h->d_window.p;
        stride = len = h->cfg.window_len;
    }
    // device output block [flag | audio | power] -> ONE copy into pinned staging -> the caller's buffers
    const size_t n_audio = audio_out ? (size_t)n_targets * N : 0, n_power = power_out ? n_targets : 0, n_all = 1 + n_audio + n_power;
    if (n_all > h->d_miso_out.n) {
        BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));
        BFLK_CUDA(h, h->d_miso_out.reserve(n_all));
        BFLK_CUDA(h, cudaMemsetAsync(h->d_miso_out.p, 0, sizeof(float), h->stream));   // the range flag starts clear
    }
    BFLK_CUDA(h, h->p_stage.reserve(n_all));
    float *d_audio = h->d_miso_out.p + 1, *d_power = d_audio + n_audio;
    int rc;
    if (h->fir_phases == 0) {
        rc = miso_launch(h, theta, phi, n_targets, wdev, stride, audio_out ? d_audio : nullptr, power_out ? d_power : nullptr,
                         reinterpret_cast<int32_t *>(h->d_miso_out.p), h->stream);
    } else {
        rc = miso_dev(h, theta, phi, n_targets, wdev, stride, len, audio_out ? d_audio : nullptr, power_out ? d_power : nullptr, h->stream);
    }
    if (rc) return rc;
    BFLK_CUDA(h, cudaMemcpyAsync(h->p_stage.p, h->d_miso_out.p, n_all * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    int32_t flag;
    std::memcpy(&flag, h->p_stage.p, sizeof(flag));
    if (h->fir_phases == 0 && flag == h->miso_epoch)
        return h->fail(BFLK_ERR_RANGE, "bflk_miso: a steering delay exceeds history %d", h->cfg.history);
    if (audio_out) std::memcpy(audio_out, h->p_stage.p + 1, n_audio * sizeof(float));
    if (power_out) std::memcpy(power_out, h->p_stage.p + 1 + n_audio, n_power * sizeof(float));
    return BFLK_OK;
}

// ---- FIR interpolation mode (SURVEY 8f, f4) ---------------------------------------------------------------------
int bflk_set_fir(bflk_handle *h, const float *coeffs, int32_t n_phases, int32_t n_taps) {
    if (!h) return BFLK_ERR_INVALID;
    if (!coeffs) {
        h->fir_phases = h->fir_taps = 0;
        return BFLK_OK;
    }
    if (n_phases < 2 || n_taps < 1 || n_taps > 64) return h->fail(BFLK_ERR_INVALID, "bflk_set_fir: %d phases x %d taps", n_phases, n_taps);
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    BFLK_CUDA(h, h->d_fir.reserve((size_t)n_phases * n_taps));
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_fir.p, coeffs, (size_t)n_phases * n_taps * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    h->fir_phases = n_phases;
    h->fir_taps = n_taps;
    return BFLK_OK;
}

// ---- monopulse step (SURVEY 8f, f2) ---------------------------------------------------------------------------
// Spherical::quadrant + normalizeSpherical in double on the host (geometry.cpp:181-217, :120-142, :11-20; particle.h:24-27).
// Eigen's 3x3 / 4x3 products are pinned as ((a0 b0 + a1 b1) + a2 b2) without contraction (this file is built with
// -ffp-contract=off), the same order oracle/oracle.c uses.
static inline double dot3(const double *a, const double *b, int sb) { return (a[0] * b[0] + a[1] * b[sb]) + a[2] * b[2 * sb]; }

static void quadrant_directions(double *theta, double phi, double spread, double theta_limit, double *near_theta, double *near_phi) {
    static const double deg[4] = {45.0, 315.0, 225.0, 135.0};
    double search[4][3];
    for (int i = 0; i < 4; i++) {
        const double a = deg[i] * (M_PI / 180.0);
        search[i][0] = 1.0 * sin(spread) * cos(a);
        search[i][1] = 1.0 * sin(spread) * sin(a);
        search[i][2] = 1.0 * cos(spread);
    }
    double rt = *theta;
    if (rt + spread > M_PI / 2.0) {
        rt -= spread;
        *theta -= spread / 2.0;
    }
    const double Rz[9] = {cos(phi), -sin(phi), 0.0, sin(phi), cos(phi), 0.0, 0.0, 0.0, 1.0};
    const double Ry[9] = {cos(rt), 0.0, sin(rt), 0.0, 1.0, 0.0, -sin(rt), 0.0, cos(rt)};
    double R[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) R[3 * i + j] = dot3(Ry + 3 * i, Rz + j, 3);
    for (int i = 0; i < 4; i++) {
        double k[3];
        for (int j = 0; j < 3; j++) k[j] = dot3(search[i], R + j, 3);
        double nt = acos(k[2]);
        double np = fmod(atan2(k[1], k[0]) - M_PI, 2.0 * M_PI);
        if (np < 0.0) np = 2.0 * M_PI + np;
        nt = nt < 0.0 ? 0.0 : (nt > theta_limit ? theta_limit : nt);
        near_theta[i] = nt;
        near_phi[i] = np;
    }
}

int bflk_monopulse(bflk_handle *h, double *theta, const double *phi, int32_t n_particles, double spread,
                   double theta_limit, double reference, const float *window, double *near_theta, double *near_phi,
                   double *q, double *gradient, double *error) {
    if (!h) return BFLK_ERR_INVALID;
    if (!theta || !phi || n_particles <= 0 || (!window && !h->resident_window))
        return h->fail(BFLK_ERR_INVALID, "bflk_monopulse: null / empty arguments (no window given and none resident)");
    const int T = 4 * n_particles;
    std::vector<double> nth(T), nph(T);
    for (int p = 0; p < n_particles; p++) quadrant_directions(&theta[p], phi[p], spread, theta_limit, &nth[4 * p], &nph[4 * p]);
    std::vector<float> power(T);
    int rc = bflk_miso(h, nth.data(), nph.data(), T, window, nullptr, power.data());   // one launch for all beams
    if (rc) return rc;
    for (int p = 0; p < n_particles; p++) {
        const double q1 = power[4 * p], q2 = power[4 * p + 1], q3 = power[4 * p + 2], q4 = power[4 * p + 3];   // beam() returns double
        const double sum = q1 + q2 + q3 + q4;
        const double gphi = (q1 + q4) - (q2 + q3), gtheta = (q3 + q4) - (q1 + q2);
        if (error) error[p] = (fabs(gphi) + fabs(gtheta)) / sum;
        if (gradient) {
            gradient[3 * p] = reference > 0.0 ? gtheta / reference : gtheta;
            gradient[3 * p + 1] = reference > 0.0 ? gphi / reference : gphi;
            gradient[3 * p + 2] = sum / 4;
        }
        if (q) { q[4 * p] = q1; q[4 * p + 1] = q2; q[4 * p + 2] = q3; q[4 * p + 3] = q4; }
    }
    if (near_theta) std::memcpy(near_theta, nth.data(), T * sizeof(double));
    if (near_phi) std::memcpy(near_phi, nph.data(), T * sizeof(double));
    return BFLK_OK;
}

// ---- Targets of the maps ------------------------------------------------------------------------------------------
// Targets carry the grid's angles: they need a bflk_set_grid_fov grid (caller tables have none, with or without a shape).
static bool fov_grid(const bflk_handle *h) { return h->have_grid && h->rows > 0 && h->cols > 0 && !h->theta.empty(); }

// Targets of k whole-grid maps d_maps[k][D] on the handle's stream, synchronously: out[k][max_targets] (records past a map's
// count are not written) and counts[k] on the host.  Work the caller enqueued on the handle's stream before is done too.
static int host_targets(bflk_handle *h, const float *d_maps, int k, int max_targets, float min_rel, bflk_target *out,
                        int32_t *counts) {
    const size_t n_rec = (size_t)k * max_targets;
    BFLK_CUDA(h, h->d_targets.reserve(n_rec));
    BFLK_CUDA(h, h->d_target_counts.reserve(k));
    BFLK_CUDA(h, h->p_targets.reserve(n_rec));
    BFLK_CUDA(h, h->p_target_counts.reserve(k));
    BFLK_CUDA(h, launch_map_targets(d_maps, k, h->rows, h->cols, max_targets, min_rel, h->d_theta.p, h->d_phi.p,
                                    h->d_targets.p, h->d_target_counts.p, h->sm_count, h->stream));
    h->launches++;
    BFLK_CUDA(h, cudaMemcpyAsync(h->p_targets.p, h->d_targets.p, n_rec * sizeof(bflk_target), cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaMemcpyAsync(h->p_target_counts.p, h->d_target_counts.p, k * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    for (int b = 0; b < k; b++) {
        const int32_t n = h->p_target_counts.p[b];
        std::memcpy(out + (size_t)b * max_targets, h->p_targets.p + (size_t)b * max_targets, n * sizeof(bflk_target));
        counts[b] = n;
    }
    return BFLK_OK;
}

int bflk_targets_batch_dev(bflk_handle *h, const float *power_dev, int32_t n_maps, int32_t max_targets, float min_rel_power,
                           bflk_target *targets_dev, int32_t *n_dev, void *cuda_stream) {
    if (!h) return BFLK_ERR_INVALID;
    if (!power_dev || !targets_dev || !n_dev || n_maps < 1 || max_targets < 1 || max_targets > 256)
        return h->fail(BFLK_ERR_INVALID, "bflk_targets_batch_dev: null buffer, n_maps = %d or max_targets = %d (1..256)", n_maps, max_targets);
    if (!fov_grid(h)) return h->fail(BFLK_ERR_STATE, "bflk_targets_batch_dev: needs a rows x cols grid (bflk_set_grid_fov)");
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : h->stream;
    // ordered like power_map_dev: after the handle's work on another stream (its maps, its angles), and recorded for the next
    if (h->last_stream != st) BFLK_CUDA(h, cudaStreamWaitEvent(st, h->caller_event, 0));
    const cudaError_t e = launch_map_targets(power_dev, n_maps, h->rows, h->cols, max_targets, min_rel_power, h->d_theta.p,
                                             h->d_phi.p, targets_dev, n_dev, h->sm_count, st);
    const int rc = note_use(h, st, false);
    BFLK_CUDA(h, e);
    h->launches++;
    return rc;
}

// ---- streaming session (bflk_internal.h: Session) ---------------------------------------------------------------
static Session *session_of(bflk_handle *h, const char *who) {
    if (!h->session) h->fail(BFLK_ERR_STATE, "%s: no session open (bflk_stream_open)", who);
    return h->session.get();
}

// ready frames: from next_frame on, the frames whose last sample (tail samples past their own N) has been pushed
static int64_t ready_frames(const bflk_handle *h, const Session *s) {
    const int64_t N = h->cfg.frame_len, end = s->pushed - N - frame_tail_samples(h);   // last ready frame starts at or before end
    return end < 0 ? 0 : std::max<int64_t>(0, end / N + 1 - s->next_frame);
}

int bflk_stream_close(bflk_handle *h) {
    if (!h) return BFLK_ERR_INVALID;
    if (!session_of(h, "bflk_stream_close")) return BFLK_ERR_STATE;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));   // a caller's stream may still read a session frame
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    if (h->session->window_frame >= 0) set_resident(h, nullptr, 0);
    h->session.reset();
    return BFLK_OK;
}

int bflk_stream_open(bflk_handle *h, int32_t max_frames) {
    if (!h) return BFLK_ERR_INVALID;
    if (max_frames < 1) return h->fail(BFLK_ERR_INVALID, "bflk_stream_open: max_frames = %d", max_frames);
    if (h->session) {
        int rc = bflk_stream_close(h);
        if (rc) return rc;
    }
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const int64_t N = h->cfg.frame_len, C = h->cfg.n_channels, tail = frame_tail_samples(h);
    // max_frames frames and the tail of the last one, in whole frames: frame starts fall on multiples of N in the ring
    const int64_t cap = ((int64_t)max_frames * N + tail + N - 1) / N * N;
    if (cap > 0x7fffffff) return h->fail(BFLK_ERR_INVALID, "bflk_stream_open: %d frames need more than 2^31 samples per channel", max_frames);
    cudaGetLastError();   // the check below is about the session's events
    std::unique_ptr<Session> s(new Session());
    BFLK_CUDA(h, cudaGetLastError());
    BFLK_CUDA(h, s->ring.reserve((size_t)C * 2 * cap));
    BFLK_CUDA(h, s->stage.reserve((size_t)C * cap));
    s->cap = cap;
    s->tail = tail;
    h->session = std::move(s);
    return BFLK_OK;
}

// One push: a single upload of the block into the stage, then history_push_kernel, on the handle's stream.
static int stream_push(bflk_handle *h, const void *block, int32_t n, bool wire, const char *who) {
    if (!h) return BFLK_ERR_INVALID;
    Session *s = session_of(h, who);
    if (!s) return BFLK_ERR_STATE;
    if (!block || n < 1 || n > s->cap)
        return h->fail(BFLK_ERR_INVALID, "%s: %d samples per channel (a push takes 1 to %lld)", who, n, (long long)s->cap);
    const int C = h->cfg.n_channels, N = h->cfg.frame_len;
    if (wire && C % 8) return h->fail(BFLK_ERR_INVALID, "%s: n_channels must be a multiple of 8 (serpentine rows)", who);
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    // the previous push's kernel has read the stage: it is earlier on the same stream
    BFLK_CUDA(h, cudaMemcpyAsync(s->stage.p, block, (size_t)C * n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, cudaEventRecord(s->copied, h->stream));
    BFLK_CUDA(h, cudaStreamWaitEvent(h->stream, h->caller_event, 0));   // earlier readers of the history it overwrites
    BFLK_CUDA(h, launch_history_push(wire ? nullptr : s->stage.p, wire ? reinterpret_cast<const int32_t *>(s->stage.p) : nullptr,
                                     n, C, s->pushed, (int)s->cap, s->ring.p, h->stream));
    h->launches++;
    BFLK_CUDA(h, cudaEventRecord(s->written, h->stream));
    s->pushed += n;
    // overrun: the samples before `held` are gone, and with them every frame that starts there
    const int64_t held = s->pushed - s->cap;
    if (held > s->next_frame * N) {
        const int64_t first = (held + N - 1) / N;
        s->skipped += first - s->next_frame;
        s->next_frame = first;
    }
    if (s->window_frame >= 0 && s->window_frame * N < held) set_resident(h, nullptr, 0);
    BFLK_CUDA(h, cudaEventSynchronize(s->copied));
    return BFLK_OK;
}

int bflk_stream_push(bflk_handle *h, const float *samples, int32_t n) {
    return stream_push(h, samples, n, false, "bflk_stream_push");
}

int bflk_stream_push_i32(bflk_handle *h, const int32_t *rows, int32_t n) {
    return stream_push(h, rows, n, true, "bflk_stream_push_i32");
}

// What a session maps call returns besides the maps: nothing (bflk_stream_power_maps), the beams (bflk_session_beams) or
// the Targets of every map (bflk_session_targets).  All three take and consume the same frames the same way.
struct SessionOut {
    enum { kMaps, kBeams, kTargets } mode = kMaps;
    float *beams = nullptr;          // kBeams: [n][count][N]
    bflk_target *targets = nullptr;  // kTargets: [n][max_targets], with the counts [n]
    int32_t *n_targets = nullptr;
    int32_t max_targets = 0;
    float min_rel = 0.f;
};

static int stream_maps(bflk_handle *h, int32_t max_frames, float *power_out, const SessionOut &o, int64_t *first_frame,
                       int32_t *n_frames, const char *who) {
    if (!h) return BFLK_ERR_INVALID;
    Session *s = session_of(h, who);
    if (!s) return BFLK_ERR_STATE;
    const bool with_beams = o.mode == SessionOut::kBeams, with_targets = o.mode == SessionOut::kTargets;
    if (!power_out || (with_beams && !o.beams) || (with_targets && (!o.targets || !o.n_targets)) || !first_frame || !n_frames || max_frames < 1)
        return h->fail(BFLK_ERR_INVALID, "%s: null output or max_frames = %d", who, max_frames);
    if (with_targets && (o.max_targets < 1 || o.max_targets > 256))
        return h->fail(BFLK_ERR_INVALID, "%s: max_targets = %d (1..256)", who, o.max_targets);
    if (!h->have_grid) return h->fail(BFLK_ERR_STATE, "%s: set geometry and grid first", who);
    if (with_targets && (!fov_grid(h) || h->dir_count != h->n_dir))
        return h->fail(BFLK_ERR_STATE, "%s: needs a rows x cols grid (bflk_set_grid_fov) and the whole map on this handle", who);
    const int64_t tail = frame_tail_samples(h);
    if (tail > s->tail)
        return h->fail(BFLK_ERR_STATE, "%s: a frame now reads %lld samples past its own, the session was opened for %lld (open it again)",
                       who, (long long)tail, (long long)s->tail);
    *first_frame = s->next_frame;
    *n_frames = 0;
    const int k = (int)std::min<int64_t>(max_frames, ready_frames(h, s));
    if (k == 0) return BFLK_OK;
    const int N = h->cfg.frame_len;
    const size_t n_beams = (size_t)k * h->dir_count * N;
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    h->last_map_on_device = false;
    BFLK_CUDA(h, h->d_maps.reserve((size_t)k * h->dir_count));
    if (with_beams) BFLK_CUDA(h, h->d_beams.reserve(n_beams));
    // the k frames and the tail of the last one: ready and still held, so at most cap samples, contiguous in the ring
    const float *window = s->ring.p + s->next_frame * N % s->cap;
    int rc = power_map_dev(h, window, 2 * s->cap, (int64_t)k * N + tail, k, h->d_maps.p, Launch{h->stream},
                           with_beams ? h->d_beams.p : nullptr);
    if (rc) return rc;
    BFLK_CUDA(h, cudaMemcpyAsync(power_out, h->d_maps.p, (size_t)k * h->dir_count * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (with_beams) BFLK_CUDA(h, cudaMemcpyAsync(o.beams, h->d_beams.p, n_beams * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (with_targets) rc = host_targets(h, h->d_maps.p, k, o.max_targets, o.min_rel, o.targets, o.n_targets);
    else BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    if (rc) return rc;
    s->next_frame += k;
    *n_frames = k;
    h->last_map_on_device = k == 1;   // d_maps[0 .. count) is the map: bflk_targets(NULL) / bflk_heatmap(NULL) use it
    return BFLK_OK;
}

int bflk_stream_power_maps(bflk_handle *h, int32_t max_frames, float *power_out, int64_t *first_frame, int32_t *n_frames) {
    return stream_maps(h, max_frames, power_out, SessionOut{}, first_frame, n_frames, "bflk_stream_power_maps");
}

int bflk_session_beams(bflk_handle *h, int32_t max_frames, float *beams_out, float *power_out, int64_t *first_frame,
                       int32_t *n_frames) {
    SessionOut o;
    o.mode = SessionOut::kBeams;
    o.beams = beams_out;
    return stream_maps(h, max_frames, power_out, o, first_frame, n_frames, "bflk_session_beams");
}

int bflk_session_targets(bflk_handle *h, int32_t max_frames, int32_t max_targets, float min_rel_power, float *power_out,
                         bflk_target *targets_out, int32_t *n_targets, int64_t *first_frame, int32_t *n_frames) {
    SessionOut o;
    o.mode = SessionOut::kTargets;
    o.targets = targets_out;
    o.n_targets = n_targets;
    o.max_targets = max_targets;
    o.min_rel = min_rel_power;
    return stream_maps(h, max_frames, power_out, o, first_frame, n_frames, "bflk_session_targets");
}

int bflk_stream_discard(bflk_handle *h, int32_t keep) {
    if (!h) return BFLK_ERR_INVALID;
    Session *s = session_of(h, "bflk_stream_discard");
    if (!s) return BFLK_ERR_STATE;
    if (keep < 0) return h->fail(BFLK_ERR_INVALID, "bflk_stream_discard: keep = %d", keep);
    const int64_t drop = ready_frames(h, s) - keep;
    if (drop > 0) {
        s->next_frame += drop;
        s->skipped += drop;
    }
    return BFLK_OK;
}

int bflk_stream_status(const bflk_handle *hc, int64_t *pushed, int64_t *next_frame, int32_t *ready, int64_t *skipped) {
    bflk_handle *h = const_cast<bflk_handle *>(hc);   // for the error message only
    if (!h) return BFLK_ERR_INVALID;
    const Session *s = session_of(h, "bflk_stream_status");
    if (!s) return BFLK_ERR_STATE;
    if (pushed) *pushed = s->pushed;
    if (next_frame) *next_frame = s->next_frame;
    if (ready) *ready = (int32_t)ready_frames(h, s);
    if (skipped) *skipped = s->skipped;
    return BFLK_OK;
}

int bflk_stream_window(bflk_handle *h, int64_t frame) {
    if (!h) return BFLK_ERR_INVALID;
    Session *s = session_of(h, "bflk_stream_window");
    if (!s) return BFLK_ERR_STATE;
    const int64_t N = h->cfg.frame_len;
    if (frame < 0 || frame * N < s->pushed - s->cap || frame * N + N + frame_tail_samples(h) > s->pushed)
        return h->fail(BFLK_ERR_STATE, "bflk_stream_window: frame %lld is not in the ring (%lld samples pushed, %lld held)",
                       (long long)frame, (long long)s->pushed, (long long)std::min(s->pushed, s->cap));
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    BFLK_CUDA(h, cudaEventSynchronize(s->written));   // its samples are in the ring before a caller's stream reads them
    set_resident(h, s->ring.p + frame * N % s->cap, 2 * s->cap, frame);
    return BFLK_OK;
}

// ---- neighbours of the path ------------------------------------------------------------------------------------
int bflk_pin_host(void *ptr, size_t bytes) {
    if (!ptr || !bytes) return BFLK_ERR_INVALID;
    return cudaHostRegister(ptr, bytes, cudaHostRegisterDefault) == cudaSuccess ? BFLK_OK : BFLK_ERR_CUDA;
}

int bflk_unpin_host(void *ptr) {
    if (!ptr) return BFLK_ERR_INVALID;
    return cudaHostUnregister(ptr) == cudaSuccess ? BFLK_OK : BFLK_ERR_CUDA;
}

int bflk_heatmap(bflk_handle *h, const float *power, int32_t n, uint8_t *heat, int32_t *argmax, float *maxv) {
    if (!h) return BFLK_ERR_INVALID;
    if (n <= 0 || (!power && !(h->last_map_on_device && n == h->dir_count)))
        return h->fail(BFLK_ERR_INVALID, "bflk_heatmap: null / empty map (and no map of that size left on the device)");
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    if (power) BFLK_CUDA(h, h->d_post.reserve(n));
    BFLK_CUDA(h, h->d_misc.reserve(4 + (n + 3) / 4));
    BFLK_CUDA(h, h->p_misc.reserve(4));
    uint8_t *d_heat = reinterpret_cast<uint8_t *>(h->d_misc.p + 4);
    if (power) BFLK_CUDA(h, cudaMemcpyAsync(h->d_post.p, power, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, launch_heatmap(power ? h->d_post.p : h->d_maps.p, n, d_heat, h->d_misc.p, reinterpret_cast<float *>(h->d_misc.p + 1), h->stream));
    h->launches++;
    BFLK_CUDA(h, cudaMemcpyAsync(h->p_misc.p, h->d_misc.p, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (heat) BFLK_CUDA(h, cudaMemcpyAsync(heat, d_heat, n, cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    if (argmax) *argmax = h->p_misc.p[0];
    if (maxv) std::memcpy(maxv, &h->p_misc.p[1], sizeof(float));
    return BFLK_OK;
}

// cv::resize coefficient tables for one axis (INTER_LINEAR, 8-bit: shorts scaled by 2048).  The horizontal axis clamps
// the fraction to 0 where the two taps would leave the image, the vertical one keeps it and clips the row (as OpenCV does).
static void resize_axis(int isz, int osz, bool clamp, int32_t *ofs, int32_t *coef) {
    const double inv = (double)osz / (double)isz, scale = 1.0 / inv;
    for (int d = 0; d < osz; d++) {
        float f = (float)((d + 0.5) * scale - 0.5);
        int sx = (int)std::floor(f);
        f -= (float)sx;
        if (clamp) {
            if (sx < 0) { f = 0.f; sx = 0; }
            if (sx >= isz - 1) { f = 0.f; sx = isz - 1; }
        }
        const int a0 = (int)std::lrintf((1.f - f) * 2048.f), a1 = (int)std::lrintf(f * 2048.f);
        ofs[d] = sx;
        coef[d] = (a0 & 0xffff) | (a1 << 16);
    }
}

int bflk_resize_u8(bflk_handle *h, const uint8_t *src, int32_t rows, int32_t cols, int32_t out_rows, int32_t out_cols, uint8_t *dst) {
    if (!h) return BFLK_ERR_INVALID;
    if (!src || !dst || rows <= 0 || cols <= 0 || out_rows <= 0 || out_cols <= 0) return h->fail(BFLK_ERR_INVALID, "bflk_resize_u8: null / empty image");
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const size_t n_in = (size_t)rows * cols, n_out = (size_t)out_rows * out_cols, n_tab = 2 * (size_t)(out_rows + out_cols);
    BFLK_CUDA(h, h->d_bytes.reserve(n_in + n_out + 16));
    BFLK_CUDA(h, h->d_misc.reserve(n_tab));
    std::vector<int32_t> tab(n_tab);
    resize_axis(cols, out_cols, true, tab.data(), tab.data() + out_cols);
    resize_axis(rows, out_rows, false, tab.data() + 2 * out_cols, tab.data() + 2 * out_cols + out_rows);
    uint8_t *d_src = h->d_bytes.p, *d_dst = h->d_bytes.p + ((n_in + 15) & ~(size_t)15);
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_misc.p, tab.data(), n_tab * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, cudaMemcpyAsync(d_src, src, n_in, cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, launch_resize_u8(d_src, rows, cols, d_dst, out_rows, out_cols, h->d_misc.p, h->stream));
    h->launches++;
    BFLK_CUDA(h, cudaMemcpyAsync(dst, d_dst, n_out, cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    return BFLK_OK;
}

int bflk_targets(bflk_handle *h, const float *power, int32_t max_targets, float min_rel_power, bflk_target *out, int32_t *n_out) {
    if (!h) return BFLK_ERR_INVALID;
    if (!out || !n_out || max_targets <= 0 || max_targets > 256) return h->fail(BFLK_ERR_INVALID, "bflk_targets: need 1..256 output slots");
    if (!fov_grid(h) || h->dir_first != 0 || h->dir_count != h->n_dir)
        return h->fail(BFLK_ERR_STATE, "bflk_targets: needs a rows x cols grid (bflk_set_grid_fov) and the whole map on this handle");
    if (!power && !h->last_map_on_device) return h->fail(BFLK_ERR_STATE, "bflk_targets: no map given and none left on the device by bflk_power_map");
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const int D = h->n_dir;
    if (power) BFLK_CUDA(h, h->d_post.reserve(D));
    if (power) BFLK_CUDA(h, cudaMemcpyAsync(h->d_post.p, power, D * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    return host_targets(h, power ? h->d_post.p : h->d_maps.p, 1, max_targets, min_rel_power, out, n_out);
}

int bflk_calibrate(bflk_handle *h, const float *signals, int32_t window_len, float reference_power_level, int32_t *index,
                   float *correction, int32_t *usable, float *median_out, float *mean_out) {
    if (!h) return BFLK_ERR_INVALID;
    if (!signals || window_len <= 0 || !index || !usable) return h->fail(BFLK_ERR_INVALID, "bflk_calibrate: null arguments");
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const int E = 64;  // ELEMENTS, antenna.h:20
    BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));   // a caller's stream may still use d_window
    BFLK_CUDA(h, h->d_window.reserve((size_t)E * window_len));
    BFLK_CUDA(h, h->d_post.reserve(E));
    BFLK_CUDA(h, h->p_out.reserve(E));
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_window.p, signals, (size_t)E * window_len * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, launch_channel_power(h->d_window.p, E, window_len, h->d_post.p, h->stream));
    h->launches++;
    BFLK_CUDA(h, cudaMemcpyAsync(h->p_out.p, h->d_post.p, E * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    const float *power = h->p_out.p;
    // median gate, aw_processing_unit.cpp:144-185 (the "median" is (m[32] + m[33]) / 2 as written there)
    float mean = 0.0f;
    for (int s = 0; s < E; s++) mean += power[s];
    float medians[E];
    std::memcpy(medians, power, sizeof(medians));
    std::sort(medians, medians + E);
    float median = (medians[E / 2] + medians[E / 2 + 1]) / 2.0;
    int count = 0;
    for (int s = 0; s < E; s++) {
        float diff = std::fabs(power[s] - median);
        if (diff > 1e-4) {
        } else if (power[s] < median * 1e-3) {
        } else {
            index[count++] = s;
            mean += power[s];
        }
    }
    mean /= static_cast<float>(count);
    if (correction)
        for (int s = 0; s < count; s++) correction[s] = reference_power_level / power[index[s]];
    *usable = count;
    if (median_out) *median_out = median;
    if (mean_out) *mean_out = mean;
    return BFLK_OK;
}

int bflk_ingest_i32(bflk_handle *h, const int32_t *frames, int32_t n, int32_t n_sensors, float *exposure) {
    if (!h) return BFLK_ERR_INVALID;
    if (!frames || !exposure || n <= 0 || n_sensors <= 0 || n_sensors % 8)
        return h->fail(BFLK_ERR_INVALID, "bflk_ingest_i32: null buffers or n_sensors not a multiple of 8");
    BFLK_CUDA(h, cudaSetDevice(h->cfg.device));
    const size_t cnt = (size_t)n * n_sensors;
    BFLK_CUDA(h, cudaEventSynchronize(h->caller_event));   // a caller's stream may still use d_window
    BFLK_CUDA(h, h->d_misc.reserve(cnt));
    BFLK_CUDA(h, h->d_window.reserve(cnt));
    BFLK_CUDA(h, cudaMemcpyAsync(h->d_misc.p, frames, cnt * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    BFLK_CUDA(h, launch_ingest(h->d_misc.p, n, n_sensors, h->d_window.p, h->stream));
    h->launches++;
    BFLK_CUDA(h, cudaMemcpyAsync(exposure, h->d_window.p, cnt * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    BFLK_CUDA(h, cudaStreamSynchronize(h->stream));
    return BFLK_OK;
}

}  // extern "C"
