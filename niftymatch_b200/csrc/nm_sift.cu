// nm_sift.cu -- parameters, workspace and the batched detect+describe driver.
//
// Host-side equivalents of SiftParams (gpu/sift/siftparams.h:30-51), PyramidData
// (gpu/sift/pyramidata.cu:24-50, 94-123) and the client's per-octave loop around the
// seven functions of gpu/sift/siftfunctions.h, for a batch of frames on one stream with
// no host synchronisation inside nm_sift_run.
#include "nm_sift_internal.cuh"
#include "nm_pyramid.cuh"
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#define NM_MAX_CHUNKS 64
#define NM_AUX_STREAMS 4      // nm_sift_run_host: stages rotate over up to 4 internal compute streams forked from the caller's

struct nm_sift_ctx {
    nm_sift_params P;
    int B, capacity, n_oct;
    NmOctaveTable tab;
    struct TmaSet {          // TMA descriptors of the internal levels for frames [first, first + n)
        int first, n;
        NmBlurTma lvl[NM_MAX_OCTAVES][5];   // source level i of octave o, box for radius radii[i+1]
        NmBlurTma ex[NM_MAX_OCTAVES];       // the six levels of octave o, box of the extrema kernel
    };
    std::vector<TmaSet*> tma_sets;
    cudaStream_t s_in, s_out, s_aux[NM_AUX_STREAMS];   // nm_sift_run_host: H2D / D2H copy streams, extra compute streams
    cudaEvent_t ev_fork, ev_join[NM_AUX_STREAMS];
    cudaStream_t s_side;                               // nm_sift_run: pyramids of octaves 1.. beside octave 0's last two levels
    cudaEvent_t ev_side_fork, ev_side_join;
    cudaEvent_t ev_in[NM_MAX_CHUNKS], ev_done[NM_MAX_CHUNKS], ev_out;
    // nm_sift_run_host: the ~47 launches of a pipeline stage replayed as one CUDA graph.  A stage's launch
    // sequence depends only on (first frame, frame count, mask texture, descriptor mode): captured once per key.
    struct StageGraph {
        cudaGraphExec_t exec = nullptr;
        int f0 = -1, n = 0, exact = 0, launches = 0;
        unsigned long long mask = 0;
    } stage_graph[NM_MAX_CHUNKS];
    float* taps[6];          // 0: base kernel, 1..5: level kernels (device)
    float  taps_host[6][96]; // the same values on the host (kernel parameters of the streaming blur)
    int    radii[6];
    int *seg_raw, *seg_cnt, *seg_off, *counts, *meta;
    float4* kpts;
    float2* orient;
    float *desc, *x, *y;
    float* frames_stage;     // device staging for nm_sift_run_host: [B][h][w]
    float* scratch;          // row-pass buffer of the generic blur, [B][h][w]; allocated when a radius exceeds 16
    int exact_desc;
    int dense_grad;          // 1: gradient maps computed everywhere (tests / tools that read them), 0: only where keypoint windows read
    unsigned long long mask_tex;   // detector mask (0 = none); mask_arr/mask_own: texture made by nm_sift_set_mask_image
    cudaArray_t mask_arr;
    cudaTextureObject_t mask_own;
    int last_launches;
    int timing;
    cudaEvent_t ev[7];
    std::vector<void*> allocs;
};

namespace {

template <typename T>
int dev_alloc(nm_sift_ctx* c, T** p, size_t count)
{
    void* q = nullptr;
    if (cudaMalloc(&q, count * sizeof(T)) != cudaSuccess) { cudaGetLastError(); return NM_ERR_ALLOC; }
    c->allocs.push_back(q);
    *p = static_cast<T*>(q);
    return NM_OK;
}

} // namespace

cudaError_t nm_ws_alloc(void** p, size_t bytes, cudaStream_t stream)
{
    static std::atomic<cudaMemPool_t> pools[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaMallocAsync(p, bytes, stream);
    cudaMemPool_t pool = pools[dev].load(std::memory_order_acquire);
    if (pool == nullptr) {
        cudaMemPoolProps props;
        std::memset(&props, 0, sizeof(props));
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev;
        cudaMemPool_t fresh = nullptr;
        if ((e = cudaMemPoolCreate(&fresh, &props)) != cudaSuccess) return e;
        unsigned long long keep = ~0ull;                       // keep freed blocks: the workspaces recur every call
        cudaMemPoolSetAttribute(fresh, cudaMemPoolAttrReleaseThreshold, &keep);
        cudaMemPool_t expected = nullptr;
        if (pools[dev].compare_exchange_strong(expected, fresh, std::memory_order_acq_rel)) pool = fresh;
        else { cudaMemPoolDestroy(fresh); pool = expected; }   // another host thread was first
    }
    return cudaMallocFromPoolAsync(p, bytes, pool, stream);
}

extern "C" const char* nm_version(void) { return "nm-b200 0.1 (sm_100a)"; }

extern "C" const char* nm_strerror(int code)
{
    switch (code) {
        case NM_OK: return "ok";
        case NM_ERR_INVALID: return "invalid argument";
        case NM_ERR_ALLOC: return "allocation failed";
        case NM_ERR_OVERFLOW: return "index range overflow";
        case NM_ERR_UNSUPPORTED: return "unsupported";
        case NM_ERR_NO_DEVICE: return "no sm_100 CUDA device";
        default: break;
    }
    if (code >= NM_ERR_CUDA_BASE) return cudaGetErrorString((cudaError_t)(code - NM_ERR_CUDA_BASE));
    return "unknown error";
}

extern "C" int nm_device_cc(void)
{
    int dev = 0, n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return NM_ERR_NO_DEVICE; }
    NM_CUDA_TRY(cudaGetDevice(&dev));
    int major = 0, minor = 0;
    NM_CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    NM_CUDA_TRY(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
    return major * 10 + minor;
}

// SiftParams(width, height): gpu/sift/siftparams.h:30-51, same mixed float/double steps.
extern "C" int nm_sift_params_init(nm_sift_params* p, int width, int height)
{
    if (!p || width <= 0 || height <= 0) return NM_ERR_INVALID;
    std::memset(p, 0, sizeof(*p));
    p->width = width; p->height = height;
    p->num_dog_levels = 3; p->sigma_n = 0.5f; p->peak_threshold = 0.f; p->edge_threshold = 10.f;
    p->level_max = p->num_dog_levels + 1;
    p->level_min = -1;
    p->num_octaves = (int)std::floor(std::log(std::min(width, height) * 2.0 / 32) / std::log(2.0));
    if (p->num_octaves <= 0) p->num_octaves = 1;
    p->sigma_k = std::pow(2.0f, 1.0f / p->num_dog_levels);
    p->sigma_0 = 1.6f * p->sigma_k;
    p->sigma_d_0 = (float)(p->sigma_0 * std::sqrt(1.0 - 1.0 / (p->sigma_k * p->sigma_k)));
    const float sa = (float)(p->sigma_0 * std::pow((double)p->sigma_k, (double)p->level_min));
    const float sb = p->sigma_n;
    if (sa > sb) p->base_smooth = std::sqrt(sa * sa - sb * sb);
    p->num_sigmas = 0;
    for (int i = p->level_min + 1; i <= p->level_max && p->num_sigmas < 8; ++i)
        p->sigmas[p->num_sigmas++] = (float)(p->sigma_d_0 * std::pow((double)p->sigma_k, (double)i));
    return NM_OK;
}

// PyramidData::create_kernel_for_sigma: gpu/sift/pyramidata.cu:105-123.
extern "C" int nm_gaussian_taps(float sigma, float* taps_host, int* radius)
{
    if (!taps_host || !radius || !(sigma > 0.f)) return NM_ERR_INVALID;
    const int r = (int)std::ceil(sigma * 4);
    if (2 * r + 1 > 91) return NM_ERR_INVALID;                   // MAX_KERNEL_LENGTH, pyramidata.h:9
    float sum = 0.f;
    for (int j = 0; j < 2 * r + 1; ++j) {
        float val = ((float)j - r) / sigma;
        val = (float)std::exp(-0.5 * (val * val));
        taps_host[j] = val;
        sum += val;
    }
    for (int j = 0; j < 2 * r + 1; ++j) taps_host[j] = taps_host[j] / sum;
    *radius = r;
    return NM_OK;
}

static void release_own_mask(nm_sift_ctx* c)
{
    if (c->mask_own) { if (c->mask_tex == c->mask_own) c->mask_tex = 0; cudaDestroyTextureObject(c->mask_own); c->mask_own = 0; }
    if (c->mask_arr) { cudaFreeArray(c->mask_arr); c->mask_arr = nullptr; }
}

extern "C" int nm_sift_destroy(nm_sift_ctx* c)
{
    if (!c) return NM_OK;
    release_own_mask(c);
    for (void* p : c->allocs) cudaFree(p);
    for (int i = 0; i < 7; ++i) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    for (auto* t : c->tma_sets) delete t;
    for (int i = 0; i < NM_MAX_CHUNKS; ++i) {
        if (c->stage_graph[i].exec) cudaGraphExecDestroy(c->stage_graph[i].exec);
        if (c->ev_in[i]) cudaEventDestroy(c->ev_in[i]);
        if (c->ev_done[i]) cudaEventDestroy(c->ev_done[i]);
    }
    if (c->ev_out) cudaEventDestroy(c->ev_out);
    if (c->s_in) cudaStreamDestroy(c->s_in);
    if (c->s_out) cudaStreamDestroy(c->s_out);
    for (int i = 0; i < NM_AUX_STREAMS; ++i) {
        if (c->s_aux[i]) cudaStreamDestroy(c->s_aux[i]);
        if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]);
    }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->s_side) cudaStreamDestroy(c->s_side);
    if (c->ev_side_fork) cudaEventDestroy(c->ev_side_fork);
    if (c->ev_side_join) cudaEventDestroy(c->ev_side_join);
    delete c;
    return NM_OK;
}

extern "C" int nm_sift_create(nm_sift_ctx** out, const nm_sift_params* params, int max_batch, int capacity)
{
    if (!out || !params || max_batch <= 0 || capacity <= 0) return NM_ERR_INVALID;
    const nm_sift_params& P = *params;
    if (P.width <= 0 || P.height <= 0 || P.num_octaves <= 0 || P.num_octaves > NM_MAX_OCTAVES ||
        P.num_dog_levels != 3 || P.num_sigmas != 5)
        return NM_ERR_INVALID;
    if ((P.width >> (P.num_octaves - 1)) < 3 || (P.height >> (P.num_octaves - 1)) < 3) return NM_ERR_INVALID;
    const int cc = nm_device_cc();
    if (cc < 0) return cc;
    if (cc / 10 != 10) return NM_ERR_NO_DEVICE;
    nm_sift_ctx* c = new (std::nothrow) nm_sift_ctx();
    if (!c) return NM_ERR_ALLOC;
    c->P = P; c->B = max_batch; c->capacity = capacity; c->n_oct = P.num_octaves;
    c->scratch = nullptr; c->exact_desc = 0; c->dense_grad = 0; c->last_launches = 0; c->timing = 0;
    c->mask_tex = 0; c->mask_arr = nullptr; c->mask_own = 0;
    for (int i = 0; i < 7; ++i) c->ev[i] = nullptr;
    c->s_in = c->s_out = nullptr; c->ev_out = c->ev_fork = nullptr;
    c->s_side = nullptr; c->ev_side_fork = c->ev_side_join = nullptr;
    for (int i = 0; i < NM_AUX_STREAMS; ++i) { c->s_aux[i] = nullptr; c->ev_join[i] = nullptr; }
    for (int i = 0; i < NM_MAX_CHUNKS; ++i) c->ev_in[i] = c->ev_done[i] = nullptr;
    int rc = NM_OK;
    // Gaussian kernels
    for (int i = 0; i < 6 && rc == NM_OK; ++i) {
        float* host = c->taps_host[i];
        rc = nm_gaussian_taps(i == 0 ? P.base_smooth : P.sigmas[i - 1], host, &c->radii[i]);
        if (rc != NM_OK) break;
        rc = dev_alloc(c, &c->taps[i], 96);
        if (rc == NM_OK && cudaMemcpy(c->taps[i], host, sizeof(float) * (2 * c->radii[i] + 1), cudaMemcpyHostToDevice) != cudaSuccess)
            rc = NM_ERR_ALLOC;
    }
    c->tab.n_oct = c->n_oct;
    const size_t B = (size_t)max_batch;
    for (int o = 0; o < c->n_oct && rc == NM_OK; ++o) {
        NmOctave& oc = c->tab.o[o];
        oc.w = P.width >> o; oc.h = P.height >> o;
        oc.pitch = (oc.w + 31) / 32 * 32;
        oc.wpr = (oc.w + 31) / 32;
        oc.level_elems = (long long)oc.h * oc.pitch;
        oc.xper = (float)std::pow(2.0, o);                        // siftfunctions.cu:118
        const size_t nwords = (size_t)oc.h * oc.wpr;
        if (rc == NM_OK) rc = dev_alloc(c, &oc.levels, B * 6 * (size_t)oc.level_elems);
        if (rc == NM_OK) rc = dev_alloc(c, &oc.grad, B * 3 * (size_t)oc.level_elems);
        if (rc == NM_OK) rc = dev_alloc(c, &oc.bitmap, B * 3 * nwords);
        if (rc == NM_OK) rc = dev_alloc(c, &oc.wprefix, B * 3 * nwords);
        if (rc == NM_OK) rc = dev_alloc(c, &oc.need, B * 3 * (size_t)nm_div_up(oc.h, 8) * oc.wpr);
        const size_t tiles = (size_t)nm_div_up(oc.w, 32) * nm_div_up(oc.h, 32);
        if (rc == NM_OK) rc = dev_alloc(c, &oc.cand_n, B * tiles);
        if (rc == NM_OK) rc = dev_alloc(c, &oc.cand, B * tiles * 32);
    }
    const size_t S = (size_t)c->n_oct * 3, cap = (size_t)capacity;
    if (rc == NM_OK) rc = dev_alloc(c, &c->seg_raw, B * S);
    if (rc == NM_OK) rc = dev_alloc(c, &c->seg_cnt, B * S);
    if (rc == NM_OK) rc = dev_alloc(c, &c->seg_off, B * S);
    if (rc == NM_OK) rc = dev_alloc(c, &c->counts, B);
    if (rc == NM_OK) rc = dev_alloc(c, &c->meta, B * cap);
    if (rc == NM_OK) rc = dev_alloc(c, &c->kpts, B * cap);
    if (rc == NM_OK) rc = dev_alloc(c, &c->orient, B * cap);
    if (rc == NM_OK) rc = dev_alloc(c, &c->desc, B * cap * 128);
    if (rc == NM_OK) rc = dev_alloc(c, &c->x, B * cap);
    if (rc == NM_OK) rc = dev_alloc(c, &c->y, B * cap);
    if (rc == NM_OK) rc = dev_alloc(c, &c->frames_stage, B * (size_t)P.width * P.height);
    // radii above 16 (sigma > 4; the reference allows up to 45, MAX_KERNEL_LENGTH 91) take the generic two-pass blur,
    // which needs a row-pass buffer: [B][h][w] of octave 0 covers every octave
    bool wide = false;
    for (int i = 0; i < 6; ++i) wide = wide || c->radii[i] > 16;
    if (rc == NM_OK && wide) rc = dev_alloc(c, &c->scratch, B * (size_t)P.width * P.height);
    if (rc == NM_OK) {
        // descriptor slots start at 0 like SiftData::initialize_data (siftdata.cu:34)
        if (cudaMemset(c->desc, 0, B * cap * 128 * sizeof(float)) != cudaSuccess) rc = NM_ERR_ALLOC;
        cudaMemset(c->counts, 0, B * sizeof(int));
        cudaMemset(c->seg_cnt, 0, B * S * sizeof(int));
    }
    for (int i = 0; i < 7 && rc == NM_OK; ++i)
        if (cudaEventCreate(&c->ev[i]) != cudaSuccess) rc = NM_ERR_ALLOC;
    if (rc == NM_OK && (cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking) != cudaSuccess ||
                        cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking) != cudaSuccess ||
                        cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
                        cudaEventCreateWithFlags(&c->ev_out, cudaEventDisableTiming) != cudaSuccess))
        rc = NM_ERR_ALLOC;
    if (rc == NM_OK && (cudaStreamCreateWithFlags(&c->s_side, cudaStreamNonBlocking) != cudaSuccess ||
                        cudaEventCreateWithFlags(&c->ev_side_fork, cudaEventDisableTiming) != cudaSuccess ||
                        cudaEventCreateWithFlags(&c->ev_side_join, cudaEventDisableTiming) != cudaSuccess))
        rc = NM_ERR_ALLOC;
    for (int i = 0; i < NM_AUX_STREAMS && rc == NM_OK; ++i)
        if (cudaStreamCreateWithFlags(&c->s_aux[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming) != cudaSuccess)
            rc = NM_ERR_ALLOC;
    for (int i = 0; i < NM_MAX_CHUNKS && rc == NM_OK; ++i)
        if (cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ev_done[i], cudaEventDisableTiming) != cudaSuccess)
            rc = NM_ERR_ALLOC;
    if (rc != NM_OK) { nm_sift_destroy(c); return rc; }
    *out = c;
    return NM_OK;
}

// Detect + describe for the frames [first, first + n) of the workspace (frames_dev = the first of
// those n frames).  All kernels index frames by block, so a range is the same launch sequence on
// pointers advanced to the range's first frame.
static int sift_run_range(nm_sift_ctx* c, const float* frames_dev, int first, int n, cudaStream_t st, bool timing,
                          bool bgra = false, bool side_octaves = false)
{
    const nm_sift_params& P = c->P;
    int launches = 0, rc;
    NmDetectParams dp{P.peak_threshold, P.edge_threshold, P.sigma_0, P.num_dog_levels, c->mask_tex};
    // workspace views of the range
    NmOctaveTable tab = c->tab;
    for (int o = 0; o < c->n_oct; ++o) {
        NmOctave& oc = tab.o[o];
        const long long nwords = (long long)oc.h * oc.wpr;
        oc.levels += (long long)first * 6 * oc.level_elems;
        oc.grad += (long long)first * 3 * oc.level_elems;
        oc.bitmap += (long long)first * 3 * nwords;
        oc.wprefix += (long long)first * 3 * nwords;
        oc.need += (long long)first * 3 * nm_div_up(oc.h, 8) * oc.wpr;
        const long long tiles = (long long)nm_div_up(oc.w, 32) * nm_div_up(oc.h, 32);
        oc.cand_n += first * tiles;
        oc.cand += first * tiles * 32;
    }
    const long long S = (long long)c->n_oct * 3, cap = c->capacity;
    int* seg_raw = c->seg_raw + first * S;
    int* seg_cnt = c->seg_cnt + first * S;
    int* seg_off = c->seg_off + first * S;
    int* counts = c->counts + first;
    int* meta = c->meta + first * cap;
    float4* kpts = c->kpts + first * cap;
    float2* orient = c->orient + first * cap;
    float* desc = c->desc + first * cap * 128;
    float* x = c->x + first * cap;
    float* y = c->y + first * cap;
    // cached TMA descriptors of the internal levels for this range
    nm_sift_ctx::TmaSet* ts = nullptr;
    for (auto* t : c->tma_sets) if (t->first == first && t->n == n) { ts = t; break; }
    if (!ts) {
        ts = new (std::nothrow) nm_sift_ctx::TmaSet();
        if (!ts) return NM_ERR_ALLOC;
        ts->first = first; ts->n = n;
        for (int o = 0; o < c->n_oct; ++o) {
            const NmOctave& oc = tab.o[o];
            for (int i = 0; i < 5; ++i)
                nm_blur_make_tma(&ts->lvl[o][i], oc.levels + i * oc.level_elems, oc.w, oc.h, oc.pitch,
                                 6 * oc.level_elems, n, c->radii[i + 1]);
            nm_extrema_make_tma(&ts->ex[o], oc, n);
        }
        c->tma_sets.push_back(ts);
    }
    if (timing) cudaEventRecord(c->ev[0], st);
    // ---- pyramid ---------------------------------------------------------------
    // side_octaves (large device-resident batches): octave 1's base is ready after octave 0's level 3, so the pyramids
    // of octaves 1.. run on a second stream beside octave 0's two widest blurs -- the launches of octaves 3+ are a
    // fraction of a wave each and would otherwise run alone, one after the other.
    auto level_blur = [&](int o, int i, cudaStream_t s) -> int {
        const NmOctave& oc = tab.o[o];
        const long long fstride = 6 * oc.level_elems;
        NmBlurArgs a{};
        a.src = oc.levels + i * oc.level_elems; a.src_pitch = oc.pitch; a.src_fstride = fstride;
        a.dst = oc.levels + (i + 1) * oc.level_elems; a.dst_pitch = oc.pitch; a.dst_fstride = fstride;
        a.taps = c->taps[i + 1]; a.taps_host = c->taps_host[i + 1]; a.radius = c->radii[i + 1]; a.w = oc.w; a.h = oc.h;
        a.batch = n;
        a.scratch = c->scratch ? c->scratch + (long long)first * P.width * P.height : nullptr;
        if (i + 1 == P.num_dog_levels && o + 1 < c->n_oct) {
            // level 3 (sigma doubled) decimated by 2 = next octave's level 0 (downsample.cu:15-16)
            const NmOctave& nx = tab.o[o + 1];
            a.dst2 = nx.levels; a.dst2_pitch = nx.pitch; a.dst2_fstride = 6 * nx.level_elems;
        }
        ++launches;
        return nm_blur_launch(a, s, &ts->lvl[o][i]);
    };
    {
        const NmOctave& oc = tab.o[0];
        NmBlurArgs a{};
        a.src = frames_dev; a.src_pitch = P.width; a.src_fstride = (long long)P.width * P.height;
        a.dst = oc.levels; a.dst_pitch = oc.pitch; a.dst_fstride = 6 * oc.level_elems;
        a.taps = c->taps[0]; a.taps_host = c->taps_host[0]; a.radius = c->radii[0]; a.w = oc.w; a.h = oc.h; a.batch = n;
        a.scratch = c->scratch ? c->scratch + (long long)first * P.width * P.height : nullptr;
        NmBlurTma base;
        nm_blur_make_tma(&base, frames_dev, P.width, P.height, P.width, (long long)P.width * P.height, n, c->radii[0], bgra);
        a.src_bgra = bgra ? 1 : 0;
        if (bgra && !nm_blur_uses_strip(a, &base)) {
            // small launch: the tile kernels do not convert -- grey frames through the staging buffer first
            float* gray = c->frames_stage + (long long)first * P.width * P.height;
            if ((rc = nm_grayscale_launch(frames_dev, gray, (long long)n * P.width * P.height, st)) != NM_OK) return rc;
            launches += 1;
            a.src = gray; a.src_bgra = 0;
            nm_blur_make_tma(&base, gray, P.width, P.height, P.width, (long long)P.width * P.height, n, c->radii[0]);
        }
        if ((rc = nm_blur_launch(a, st, &base)) != NM_OK) return rc;
        ++launches;
    }
    const bool side = side_octaves && c->n_oct >= 2 && P.num_dog_levels < 5 && c->s_side != nullptr;
    for (int o = 0; o < c->n_oct; ++o) {
        cudaStream_t so = (side && o >= 1) ? c->s_side : st;
        for (int i = 0; i < 5; ++i) {
            if ((rc = level_blur(o, i, so)) != NM_OK) return rc;
            if (side && o == 0 && i + 1 == P.num_dog_levels) {
                // octave 1's base is written: the other octaves start on the side stream
                NM_CUDA_TRY(cudaEventRecord(c->ev_side_fork, st));
                NM_CUDA_TRY(cudaStreamWaitEvent(c->s_side, c->ev_side_fork, 0));
            }
        }
    }
    if (side) {
        NM_CUDA_TRY(cudaEventRecord(c->ev_side_join, c->s_side));
        NM_CUDA_TRY(cudaStreamWaitEvent(st, c->ev_side_join, 0));
    }
    if (timing) cudaEventRecord(c->ev[1], st);
    // ---- DoG + extrema + refinement -----------------------------------------------------
    for (int o = 0; o < c->n_oct; ++o) {
        if ((rc = nm_extrema_launch(tab.o[o], dp, n, st, &ts->ex[o])) != NM_OK) return rc;
        launches += 2;
    }
    if (timing) cudaEventRecord(c->ev[2], st);
    // ---- ordered compaction (kprefine also marks the gradient blocks the keypoint windows read) ----
    if ((rc = nm_rank_launch(tab, n, seg_raw, st)) != NM_OK) return rc;
    if ((rc = nm_plan_launch(seg_raw, seg_cnt, seg_off, counts, c->n_oct, n, c->capacity, st)) != NM_OK) return rc;
    launches += 2;
    for (int o = 0; o < c->n_oct; ++o) {
        if ((rc = nm_emit_launch(tab.o[o], o, c->n_oct, n, seg_cnt, seg_off, c->capacity, kpts, meta, st)) != NM_OK) return rc;
        ++launches;
    }
    if ((rc = nm_kprefine_launch(tab, dp, n, c->capacity, counts, kpts, meta, st)) != NM_OK) return rc;
    ++launches;
    if (timing) cudaEventRecord(c->ev[3], st);
    // ---- gradient maps of the marked blocks ----------------------------------------------
    if ((rc = nm_gradmap_launch(tab, n, c->dense_grad, st)) != NM_OK) return rc;
    launches += c->n_oct;
    if (timing) cudaEventRecord(c->ev[4], st);
    // ---- orientation, descriptor -----------------------------------------------------
    if ((rc = nm_orient_launch(tab, n, c->capacity, counts, kpts, meta, orient, st)) != NM_OK) return rc;
    ++launches;
    if (timing) cudaEventRecord(c->ev[5], st);
    if ((rc = nm_describe_launch(tab, n, c->capacity, counts, kpts, meta, orient, desc, x, y, P.num_dog_levels,
                                 c->exact_desc, st)) != NM_OK) return rc;
    ++launches;
    if (timing) cudaEventRecord(c->ev[6], st);
    c->last_launches = launches;
    return NM_OK;
}

extern "C" int nm_sift_run_bgra(nm_sift_ctx* c, const void* frames_bgra_dev, int n_frames, nm_stream_t stream)
{
    if (!c || !frames_bgra_dev || n_frames <= 0 || n_frames > c->B) return NM_ERR_INVALID;
    if (reinterpret_cast<uintptr_t>(frames_bgra_dev) & 3) return NM_ERR_INVALID;
    return sift_run_range(c, static_cast<const float*>(frames_bgra_dev), 0, n_frames, (cudaStream_t)stream, c->timing != 0, true);
}

extern "C" int nm_sift_run(nm_sift_ctx* c, const float* frames_dev, int n_frames, nm_stream_t stream)
{
    if (!c || !frames_dev || n_frames <= 0 || n_frames > c->B) return NM_ERR_INVALID;
    // octaves 1.. beside octave 0's last levels when octave 0 alone fills the device for a while
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    const bool cap_ok = cudaStreamIsCapturing((cudaStream_t)stream, &cap) == cudaSuccess;
    if (!cap_ok) cudaGetLastError();
    const bool side = cap_ok && cap == cudaStreamCaptureStatusNone &&
                      (long long)n_frames * c->P.width * c->P.height >= 16LL * 1920 * 1080;
    // (measured and not kept: the two halves of the batch as two ranges on two streams, 7.24 -> 7.16 ms per 64 frames)
    return sift_run_range(c, frames_dev, 0, n_frames, (cudaStream_t)stream, c->timing != 0, false, side);
}

// End to end from host memory, software pipelined in stages of a few frames: the H2D copy
// of chunk k+1 (stream s_in), the kernels of chunk k (caller's stream) and the D2H copies of chunk
// k-1 (stream s_out) overlap; the host only waits for a chunk's 4-byte counts before it sizes that
// chunk's result copies.  Host buffers should be pinned for the copies to be asynchronous.
extern "C" int nm_sift_run_host(nm_sift_ctx* c, const float* frames_host, int n_frames, int* counts_host,
                                float* desc_host, float* x_host, float* y_host, nm_stream_t stream)
{
    if (!c || !frames_host || !counts_host || n_frames <= 0 || n_frames > c->B) return NM_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t fpix = (size_t)c->P.width * c->P.height;
    // Pipeline stages: the uploads pace the pipeline (1080p: 6.7 frames/ms over PCIe against 7.5 frames/ms of
    // kernels at full batch), so the end-to-end time is (all uploads) + (what the kernels still have to do when
    // the last frame lands).  Small stages keep that tail short; their under-filled launches (octaves 2+ are a
    // fraction of a wave) are covered by running up to four stages concurrently on separate streams, and their
    // launch cost by replaying each stage as one CUDA graph.  Measured at 64 x 1080p, 4 streams, graphs:
    // stages of 3 frames 11.45 ms, 4: 11.67, 5: 11.60, 6: 11.73, 8: 12.16 (uploads alone: 9.58 ms);
    // without graphs 6-frame stages were best at 12.33 (B200).
    constexpr int stage = 3;
    int bounds[NM_MAX_CHUNKS + 1];
    int n_chunks = 0;
    bounds[0] = 0;
    if (n_frames <= 8) {
        bounds[++n_chunks] = n_frames;
    } else {
        // uniform stages, tapered at the end (2, 1, 1 frames): what remains to be done when the LAST frame has landed
        // is that frame's kernels and its result copy, not a whole 3-frame stage
        const int per = std::max(stage, nm_div_up(n_frames, NM_MAX_CHUNKS - 4));
        int f = 0;
        while (f < n_frames) {
            const int left = n_frames - f;
            int take = per;
            if (left <= per + 1) take = left >= 3 ? 2 : 1;
            if (take > left) take = left;
            f += take;
            bounds[++n_chunks] = f;
        }
    }
    if (n_chunks > NM_MAX_CHUNKS) return NM_ERR_INVALID;
    int launches = 0;
    auto drain = [&](int k) -> int {
        // results of chunk k: wait for its counts, then copy the filled part of every frame
        NM_CUDA_TRY(cudaEventSynchronize(c->ev_done[k]));
        for (int f = bounds[k]; f < bounds[k + 1]; ++f) {
            const size_t n = (size_t)counts_host[f], off = (size_t)f * c->capacity;
            if (n == 0) continue;
            if (desc_host) NM_CUDA_TRY(cudaMemcpyAsync(desc_host + off * 128, c->desc + off * 128, n * 128 * sizeof(float), cudaMemcpyDeviceToHost, c->s_out));
            if (x_host) NM_CUDA_TRY(cudaMemcpyAsync(x_host + off, c->x + off, n * sizeof(float), cudaMemcpyDeviceToHost, c->s_out));
            if (y_host) NM_CUDA_TRY(cudaMemcpyAsync(y_host + off, c->y + off, n * sizeof(float), cudaMemcpyDeviceToHost, c->s_out));
        }
        return NM_OK;
    };
    for (int k = 0; k < n_chunks; ++k) {        // the uploads do not depend on anything: queue them all
        const int f0 = bounds[k], n = bounds[k + 1] - bounds[k];
        NM_CUDA_TRY(cudaMemcpyAsync(c->frames_stage + f0 * fpix, frames_host + f0 * fpix, fpix * n * sizeof(float),
                                    cudaMemcpyHostToDevice, c->s_in));
        NM_CUDA_TRY(cudaEventRecord(c->ev_in[k], c->s_in));
    }
    // stages rotate over the internal compute streams: the launch-bound tail of one stage (small octaves,
    // orientation) overlaps the big blur kernels of the next; the host may only block on a stage once the next
    // n_streams - 1 stages are queued behind it
    constexpr int n_streams = NM_AUX_STREAMS, lag = n_streams > 1 ? n_streams - 1 : 1;
    // with several stages the launches of a stage are replayed as one CUDA graph (11 stages x 47 launches per
    // 64-frame call otherwise)
    const bool use_graphs = n_chunks > 1;
    NM_CUDA_TRY(cudaEventRecord(c->ev_fork, st));
    // every stage runs on an internal stream (the caller's may be the legacy default stream, which cannot be captured)
    for (int i = 0; i < n_streams; ++i) NM_CUDA_TRY(cudaStreamWaitEvent(c->s_aux[i], c->ev_fork, 0));
    for (int k = 0; k < n_chunks; ++k) {
        const int f0 = bounds[k], n = bounds[k + 1] - bounds[k];
        cudaStream_t sk = c->s_aux[k % n_streams];
        NM_CUDA_TRY(cudaStreamWaitEvent(sk, c->ev_in[k], 0));
        int rc;
        if (use_graphs) {
            nm_sift_ctx::StageGraph& g = c->stage_graph[k];
            if (!g.exec || g.f0 != f0 || g.n != n || g.mask != c->mask_tex || g.exact != (c->exact_desc | (c->dense_grad << 1))) {
                if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
                cudaGraph_t graph = nullptr;
                NM_CUDA_TRY(cudaStreamBeginCapture(sk, cudaStreamCaptureModeThreadLocal));
                rc = sift_run_range(c, c->frames_stage + f0 * fpix, f0, n, sk, false);
                const cudaError_t ce = cudaStreamEndCapture(sk, &graph);
                if (rc != NM_OK || ce != cudaSuccess) {
                    if (graph) cudaGraphDestroy(graph);
                    return rc != NM_OK ? rc : nm_cuda_err(ce);
                }
                const cudaError_t ie = cudaGraphInstantiate(&g.exec, graph, 0);
                cudaGraphDestroy(graph);
                if (ie != cudaSuccess) { g.exec = nullptr; return nm_cuda_err(ie); }
                g.f0 = f0; g.n = n; g.mask = c->mask_tex; g.exact = c->exact_desc | (c->dense_grad << 1); g.launches = c->last_launches;
            }
            NM_CUDA_TRY(cudaGraphLaunch(g.exec, sk));
            launches += g.launches;
        } else {
            rc = sift_run_range(c, c->frames_stage + f0 * fpix, f0, n, sk, false);
            if (rc != NM_OK) return rc;
            launches += c->last_launches;
        }
        NM_CUDA_TRY(cudaMemcpyAsync(counts_host + f0, c->counts + f0, sizeof(int) * n, cudaMemcpyDeviceToHost, sk));
        NM_CUDA_TRY(cudaEventRecord(c->ev_done[k], sk));
        if (k >= lag && (rc = drain(k - lag)) != NM_OK) return rc;
    }
    for (int k = n_chunks - lag; k < n_chunks; ++k) {
        if (k < 0) continue;
        int rc = drain(k);
        if (rc != NM_OK) return rc;
    }
    // the caller's stream is complete when all compute streams and the result copies are
    for (int i = 0; i < n_streams; ++i) {
        NM_CUDA_TRY(cudaEventRecord(c->ev_join[i], c->s_aux[i]));
        NM_CUDA_TRY(cudaStreamWaitEvent(st, c->ev_join[i], 0));
    }
    NM_CUDA_TRY(cudaEventRecord(c->ev_out, c->s_out));
    NM_CUDA_TRY(cudaStreamWaitEvent(st, c->ev_out, 0));
    NM_CUDA_TRY(cudaStreamSynchronize(st));
    c->last_launches = launches;
    return NM_OK;
}

// compute_keypoints_with_mask (gpu/sift/siftfunctions.cu:65-98) for the batched path: the caller's
// texture object, sampled at ((x+.5)*xper, (y+.5)*xper) in every octave (keypoint.cu:214).  0 = unmasked.
extern "C" int nm_sift_set_mask(nm_sift_ctx* c, unsigned long long tex_mask)
{
    if (!c) return NM_ERR_INVALID;
    if (tex_mask != c->mask_own) release_own_mask(c);
    c->mask_tex = tex_mask;
    return NM_OK;
}

// Convenience: bind a width x height float mask image (host or device memory) the way a reference client
// does -- a cudaArray behind a texture with the CudaTex2D settings (gpu/utils/cudatex2D.cu:12-19: border
// addressing, linear filter, unnormalised coordinates) and element-type reads.  The context owns it.
extern "C" int nm_sift_set_mask_image(nm_sift_ctx* c, const float* mask, int width, int height)
{
    if (!c || !mask || width <= 0 || height <= 0) return NM_ERR_INVALID;
    release_own_mask(c);
    cudaChannelFormatDesc fd = cudaCreateChannelDesc<float>();
    if (cudaMallocArray(&c->mask_arr, &fd, width, height) != cudaSuccess) { cudaGetLastError(); c->mask_arr = nullptr; return NM_ERR_ALLOC; }
    cudaError_t e = cudaMemcpy2DToArray(c->mask_arr, 0, 0, mask, (size_t)width * sizeof(float), (size_t)width * sizeof(float),
                                        height, cudaMemcpyDefault);
    if (e != cudaSuccess) { release_own_mask(c); return nm_cuda_err(e); }
    cudaResourceDesc rd; std::memset(&rd, 0, sizeof(rd));
    rd.resType = cudaResourceTypeArray; rd.res.array.array = c->mask_arr;
    cudaTextureDesc td; std::memset(&td, 0, sizeof(td));
    td.addressMode[0] = td.addressMode[1] = cudaAddressModeBorder;
    td.filterMode = cudaFilterModeLinear;
    td.readMode = cudaReadModeElementType;
    td.normalizedCoords = 0;
    e = cudaCreateTextureObject(&c->mask_own, &rd, &td, nullptr);
    if (e != cudaSuccess) { c->mask_own = 0; release_own_mask(c); return nm_cuda_err(e); }
    c->mask_tex = c->mask_own;
    return NM_OK;
}

extern "C" int nm_sift_results(nm_sift_ctx* c, const float** desc, const float** x, const float** y,
                               const int** counts, const float** kpts4, const float** orient2,
                               const int** seg_counts)
{
    if (!c) return NM_ERR_INVALID;
    if (desc) *desc = c->desc;
    if (x) *x = c->x;
    if (y) *y = c->y;
    if (counts) *counts = c->counts;
    if (kpts4) *kpts4 = reinterpret_cast<const float*>(c->kpts);
    if (orient2) *orient2 = reinterpret_cast<const float*>(c->orient);
    if (seg_counts) *seg_counts = c->seg_cnt;
    return NM_OK;
}

extern "C" int nm_sift_level(nm_sift_ctx* c, int frame, int octave, int level, const float** ptr, int* pitch,
                             int* w, int* h)
{
    if (!c || frame < 0 || frame >= c->B || octave < 0 || octave >= c->n_oct || level < 0 || level > 5) return NM_ERR_INVALID;
    const NmOctave& oc = c->tab.o[octave];
    if (ptr) *ptr = oc.levels + ((long long)frame * 6 + level) * oc.level_elems;
    if (pitch) *pitch = oc.pitch;
    if (w) *w = oc.w;
    if (h) *h = oc.h;
    return NM_OK;
}

extern "C" int nm_sift_grad(nm_sift_ctx* c, int frame, int octave, int level, const float** ptr2, int* pitch,
                            int* w, int* h)
{
    if (!c || frame < 0 || frame >= c->B || octave < 0 || octave >= c->n_oct || level < 0 || level > 2) return NM_ERR_INVALID;
    const NmOctave& oc = c->tab.o[octave];
    if (ptr2) *ptr2 = reinterpret_cast<const float*>(oc.grad + ((long long)frame * 3 + level) * oc.level_elems);
    if (pitch) *pitch = oc.pitch;
    if (w) *w = oc.w;
    if (h) *h = oc.h;
    return NM_OK;
}

extern "C" int nm_sift_last_launches(nm_sift_ctx* c) { return c ? c->last_launches : NM_ERR_INVALID; }

extern "C" int nm_sift_enable_timing(nm_sift_ctx* c, int enable)
{
    if (!c) return NM_ERR_INVALID;
    c->timing = enable ? 1 : 0;
    return NM_OK;
}

// ms6 = {pyramid, extrema + gradient maps, compaction, orientation, descriptor, total} of the last timed run
extern "C" int nm_sift_stage_ms(nm_sift_ctx* c, float* ms6)
{
    float m[7];
    const int rc = nm_sift_stage_ms7(c, m);
    if (rc != NM_OK || !ms6) return rc != NM_OK ? rc : NM_ERR_INVALID;
    ms6[0] = m[0]; ms6[1] = m[1] + m[3]; ms6[2] = m[2]; ms6[3] = m[4]; ms6[4] = m[5]; ms6[5] = m[6];
    return NM_OK;
}

// ms7 = {pyramid, extrema, compaction, gradient maps, orientation, descriptor, total}
extern "C" int nm_sift_stage_ms7(nm_sift_ctx* c, float* ms7)
{
    if (!c || !ms7) return NM_ERR_INVALID;
    NM_CUDA_TRY(cudaEventSynchronize(c->ev[6]));
    for (int i = 0; i < 6; ++i) NM_CUDA_TRY(cudaEventElapsedTime(&ms7[i], c->ev[i], c->ev[i + 1]));
    NM_CUDA_TRY(cudaEventElapsedTime(&ms7[6], c->ev[0], c->ev[6]));
    return NM_OK;
}

// 1: gradient maps computed for every pixel (callers that read nm_sift_grad); 0 (default): only the 8 x 32 blocks an
// orientation / descriptor window of an emitted keypoint reads -- the results of the run are identical.
extern "C" int nm_sift_set_dense_gradients(nm_sift_ctx* c, int dense)
{
    if (!c) return NM_ERR_INVALID;
    c->dense_grad = dense ? 1 : 0;
    return NM_OK;
}

extern "C" int nm_sift_set_exact_descriptor(nm_sift_ctx* c, int exact)
{
    if (!c) return NM_ERR_INVALID;
    c->exact_desc = exact ? 1 : 0;
    return NM_OK;
}
