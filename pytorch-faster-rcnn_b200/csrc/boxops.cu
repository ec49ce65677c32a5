// boxops.cu -- K1 anchor grid, a2 masks, a3 IoU tables, K8 delta encode/decode.
// All HBM-write/read bound elementwise kernels: coalesced SoA rows, 128-bit
// stores where the row pitch allows, grids sized to the work (tiny launches).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>

#include "common.cuh"

namespace b2d {

static std::mutex g_err_mu;
static std::string g_err = "";

void set_error(const char* msg) {
    std::lock_guard<std::mutex> l(g_err_mu);
    g_err = msg ? msg : "";
}

static Knobs g_knobs;
static std::once_flag g_knobs_once;

static void load_knobs() {
    auto geti = [](const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; };
    Knobs k;
    k.dbg = geti("B2D_DBG", 0);
    k.rpn_chains = geti("B2D_RPN_CHAINS", 1);
    k.rpn_front = geti("B2D_RPN_FRONT", 1);
    k.rpn_back = geti("B2D_RPN_BACK", 1);
    { const char* e = getenv("B2D_NMS_CUT"); k.nms_cut = e ? atof(e) : 1.5; }
    k.nms_p1_chains = geti("B2D_NMS_P1_CHAINS", 0);
    k.nms_sweep = geti("B2D_NMS_SWEEP", 1);
    k.sweep_t = geti("B2D_SWEEP_T", 0);
    k.sweep_g = geti("B2D_SWEEP_G", 0);
    k.roi_bwd_tile = geti("B2D_ROI_BWD_TILE", 2);
    k.assign_old = getenv("B2D_ASSIGN_OLD") != nullptr;
    k.sample_threads = geti("B2D_SAMPLE_THREADS", 1024);
    k.pdl = geti("B2D_PDL", 0);           // measured r2: 258 vs 250 us per step with the edges on (DESIGN.md 6a)
    k.debug_sync = getenv("B2D_DEBUG_SYNC") != nullptr;
    g_knobs = k;
}

const Knobs& knobs() {
    std::call_once(g_knobs_once, load_knobs);
    return g_knobs;
}

int check_launch(const char* what) {
    if (knobs().debug_sync) cudaDeviceSynchronize();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        char buf[512];
        snprintf(buf, sizeof(buf), "%s: %s", what, cudaGetErrorString(e));
        set_error(buf);
        return (int)e;
    }
    return B2D_OK;
}

// ------------------------------------------------------------------ K1
// out [4][A*H*W]; one thread per anchor, 4 coalesced row stores.
__global__ void __launch_bounds__(256) k_anchor_grid(float* __restrict__ out, b2d_level lv, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Box b = anchor_flat(lv, (int)i);
    out[i] = b.x1; out[n + i] = b.y1; out[2 * n + i] = b.x2; out[3 * n + i] = b.y2;
}

__global__ void __launch_bounds__(256) k_inside_anchor_mask(uint8_t* __restrict__ mask,
                                                            const float* __restrict__ a, long long n,
                                                            float img_h, float img_w, float border) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool ok = true;
    if (border >= 0.0f)
        ok = a[i] >= -border && a[n + i] >= -border && a[2 * n + i] < img_w + border &&
             a[3 * n + i] < img_h + border;
    mask[i] = ok ? 1 : 0;
}

__global__ void __launch_bounds__(256) k_inside_grid_mask(float* __restrict__ flags, int A, int H, int W,
                                                          int in_h, int in_w) {
    const long long n = (long long)A * H * W;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int r = (int)(i % ((long long)H * W));
    const int y = r / W, x = r - y * W;
    flags[i] = (y < in_h && x < in_w) ? 1.0f : 0.0f;
}

// ------------------------------------------------------------------ a3
// [N,K] table, one thread per (i, j) with j fastest -> coalesced row-major stores.
__global__ void __launch_bounds__(256) k_calc_iou(float* __restrict__ out, const float* __restrict__ a,
                                                  long long N, const float* __restrict__ g, long long K) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N * K) return;
    const long long i = t / K, j = t - i * K;
    Box A{a[i], a[N + i], a[2 * N + i], a[3 * N + i]};
    Box G{g[j], g[K + j], g[2 * K + j], g[3 * K + j]};
    // the table must reproduce the divide result for every pair, incl. signed zeros
    out[t] = iou_plus1(A, area_plus1(A), G, area_plus1(G));
}

__global__ void __launch_bounds__(256) k_elem_iou(float* __restrict__ out, const float* __restrict__ a,
                                                  const float* __restrict__ b, long long N) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const float tlx = fmaxf(a[i], b[i]), tly = fmaxf(a[N + i], b[N + i]);
    const float brx = fminf(a[2 * N + i], b[2 * N + i]), bry = fminf(a[3 * N + i], b[3 * N + i]);
    float ai = (brx - tlx) * (bry - tly);
    ai = ai * ((tlx < brx && tly < bry) ? 1.0f : 0.0f);
    const float aa = (a[2 * N + i] - a[i]) * (a[3 * N + i] - a[N + i]);
    const float ab = (b[2 * N + i] - b[i]) * (b[3 * N + i] - b[N + i]);
    out[i] = ai / ((aa + ab) - ai);
}

// ------------------------------------------------------------------ K8
struct MS { float v[8]; };  // means[4], stds[4]

__global__ void __launch_bounds__(256) k_bbox2param(float* __restrict__ out, const float* __restrict__ base,
                                                    const float* __restrict__ bbox, long long n, MS ms) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float bw = (base[2 * n + i] - base[i]) + 1.0f, bh = (base[3 * n + i] - base[n + i]) + 1.0f;
    const float gw = (bbox[2 * n + i] - bbox[i]) + 1.0f, gh = (bbox[3 * n + i] - bbox[n + i]) + 1.0f;
    const float bcx = (base[2 * n + i] + base[i]) / 2.0f, bcy = (base[3 * n + i] + base[n + i]) / 2.0f;
    const float gcx = (bbox[2 * n + i] + bbox[i]) / 2.0f, gcy = (bbox[3 * n + i] + bbox[n + i]) / 2.0f;
    out[i] = ((gcx - bcx) / bw - ms.v[0]) / ms.v[4];
    out[n + i] = ((gcy - bcy) / bh - ms.v[1]) / ms.v[5];
    out[2 * n + i] = (logf(gw / bw) - ms.v[2]) / ms.v[6];
    out[3 * n + i] = (logf(gh / bh) - ms.v[3]) / ms.v[7];
}

__global__ void __launch_bounds__(256) k_param2bbox(float* __restrict__ out, const float* __restrict__ base,
                                                    const float* __restrict__ p, long long n, MS ms, int clamp,
                                                    float img_h, float img_w) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Box b{base[i], base[n + i], base[2 * n + i], base[3 * n + i]};
    const Box o = decode_box(b, p[i], p[n + i], p[2 * n + i], p[3 * n + i], ms.v, clamp != 0, img_h, img_w);
    out[i] = o.x1; out[n + i] = o.y1; out[2 * n + i] = o.x2; out[3 * n + i] = o.y2;
}

__global__ void __launch_bounds__(256) k_clamp_bbox(float* __restrict__ out, const float* __restrict__ b,
                                                    long long n, float img_h, float img_w) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float mx = img_w - 1.0f, my = img_h - 1.0f;
    out[i] = fminf(fmaxf(b[i], 0.0f), mx);
    out[n + i] = fminf(fmaxf(b[n + i], 0.0f), my);
    out[2 * n + i] = fminf(fmaxf(b[2 * n + i], 0.0f), mx);
    out[3 * n + i] = fminf(fmaxf(b[3 * n + i], 0.0f), my);
}

}  // namespace b2d

using namespace b2d;

extern "C" {

const char* b2d_last_error_string(void) {
    static thread_local std::string copy;
    std::lock_guard<std::mutex> l(g_err_mu);
    copy = g_err;
    return copy.c_str();
}

int b2d_version(void) { return 200; }

void b2d_reload_knobs(void) { knobs(); load_knobs(); }

int b2d_anchor_grid(float* out, const float* ws_host, const float* hs_host, int A, int H, int W, float stride,
                    int center_lt, void* stream) {
    B2D_REQUIRE(out && ws_host && hs_host, "anchor_grid: null pointer");
    B2D_REQUIRE(A >= 1 && A <= B2D_MAX_ANCHORS && H >= 0 && W >= 0, "anchor_grid: bad A/H/W");
    b2d_level lv;
    memset(&lv, 0, sizeof(lv));
    lv.H = H; lv.W = W; lv.A = A; lv.center_lt = center_lt; lv.stride = stride;
    for (int a = 0; a < A; ++a) { lv.ws[a] = ws_host[a]; lv.hs[a] = hs_host[a]; }
    const long long n = (long long)A * H * W;
    if (n == 0) return B2D_OK;
    k_anchor_grid<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(out, lv, n);
    return check_launch("anchor_grid");
}

int b2d_inside_anchor_mask(uint8_t* mask, const float* anchors, long long n, float img_h, float img_w,
                           float border, void* stream) {
    B2D_REQUIRE(mask && anchors && n >= 0, "inside_anchor_mask: bad args");
    if (n == 0) return B2D_OK;
    k_inside_anchor_mask<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(mask, anchors, n, img_h, img_w, border);
    return check_launch("inside_anchor_mask");
}

int b2d_inside_grid_mask(float* flags, int A, int H, int W, int in_h, int in_w, void* stream) {
    B2D_REQUIRE(flags && A >= 0 && H >= 0 && W >= 0, "inside_grid_mask: bad args");
    const long long n = (long long)A * H * W;
    if (n == 0) return B2D_OK;
    k_inside_grid_mask<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(flags, A, H, W, in_h, in_w);
    return check_launch("inside_grid_mask");
}

int b2d_calc_iou(float* out, const float* a, long long N, const float* b, long long K, void* stream) {
    B2D_REQUIRE(out && a && b && N >= 0 && K >= 0, "calc_iou: bad args");
    if (N * K == 0) return B2D_OK;
    k_calc_iou<<<cdiv(N * K, 256), 256, 0, (cudaStream_t)stream>>>(out, a, N, b, K);
    return check_launch("calc_iou");
}

int b2d_elem_iou(float* out, const float* a, const float* b, long long N, void* stream) {
    B2D_REQUIRE(out && a && b && N >= 0, "elem_iou: bad args");
    if (N == 0) return B2D_OK;
    k_elem_iou<<<cdiv(N, 256), 256, 0, (cudaStream_t)stream>>>(out, a, b, N);
    return check_launch("elem_iou");
}

static MS make_ms(const float* means, const float* stds) {
    MS ms;
    for (int i = 0; i < 4; ++i) { ms.v[i] = means ? means[i] : 0.0f; ms.v[4 + i] = stds ? stds[i] : 1.0f; }
    return ms;
}

int b2d_bbox2param(float* out, const float* base, const float* bbox, long long n, const float* means_host,
                   const float* stds_host, void* stream) {
    B2D_REQUIRE(out && base && bbox && n >= 0, "bbox2param: bad args");
    if (n == 0) return B2D_OK;
    k_bbox2param<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(out, base, bbox, n, make_ms(means_host, stds_host));
    return check_launch("bbox2param");
}

int b2d_param2bbox(float* out, const float* base, const float* param, long long n, const float* means_host,
                   const float* stds_host, int clamp, float img_h, float img_w, void* stream) {
    B2D_REQUIRE(out && base && param && n >= 0, "param2bbox: bad args");
    if (n == 0) return B2D_OK;
    k_param2bbox<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(out, base, param, n, make_ms(means_host, stds_host),
                                                                clamp, img_h, img_w);
    return check_launch("param2bbox");
}

int b2d_clamp_bbox(float* out, const float* bbox, long long n, float img_h, float img_w, void* stream) {
    B2D_REQUIRE(out && bbox && n >= 0, "clamp_bbox: bad args");
    if (n == 0) return B2D_OK;
    k_clamp_bbox<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(out, bbox, n, img_h, img_w);
    return check_launch("clamp_bbox");
}

}  // extern "C"
