// rtrb_api.cu — C ABI (include/rtrb_b200.h): scene baking, buffers, frame orchestration, the
// resolve kernels (Camera#render_at's mean / variance test / final average, camera.rb:80-98, and
// array_to_color, camera.rb:153-156), multi-GPU tile gather through peer mappings, and the FMA
// issue microbenchmark used as the roofline denominator.
//
// Compiled with -fmad=false: the host-side baking and the resolve arithmetic must round exactly
// like the reference's scalar FP64 code.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/rtrb_b200.h"
#include "rtrb_launch.h"
#include "rtrb_png.h"
#include "rtrb_rays.h"
#include "rtrb_trace.cuh"
#include "rtrb_types.h"

// Scenes with at most this many spheres use the linear-scan filter kernels and keep cull_sph[] in
// world order; larger scenes get the BVH kernels (measured crossover, see rtrb_trace_fast.cuh).
#define RTRB_BVH_MIN_SPHERES 32

namespace {

thread_local std::string g_last_error;
std::atomic<unsigned long long> g_launches{0};

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}
#define CUDA_TRY(expr)                                                                              \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess)                                                                          \
      return fail(RTRB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

// ---- host FP64 vector helpers in the reference's evaluation order (fast_4d_matrix.c) -------------
struct H3 { double x, y, z; };
inline H3 h3(const double* p) { return H3{p[0], p[1], p[2]}; }
inline double hnorm(H3 a) { return sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }
inline H3 hnormalize(H3 a) { double r = hnorm(a); return H3{a.x / r, a.y / r, a.z / r}; }
inline H3 hcross(H3 a, H3 b) { return H3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline H3 hadd(H3 a, H3 b) { return H3{a.x + b.x, a.y + b.y, a.z + b.z}; }
inline H3 hsub(H3 a, H3 b) { return H3{a.x - b.x, a.y - b.y, a.z - b.z}; }
inline H3 hmul(H3 a, double s) { return H3{a.x * s, a.y * s, a.z * s}; }
inline void put(double* d, H3 a) { d[0] = a.x; d[1] = a.y; d[2] = a.z; }

// Apex table entry for sphere (C, R) seen from apex A with positional uncertainty rho (see FrameParams).
// Margins: rounding of v and of the FP32 direction (8 eps |v| on b, hence 16 eps |v|^2 on b^2), the
// apex uncertainty, and the filter's usual scale term; Kq is rounded DOWN so the test only ever errs
// towards keeping a sphere.
float4 apex_entry(const double A[3], double rho, const double C[3], double R, double m_scale) {
  const double eps = 5.9604644775390625e-8;  // 2^-24
  const double vx = C[0] - A[0], vy = C[1] - A[1], vz = C[2] - A[2];
  const double v2 = vx * vx + vy * vy + vz * vz, vlen = sqrt(v2);
  const double Rp = fabs(R) + rho + 96.0 * eps * (m_scale + vlen) + 8.0 * eps * vlen;
  const double K = Rp * Rp + 32.0 * eps * v2;
  const double Kq = v2 - K;
  float kf = (float)Kq;
  if ((double)kf > Kq) kf = nextafterf(kf, -INFINITY);
  if (!(Kq == Kq)) kf = -INFINITY;  // NaN: always survive
  return make_float4((float)vx, (float)vy, (float)vz, kf);
}

// MT19937 (Matsumoto & Nishimura 1998) exactly as Ruby drives it: Random.srand(seed) with a seed that fits 32
// bits runs init_genrand(seed) (random.c rand_init), and every Random.rand is genrand_res53.  Used only by the
// RTRB_RNG_MT validation mode: the stream is generated here and the device indexes into it.
struct HostMT {
  uint32_t mt[624];
  int idx = 625;
  void seed(uint32_t s) {
    mt[0] = s;
    for (int i = 1; i < 624; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
    idx = 624;
  }
  uint32_t next32() {
    if (idx >= 624) {
      for (int k = 0; k < 624; ++k) {
        uint32_t y = (mt[k] & 0x80000000u) | (mt[(k + 1) % 624] & 0x7fffffffu);
        mt[k] = mt[(k + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
      }
      idx = 0;
    }
    uint32_t y = mt[idx++];
    y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
    return y;
  }
  double res53() {
    const uint32_t a = next32() >> 5, b = next32() >> 6;
    return ((double)a * 67108864.0 + (double)b) * (1.0 / 9007199254740992.0);
  }
};

// Frame control block: every small per-frame device word in ONE buffer (one memset, one D2H copy).  The kernels
// reach its fields through FrameParams (bind_ctl).
struct CtlBlock {
  unsigned long long counters[RTRB_CNT_N];      // RTRB_CNT_*
  unsigned long long first_bad;                 // max over flagged pixels of ~(x * H + y), 0 = none
  unsigned long long work[2];                   // work-claim counters
  uint32_t status, max_stack;
  uint32_t extra_count, pad;
  unsigned long long hot[2 * RTRB_HOT_SLICES];  // sliced (rays, shadow) counters
};
static_assert(sizeof(CtlBlock) == (RTRB_CNT_N + 5 + 2 * RTRB_HOT_SLICES) * 8, "control block layout");

// Pinned host mirror of a control block, mapped into the device's address space.
struct CtlMirror {
  CtlBlock blk;
  unsigned long long png_bytes;  // rtrb_submit_png frames: the file size, stored by the encoder
};

#define RTRB_PIPE_SLOTS 4  // frames that may be in flight between rtrb_submit and rtrb_wait
#define RTRB_CTL_RING 4    // control blocks of the synchronous frame path (frame overlap, render_impl)
struct FrameCtl {
  DevBuf<CtlBlock> d;          // its control block, or the ring of them (main_ctl)
  CtlBlock* blk = nullptr;     // the one the frame in this slot reports into
  CtlMirror* h = nullptr;      // pinned host mirror
  CtlMirror* h_dev = nullptr;  // ... and the address the device stores to (publish_ctl_kernel)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evt0 = nullptr, evt1 = nullptr, copied = nullptr, ctl_copied = nullptr;
  DevBuf<uint8_t> rgba;             // pipeline slots own a framebuffer; the main slot uses rtrb_renderer::rgba
  size_t* png_bytes_out = nullptr;  // rtrb_submit_png frames: where rtrb_wait stores h->png_bytes
  // facts of the frame in flight, needed to finish its stats later
  int W = 0, H = 0, S = 0, E = 0, n_tiles = 0;
  bool detail = false, in_flight = false, timed = false;
  unsigned ticket = 0;              // the rtrb_submit ticket occupying this slot while in_flight
  size_t px_count = 0;
  // Allocates on first use, so that slots a renderer never uses cost nothing.
  cudaError_t init(size_t blocks = 1) {
    cudaError_t e;
    if ((e = d.ensure(blocks)) != cudaSuccess) return e;
    blk = d.p;
    if ((e = cudaHostAlloc((void**)&h, sizeof(CtlMirror), cudaHostAllocMapped)) != cudaSuccess) return e;
    if ((e = cudaHostGetDevicePointer((void**)&h_dev, h, 0)) != cudaSuccess) return e;
    for (cudaEvent_t* ev : {&ev0, &ev1, &evt0, &evt1, &copied, &ctl_copied})
      if ((e = cudaEventCreate(ev)) != cudaSuccess) return e;
    return cudaSuccess;
  }
  ~FrameCtl() {
    if (h) cudaFreeHost(h);
    for (cudaEvent_t ev : {ev0, ev1, evt0, evt1, copied, ctl_copied})
      if (ev) cudaEventDestroy(ev);
  }
};

// The per-column / per-row scalars of camera.rb:133-134 in the reference's order: [W] x offsets, then [H] y offsets.
std::vector<double> lens_table(const rtrb_camera_desc* cam) {
  const int W = cam->width, H = cam->height;
  std::vector<double> tab((size_t)W + H);
  for (int x = 0; x < W; ++x) tab[x] = 2.0 * ((double)x / W - 0.5) * cam->retina_width;
  for (int y = 0; y < H; ++y) tab[(size_t)W + y] = 2 * ((double)y / H - 0.5) * cam->retina_height;
  return tab;
}

// Lens tables on the device (cached): evaluated on the host in the reference's order so the device does two loads
// instead of two FP64 divisions per sample.
struct LensTable {
  DevBuf<double> tab;            // [W + H] per-column / per-row retina offsets
  double key[4] = {0, 0, 0, 0};  // (W, H, retina_width, retina_height) the table was built for
  int ensure(const rtrb_camera_desc* cam, cudaStream_t s) {
    const double k[4] = {(double)cam->width, (double)cam->height, cam->retina_width, cam->retina_height};
    if (memcmp(k, key, sizeof(k)) == 0 && tab.p) return RTRB_OK;
    const std::vector<double> t = lens_table(cam);
    CUDA_TRY(tab.ensure(t.size()));
    CUDA_TRY(cudaMemcpyAsync(tab.p, t.data(), t.size() * sizeof(double), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    memcpy(key, k, sizeof(k));
    return RTRB_OK;
  }
};

// A window of a W x H frame, and the share of its super-tiles one rank renders.
struct Window {
  int x0, y0, x1, y1, rank, world;
  bool whole;  // the whole frame on one rank
};

// {0, 0, 0, 0} is the whole frame; tile_world <= 1 is one rank.
int make_window(int W, int H, int x0, int y0, int x1, int y1, int tile_rank, int tile_world, Window& w) {
  if (x0 == 0 && y0 == 0 && x1 == 0 && y1 == 0) { x1 = W; y1 = H; }
  if (x0 < 0 || y0 < 0 || x1 > W || y1 > H || x0 >= x1 || y0 >= y1) return fail(RTRB_ERR_INVALID, "bad window");
  const int world = tile_world <= 1 ? 1 : tile_world, rank = world == 1 ? 0 : tile_rank;
  if (rank < 0 || rank >= world) return fail(RTRB_ERR_INVALID, "tile_rank %d outside tile_world %d", rank, world);
  w = Window{x0, y0, x1, y1, rank, world, x0 == 0 && y0 == 0 && x1 == W && y1 == H && world == 1};
  return RTRB_OK;
}

void enumerate_tiles(int W, const Window& w, std::vector<int32_t>& out) {
  const int stx_count = (W + RTRB_SUPER - 1) / RTRB_SUPER;
  out.clear();
  // deal the window's super-tiles round-robin in row-major order: shares differ by at most one tile
  int i = 0;
  for (int ty = w.y0 / RTRB_SUPER; ty <= (w.y1 - 1) / RTRB_SUPER; ++ty)
    for (int tx = w.x0 / RTRB_SUPER; tx <= (w.x1 - 1) / RTRB_SUPER; ++tx, ++i)
      if (i % w.world == w.rank) out.push_back(ty * stx_count + tx);
}

// The super-tiles of a window that one rank renders (cached: rebuilt when the frame size, window or partition changes).
struct TileList {
  DevBuf<int32_t> dev;             // packed tx | ty << 16
  std::vector<int32_t> host;       // global ids ty * stx_count + tx
  size_t px_count = 0;             // pixels of the window covered by host
  uint32_t magic = 0;              // see FrameParams::tiles_magic (0 when the list is not plain row-major)
  int key[8] = {-1, -1, -1, -1, -1, -1, -1, -1};
  int ensure(int W, int H, const Window& w, cudaStream_t s) {
    const int k[8] = {W, H, w.x0, w.y0, w.x1, w.y1, w.rank, w.world};
    if (memcmp(k, key, sizeof(k)) == 0) return RTRB_OK;
    const int stx_count = (W + RTRB_SUPER - 1) / RTRB_SUPER;
    enumerate_tiles(W, w, host);
    std::vector<int32_t> packed(host.size());
    for (size_t i = 0; i < packed.size(); ++i) packed[i] = (host[i] % stx_count) | ((host[i] / stx_count) << 16);
    CUDA_TRY(dev.ensure(std::max<size_t>(1, packed.size())));
    if (!packed.empty())
      CUDA_TRY(cudaMemcpyAsync(dev.p, packed.data(), packed.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    memcpy(key, k, sizeof(k));
    magic = 0;
    if (stx_count > 0 && stx_count < 65536 && host.size() < 65536) {
      const uint32_t m = (uint32_t)((1ull << 32) / (unsigned)stx_count) + 1u;
      bool ok = true;
      for (size_t i = 0; i < host.size() && ok; ++i) {
        const uint32_t ty = (uint32_t)(((unsigned long long)i * m) >> 32);
        ok = host[i] == (int32_t)i && ty == (uint32_t)i / (unsigned)stx_count;
      }
      if (ok) magic = m;
    }
    px_count = 0;
    for (int b : host) {
      int tx = b % stx_count, ty = b / stx_count;
      int ax0 = std::max(w.x0, tx * RTRB_SUPER), ax1 = std::min(w.x1, (tx + 1) * RTRB_SUPER);
      int ay0 = std::max(w.y0, ty * RTRB_SUPER), ay1 = std::min(w.y1, (ty + 1) * RTRB_SUPER);
      if (ax1 > ax0 && ay1 > ay0) px_count += (size_t)(ax1 - ax0) * (ay1 - ay0);
    }
    return RTRB_OK;
  }
};

// RTRB_RNG_MT validation mode: serial by construction (every pixel's first draw depends on how many draws all earlier
// pixels made), so the frame iterates to a fixed point of its per-pixel draw offsets.
struct MtState {
  DevBuf<double> draws;
  DevBuf<uint32_t> offset, count;
  std::vector<double> host;        // the first host.size() draws after init_genrand(seed)
  HostMT gen;
  uint64_t seed = ~0ull;
  size_t uploaded = 0;
  int iterations = 0;              // iterations the last MT frame needed to reach its fixed point

  // Offsets = exclusive prefix sums of the per-pixel draw counts, iterated until stable.  The first pixel whose offset
  // is wrong is right after the next pass (its predecessors no longer move), so the loop ends after at most one pass
  // per pixel; in practice a handful of passes per data-dependent pixel.
  int trace(FrameParams& P, FrameCtl& fc, uint64_t frame_seed, int capacity, cudaStream_t s) {
    const int S = P.pre;
    const size_t npx = (size_t)(P.x1 - P.x0) * (size_t)(P.y1 - P.y0);
    if (npx * (size_t)std::max(S, P.max_samples) > 0x3fffffffull) return fail(RTRB_ERR_UNSUPPORTED, "window too large for RTRB_RNG_MT");
    CUDA_TRY(offset.ensure(npx));
    CUDA_TRY(count.ensure(npx));
    std::vector<uint32_t> off(npx), cnt(npx), nxt(npx);
    for (size_t i = 0; i < npx; ++i) off[i] = (uint32_t)(i * (size_t)S);
    if (seed != frame_seed) {
      host.clear(); gen.seed((uint32_t)frame_seed); seed = frame_seed; uploaded = 0;
    }
    size_t want_len = npx * (size_t)(S + 1) + 4096;
    const int max_iter = 200000;
    int it = 0;
    for (;; ++it) {
      if (it >= max_iter) return fail(RTRB_ERR_UNSUPPORTED, "RTRB_RNG_MT did not reach its fixed point in %d passes", max_iter);
      if (host.size() < want_len) {
        host.reserve(want_len);
        while (host.size() < want_len) host.push_back(gen.res53());
      }
      if (uploaded < host.size()) {
        CUDA_TRY(draws.ensure(host.size()));
        CUDA_TRY(cudaMemcpyAsync(draws.p, host.data(), host.size() * sizeof(double), cudaMemcpyHostToDevice, s));
        uploaded = host.size();
      }
      P.mt_stream = draws.p; P.mt_len = (uint32_t)std::min<size_t>(host.size(), 0xfffffff0u);
      P.mt_offset = offset.p; P.mt_count = count.p;
      CUDA_TRY(cudaMemcpyAsync(offset.p, off.data(), npx * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
      CUDA_TRY(cudaMemsetAsync(fc.blk, 0, sizeof(CtlBlock), s));
      if (fc.timed) CUDA_TRY(cudaEventRecord(fc.evt0, s));
      CUDA_TRY(rtrb_launch_trace_mt_strict(P, capacity, s));
      if (fc.timed) CUDA_TRY(cudaEventRecord(fc.evt1, s));
      g_launches++;
      CUDA_TRY(cudaMemcpyAsync(cnt.data(), count.p, npx * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
      CUDA_TRY(cudaStreamSynchronize(s));
      bool overflow = false;
      for (size_t i = 0; i < npx && !overflow; ++i) overflow = cnt[i] == 0xFFFFFFFFu;
      if (overflow) {  // some pixel ran past the end of the stream: generate more and repeat the pass
        want_len = host.size() * 2;
        if (want_len > 0xfffffff0ull) return fail(RTRB_ERR_UNSUPPORTED, "RTRB_RNG_MT stream would exceed 2^32 draws");
        continue;
      }
      size_t acc = 0;
      bool same = true;
      for (size_t i = 0; i < npx; ++i) {
        nxt[i] = (uint32_t)acc;
        same = same && nxt[i] == off[i];
        acc += cnt[i];
      }
      if (acc > 0xfffffff0ull) return fail(RTRB_ERR_UNSUPPORTED, "RTRB_RNG_MT stream would exceed 2^32 draws");
      if (same) break;
      off.swap(nxt);
      want_len = std::max(want_len, acc + 4096);
    }
    iterations = it + 1;
    return RTRB_OK;
  }
};

// The baked scene on the host: every fact the frames read from the renderer and the contents of every scene buffer.
// build_scene_image makes it from a descriptor (pure host); apply_scene puts it on the device.  Two images of the same
// description are equal byte for byte (same_image).
struct SceneImage {
  struct Facts {  // memset before use: compared as bytes
    int n_objects, n_lights, n_boxes, n_sph, n_pl;
    int scene_class;             // RTRB_SCENE_CLASS_* bits (FrameParams::scene_class)
    int small_scene;             // <= 32 spheres/boxes, <= 8 planes, <= 2 lights: linear-filter kernels
    double max_distance, soft_shadow_exponent;
    float m_scene, max_distance_f;
    // small scenes: the per-ray tables that travel in the kernel parameters (FrameParams::k_*)
    struct SmallTables {
      float4 light_tab[RTRB_K_LIGHTS][RTRB_APEX_MAX];
      float4 cull_sph[RTRB_APEX_MAX];
      float4 cull_pl[2 * RTRB_K_PLANES];
      DevLight lights[RTRB_K_LIGHTS];
      DevLightF lights_f[RTRB_K_LIGHTS];
      int32_t pl_index[RTRB_K_PLANES];
      int32_t has_light_tab;
    } k;
  } f;
  std::vector<double> sph_world;       // (cx, cy, cz, R) in cull_sph[] order, FP64, for the per-frame camera table
  std::vector<DevGeom> geom;
  std::vector<DevMat> mat;             // DevMat::tex left NULL: the device copy points at textures[mat_tex[i]]
  std::vector<int32_t> mat_tex;        // texture index of each object, -1 = none
  std::vector<DevLight> lights;
  std::vector<DevBox> boxes;
  std::vector<float4> cull_sph, cull_pl;  // FP32 filter view (FAST64)
  std::vector<int32_t> sph_index, pl_index;
  std::vector<DevLightF> lights_f;
  std::vector<BvhNode> bvh;
  std::vector<float4> light_tab;       // apex tables of the lights (linear-filter scenes with spheres and lights)
  std::vector<std::vector<uint8_t>> textures;
};

template <typename T>
bool same_bytes(const std::vector<T>& a, const std::vector<T>& b) {
  return a.size() == b.size() && (a.empty() || memcmp(a.data(), b.data(), a.size() * sizeof(T)) == 0);
}

bool same_image(const SceneImage& a, const SceneImage& b) {
  if (memcmp(&a.f, &b.f, sizeof(a.f)) != 0 || a.textures.size() != b.textures.size()) return false;
  for (size_t i = 0; i < a.textures.size(); ++i)
    if (!same_bytes(a.textures[i], b.textures[i])) return false;
  return same_bytes(a.sph_world, b.sph_world) && same_bytes(a.geom, b.geom) && same_bytes(a.mat, b.mat) &&
         same_bytes(a.mat_tex, b.mat_tex) && same_bytes(a.lights, b.lights) && same_bytes(a.boxes, b.boxes) &&
         same_bytes(a.cull_sph, b.cull_sph) && same_bytes(a.cull_pl, b.cull_pl) && same_bytes(a.sph_index, b.sph_index) &&
         same_bytes(a.pl_index, b.pl_index) && same_bytes(a.lights_f, b.lights_f) && same_bytes(a.bvh, b.bvh) &&
         same_bytes(a.light_tab, b.light_tab);
}

}  // namespace

struct rtrb_renderer {
  int device = 0;
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  cudaEvent_t push_ev = nullptr, push_done_ev = nullptr;  // rtrb_peer_push ordering (no timing)
  cudaEvent_t png_ev = nullptr;  // rtrb_encode_png waits for the pipelined encodes that share png
  RtrbPngScratch png;            // device PNG encoder scratch (rtrb_png.cu)
  FrameCtl main_ctl;       // synchronous calls: a ring of RTRB_CTL_RING control blocks
  FrameCtl pipe_ctl[RTRB_PIPE_SLOTS];  // rtrb_submit / rtrb_wait frame slots
  // Frame overlap (render_impl): on unless RTRB_FRAME_OVERLAP=0 when the renderer is created.
  bool frame_overlap = true;
  unsigned ring_next = 0;              // the main_ctl ring slot the next synchronous frame takes
  bool ring_zeroed = false;            // ... was zeroed by the last frame launched on ring_stream
  cudaStream_t ring_stream = nullptr;
  bool pipe_ready = false;
  unsigned next_ticket = 0;
  // baked scene: its host image and the device buffers that hold it
  SceneImage scene;
  DevBuf<DevGeom> geom;
  DevBuf<DevMat> mat;
  DevBuf<DevLight> lights;
  DevBuf<DevBox> boxes;
  DevBuf<float4> cull_sph, cull_pl;
  DevBuf<BvhNode> bvh;
  DevBuf<float4> light_tab;
  DevBuf<int32_t> sph_index, pl_index;
  DevBuf<DevLightF> lights_f;
  std::vector<DevBuf<uint8_t>> textures;  // DevMat::tex holds their addresses
  // rtrb_scene_update ordering (DESIGN.md §13)
  unsigned scene_gen = 0;                 // updates so far
  std::vector<cudaStream_t> scene_streams;  // streams that launched scene-reading work since the last bake
  cudaEvent_t scene_prior_ev = nullptr;   // recorded on each of them by an update, waited for by its copies
  cudaEvent_t scene_ready_ev = nullptr;   // the last update's copies are done
  uint8_t* staging = nullptr;             // pinned: the host side of an update's copies
  size_t staging_bytes = 0;
  std::vector<void*> retired;             // scene buffers an update outgrew; freed once the work before it is done
  // per-frame caches and scratch
  TileList tiles;
  LensTable lens;
  DevBuf<double> samples, extra_samples, pre_avg, rgb;
  DevBuf<uint32_t> extra_list;
  MtState mt;
  DevBuf<int32_t> hit;
  DevBuf<uint8_t> rgba;
  bool fb_exported = false;            // its address / IPC handle has been handed out: it may no longer move
  int fb_w = 0, fb_h = 0;
  // last frame
  int last_w = 0, last_h = 0;
  bool last_has_rgb = false, last_has_hit = false, last_rgba_own = true;
  int last_format = RTRB_FMT_RGBA8;
  cudaStream_t last_stream = nullptr;
  // ray-level calls (rtrb_trace_rays & co.): their own control block, scratch and lens tables, never the frames'
  FrameCtl ray_ctl;
  bool ray_ready = false;
  DevBuf<uint8_t> ray_scratch;         // host-buffer calls: inputs and outputs staged on the device
  LensTable ray_lens;                  // rtrb_camera_rays
  // The members free their own device memory; the renderer's device must be current (rtrb_renderer_destroy).
  ~rtrb_renderer() {
    for (void* p : retired) cudaFree(p);
    if (staging) cudaFreeHost(staging);
    for (cudaEvent_t ev : {push_ev, push_done_ev, png_ev, scene_prior_ev, scene_ready_ev})
      if (ev) cudaEventDestroy(ev);
    for (cudaStream_t s : {stream, copy_stream})
      if (s) cudaStreamDestroy(s);
  }
};

// A progressive frame (rtrb_progressive_*, DESIGN.md §14): one camera and its options, whose pre samples are traced in
// passes.  It owns everything its passes write, so that other work on the renderer between two passes neither
// disturbs it nor is disturbed by it.
struct rtrb_progressive {
  rtrb_renderer* r = nullptr;
  cudaStream_t stream = nullptr;
  FrameParams P;               // as baked at create; P.pre = S is the sample buffer's stride
  int capacity = 0, S = 0, E = 0;
  int done = 0;                // samples traced so far: every pass covers [done, sample_end)
  unsigned scene_gen = 0;      // the renderer's scene_gen at create (an update that applied since invalidates the frame)
  bool strict = false;
  FrameCtl fc;                 // its control block: counters, status, first_bad and max_stack accumulate over the passes
  TileList tiles;
  LensTable lens;
  DevBuf<double> samples, extra_samples, pre_avg, rgb;  // [slots][S][3], [slots][E][3], [slots][3], [H][W][3]
  DevBuf<uint32_t> extra_list;
  DevBuf<int32_t> hit;
  DevBuf<uint8_t> frame;       // the 8-bit frame, unless it goes to opts.rgba_device_out
  size_t frame_bytes = 0;
  int W = 0, H = 0, format = RTRB_FMT_RGBA8;
  bool own_frame = true;
  // its buffers are freed with it; its device must be current (rtrb_progressive_destroy)
};

namespace {

// ---- resolve kernels ---------------------------------------------------------------------------
using rtrb::decode_pixel;
using rtrb::final_average;
using rtrb::pre_mean;
using rtrb::pre_mean_of;
using rtrb::queue_adaptive;
using rtrb::write_pixel;

// 256-thread blocks over n_tiles * 1024 slots: every warp is whole, as queue_adaptive requires
__global__ void __launch_bounds__(256) resolve_kernel(const __grid_constant__ FrameParams P) {
  const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  int x = 0, y = 0;
  const bool valid = slot < (uint32_t)P.n_tiles * RTRB_SUPER_PIXELS && decode_pixel(P, slot, x, y);
  double ax = 0, ay = 0, az = 0, variance = 0;
  if (valid) pre_mean(P, slot, ax, ay, az, variance);
  const bool queued = queue_adaptive(P, valid && variance >= P.variant_threshold, slot, ax, ay, az);
  if (valid && !queued) write_pixel(P, x, y, ax, ay, az);
}

__global__ void __launch_bounds__(256) resolve_extra_kernel(const __grid_constant__ FrameParams P) {
  const uint32_t n = *P.extra_count;
  const int E = P.max_samples - P.pre;
  for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    const uint32_t slot = P.extra_list[e];
    int x, y;
    if (!decode_pixel(P, slot, x, y)) continue;
    const double* m = P.pre_avg + (size_t)e * 3;
    double ax = m[0], ay = m[1], az = m[2];
    const double* s = P.extra_samples + (size_t)e * E * 3;
    double cx = 0.0, cy = 0.0, cz = 0.0;
    for (int j = 0; j < E; ++j) { cx += s[j * 3 + 0]; cy += s[j * 3 + 1]; cz += s[j * 3 + 2]; }
    final_average(ax, ay, az, P.pre, cx, cy, cz, P.max_samples);
    write_pixel(P, x, y, ax, ay, az);
  }
}

// A progressive frame's preview: resolve_kernel over the first P.pre samples of each pixel of a sample buffer whose
// pixels are `stride` samples apart.  The host sets P.max_samples = P.pre, so queue_adaptive counts the adaptive pixels
// and rescales them in place, exactly as in a frame of pre = max = P.pre samples.
__global__ void __launch_bounds__(256) resolve_prefix_kernel(const __grid_constant__ FrameParams P, int stride) {
  const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  int x = 0, y = 0;
  const bool valid = slot < (uint32_t)P.n_tiles * RTRB_SUPER_PIXELS && decode_pixel(P, slot, x, y);
  double ax = 0, ay = 0, az = 0, variance = 0;
  if (valid) pre_mean_of(P.samples + (size_t)slot * stride * 3, P.pre, ax, ay, az, variance);
  const bool queued = queue_adaptive(P, valid && variance >= P.variant_threshold, slot, ax, ay, az);
  if (valid && !queued) write_pixel(P, x, y, ax, ay, az);
}

// Frame control block -> its pinned host mirror by direct stores (zero-copy over PCIe): see rtrb_submit.
__global__ void publish_ctl_kernel(unsigned long long* host, const unsigned long long* dev, int n) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) host[i] = dev[i];
}

__global__ void fill_i32_kernel(int32_t* p, size_t n, int32_t v) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ---- FMA issue microbenchmark ------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) fma_peak_kernel(T* out, int iters, T a, T b) {
  T r0 = (T)threadIdx.x, r1 = r0 + 1, r2 = r0 + 2, r3 = r0 + 3, r4 = r0 + 4, r5 = r0 + 5, r6 = r0 + 6, r7 = r0 + 7;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      r0 = fma(r0, a, b); r1 = fma(r1, a, b); r2 = fma(r2, a, b); r3 = fma(r3, a, b);
      r4 = fma(r4, a, b); r5 = fma(r5, a, b); r6 = fma(r6, a, b); r7 = fma(r7, a, b);
    }
  }
  T s = r0 + r1 + r2 + r3 + r4 + r5 + r6 + r7;
  if (s == (T)-12345.678) out[0] = s;  // never true; keeps the chains alive
}

template <typename T>
int measure_fma(int device, double* tflops_out) {
  CUDA_TRY(cudaSetDevice(device));
  int sms = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  DevBuf<T> d;
  CUDA_TRY(d.ensure(1));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  std::unique_ptr<CUevent_st, decltype(&cudaEventDestroy)> own_e0(e0, cudaEventDestroy);
  CUDA_TRY(cudaEventCreate(&e1));
  std::unique_ptr<CUevent_st, decltype(&cudaEventDestroy)> own_e1(e1, cudaEventDestroy);
  const int blocks = sms * 8, threads = 256, iters = 4096;
  fma_peak_kernel<T><<<blocks, threads>>>(d.p, 64, (T)1.0000001, (T)1e-9);  // warm-up
  g_launches++;
  CUDA_TRY(cudaDeviceSynchronize());
  double best = 0;
  for (int rep = 0; rep < 5; ++rep) {
    CUDA_TRY(cudaEventRecord(e0));
    fma_peak_kernel<T><<<blocks, threads>>>(d.p, iters, (T)1.0000001, (T)1e-9);
    g_launches++;
    CUDA_TRY(cudaEventRecord(e1));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    double flops = 2.0 * 64.0 * (double)iters * (double)blocks * (double)threads;
    double tf = flops / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  *tflops_out = best;
  return RTRB_OK;
}

// ---- scene baking ------------------------------------------------------------------------------
int validate_scene(const rtrb_scene_desc* s) {
  if (!s) return fail(RTRB_ERR_INVALID, "scene is NULL");
  if (s->n_objects < 0 || s->n_lights < 0 || s->n_textures < 0) return fail(RTRB_ERR_INVALID, "negative count");
  if (s->n_lights > RTRB_MAX_LIGHTS) return fail(RTRB_ERR_UNSUPPORTED, "more than %d lights", RTRB_MAX_LIGHTS);
  if (s->n_objects > 0 && !s->objects) return fail(RTRB_ERR_INVALID, "objects is NULL");
  if (s->n_lights > 0 && !s->lights) return fail(RTRB_ERR_INVALID, "lights is NULL");
  for (int i = 0; i < s->n_objects; ++i) {
    const rtrb_object_desc& o = s->objects[i];
    if (o.type != RTRB_OBJ_PLANE && o.type != RTRB_OBJ_SPHERE && o.type != RTRB_OBJ_BOX)
      return fail(RTRB_ERR_UNSUPPORTED, "object %d: unknown type %d", i, o.type);
    if (o.type == RTRB_OBJ_BOX) {
      H3 c = hcross(h3(o.front), h3(o.up));
      if (hnorm(c) == 0)  // box.rb:23 `front.cross(up).normalize` raises 'zero vector' in World#initialize
        return fail(RTRB_ERR_INVALID, "object %d: box front x up is the zero vector (fast_4d_matrix.c:290 would raise)", i);
    }
    if (o.texture >= s->n_textures) return fail(RTRB_ERR_INVALID, "object %d: texture index out of range", i);
    if (o.type == RTRB_OBJ_SPHERE && !o.has_refraction)
      return fail(RTRB_ERR_INVALID, "object %d: a sphere needs refractive_rate (sphere.rb:93 divides unconditionally)", i);
  }
  for (int i = 0; i < s->n_textures; ++i)
    if (!s->textures[i].rgb8 || s->textures[i].width <= 0 || s->textures[i].height <= 0)
      return fail(RTRB_ERR_INVALID, "texture %d is empty", i);
  return RTRB_OK;
}

// Descriptor -> host image of the baked scene (validate_scene has accepted `s`).  Pure host: no device is needed.
void build_scene_image(const rtrb_scene_desc* s, SceneImage& img) {
  SceneImage::Facts& fa = img.f;
  memset(&fa, 0, sizeof(fa));
  fa.n_objects = s->n_objects;
  fa.n_lights = s->n_lights;
  fa.max_distance = s->max_distance;
  fa.soft_shadow_exponent = s->soft_shadow_exponent;
  {
    bool textured = false;
    for (int i = 0; i < s->n_objects; ++i) textured = textured || (s->objects[i].texture >= 0 && s->objects[i].type != RTRB_OBJ_BOX);
    if (s->n_lights == 1 && s->soft_shadow_exponent == 2.0) {
      fa.scene_class |= RTRB_SCENE_CLASS_ONE_LIGHT;
      if (s->lights[0].radius == 0.0 && !textured) fa.scene_class |= RTRB_SCENE_CLASS_LEAN;
    }
  }
  img.textures.resize(s->n_textures);
  for (int i = 0; i < s->n_textures; ++i) {
    const rtrb_texture_desc& t = s->textures[i];
    img.textures[i].assign(t.rgb8, t.rgb8 + (size_t)t.width * t.height * 3);
  }
  std::vector<DevGeom>& geom = img.geom;
  std::vector<DevMat>& mat = img.mat;
  std::vector<DevBox>& boxes = img.boxes;
  geom.resize(s->n_objects);
  mat.resize(s->n_objects);
  img.mat_tex.assign(s->n_objects, -1);
  std::vector<double> box_radius;  // filter bound per box (INFINITY = none)
  for (int i = 0; i < s->n_objects; ++i) {
    const rtrb_object_desc& o = s->objects[i];
    DevGeom& g = geom[i];
    DevMat& m = mat[i];
    memset(&g, 0, sizeof(g));
    memset(&m, 0, sizeof(m));
    g.type = o.type;
    g.px = o.point[0]; g.py = o.point[1]; g.pz = o.point[2];
    g.radius = o.type == RTRB_OBJ_SPHERE ? o.radius : 0.0;
    g.nx = o.front[0]; g.ny = o.front[1]; g.nz = o.front[2];
    if (o.type == RTRB_OBJ_BOX) {
      // Box#initialize (box.rb:22-73) in the reference's evaluation order
      const H3 pt = h3(o.point), fr = h3(o.front), up = h3(o.up);
      const H3 left = hnormalize(hcross(fr, up));
      const H3 nfr = H3{-fr.x, -fr.y, -fr.z}, nup = H3{-up.x, -up.y, -up.z}, nleft = H3{-left.x, -left.y, -left.z};
      struct Spec { H3 front, up, point; double uu, vu; };
      const Spec spec[6] = {
          {up, left, hadd(pt, hmul(hmul(up, o.width_up), 0.5)), o.width_front, o.width_left},
          {nup, left, hsub(pt, hmul(hmul(up, o.width_up), 0.5)), o.width_front, o.width_left},
          {fr, up, hadd(pt, hmul(hmul(fr, o.width_front), 0.5)), o.width_left, o.width_up},
          {nfr, up, hsub(pt, hmul(hmul(fr, o.width_front), 0.5)), o.width_left, o.width_up},
          {left, up, hadd(pt, hmul(hmul(left, o.width_left), 0.5)), o.width_front, o.width_up},
          {nleft, up, hsub(pt, hmul(hmul(left, o.width_left), 0.5)), o.width_front, o.width_up}};
      DevBox bx;
      double bound = 0;
      // front _|_ up makes every face frame (left^, up^) orthonormal and in-plane, so a face's accepted
      // region is the rectangle |u|,|v| <= 1/2 around its point; otherwise the filter gets no bound
      const double fu = (fr.x * up.x + fr.y * up.y + fr.z * up.z) / (hnorm(fr) * hnorm(up));
      bool bounded = fabs(fu) < 1e-9;
      for (int k = 0; k < 6; ++k) {
        DevBoxFace& F = bx.f[k];
        const H3 fl = hnormalize(hcross(spec[k].front, spec[k].up));  // Plane#reinit, plane.rb:21-23
        const H3 l2 = hnormalize(fl), u2 = hnormalize(spec[k].up);     // Plane#get_uv, plane.rb:82-83
        F.px = spec[k].point.x; F.py = spec[k].point.y; F.pz = spec[k].point.z;
        F.nx = spec[k].front.x; F.ny = spec[k].front.y; F.nz = spec[k].front.z;
        F.lx = l2.x; F.ly = l2.y; F.lz = l2.z;
        F.ux = u2.x; F.uy = u2.y; F.uz = u2.z;
        F.u_unit = spec[k].uu; F.v_unit = spec[k].vu;
        const double half = 0.5 * sqrt(spec[k].uu * spec[k].uu + spec[k].vu * spec[k].vu);
        const double reach = hnorm(hsub(spec[k].point, pt)) + half;
        if (!(reach == reach) || reach > 1e30) bounded = false;
        bound = fmax(bound, reach);
      }
      box_radius.push_back(bounded ? bound * 1.001 : (double)INFINITY);
      g.aux = (int32_t)boxes.size();
      boxes.push_back(bx);
    }
    for (int k = 0; k < 3; ++k) {
      m.diffuse[k] = o.diffuse_rate[k]; m.refl[k] = o.reflective_attenuation[k];
      m.refr[k] = o.refractive_attenuation[k]; m.ambient[k] = o.ambient[k];
    }
    m.refractive_rate = o.refractive_rate;
    m.has_refraction = o.has_refraction;
    if (o.type == RTRB_OBJ_PLANE) {
      H3 f = h3(o.front);
      m.plane_nn_valid = hnorm(f) != 0 ? 1 : 0;
      if (m.plane_nn_valid) put(m.plane_nn, hnormalize(f));
    }
    m.u_unit = o.u_unit; m.v_unit = o.v_unit;
    m.hscale = o.texture_horizontal_scale; m.vscale = o.texture_vertical_scale;
    m.uoff = o.texture_u_offset; m.voff = o.texture_v_offset;
    if (o.texture >= 0 && o.type != RTRB_OBJ_BOX) {  // a box never samples its texture (box.rb has no local_lighting)
      img.mat_tex[i] = o.texture;
      m.tex_w = s->textures[o.texture].width;
      m.tex_h = s->textures[o.texture].height;
      if (o.type == RTRB_OBJ_SPHERE) {
        H3 gw = h3(o.greenwich_vec), np = h3(o.north_pole_vec);
        H3 east = hcross(np, gw);  // sphere.rb:19
        put(m.e0, hnormalize(gw)); put(m.e1, hnormalize(east)); put(m.e2, hnormalize(np));  // sphere.rb:113-115
      } else {
        H3 left = hnormalize(hcross(h3(o.front), h3(o.up)));  // plane.rb:21-23
        put(m.e0, hnormalize(left));                          // plane.rb:82 normalises again
        put(m.e1, hnormalize(h3(o.up)));
      }
    }
  }
  std::vector<DevLight>& lights = img.lights;
  lights.resize(s->n_lights);
  for (int i = 0; i < s->n_lights; ++i) {
    const rtrb_light_desc& l = s->lights[i];
    DevLight& d = lights[i];
    d.px = l.position[0]; d.py = l.position[1]; d.pz = l.position[2];
    for (int k = 0; k < 3; ++k) {
      d.color[k] = l.color[k];
      d.color_hl[k] = l.color[k] * l.high_light_rate;  // world.rb:94
    }
    d.radius = l.radius;
    d.hl_threshold = l.high_light_angle / 180.0 * 3.141592653589793;  // world.rb:92
  }
  // ---- FP32 filter view: conversions round to nearest; the filter's margins cover that error ----
  std::vector<float4>& csph = img.cull_sph;
  std::vector<float4>& cpl = img.cull_pl;
  std::vector<int32_t>& isph = img.sph_index;
  std::vector<int32_t>& ipl = img.pl_index;
  std::vector<BvhBuildSphere> bsph;
  float m_scene = 0.0f;
  for (int i = 0; i < s->n_objects; ++i) {
    const rtrb_object_desc& o = s->objects[i];
    if (o.type == RTRB_OBJ_SPHERE || o.type == RTRB_OBJ_BOX) {
      // a box enters the sphere filter through its bounding sphere (flagged: line test only)
      const bool is_box = o.type == RTRB_OBJ_BOX;
      const double rad = is_box ? box_radius[geom[i].aux] : o.radius;
      BvhBuildSphere bs;
      bs.c[0] = o.point[0]; bs.c[1] = o.point[1]; bs.c[2] = o.point[2]; bs.r = rad; bs.world_index = i;
      bs.bound_only = is_box ? 1 : 0;
      bsph.push_back(bs);
      double cm = fmax(fabs(o.point[0]), fmax(fabs(o.point[1]), fabs(o.point[2]))) + (fabs(rad) < 1e30 ? fabs(rad) : 0.0);
      m_scene = fmaxf(m_scene, nextafterf((float)cm, INFINITY));
    } else {
      double n1 = fabs(o.front[0]) + fabs(o.front[1]) + fabs(o.front[2]);
      double pm = fmax(fabs(o.point[0]), fmax(fabs(o.point[1]), fabs(o.point[2])));
      cpl.push_back(make_float4((float)o.front[0], (float)o.front[1], (float)o.front[2], nextafterf((float)n1, INFINITY)));
      cpl.push_back(make_float4((float)o.point[0], (float)o.point[1], (float)o.point[2], nextafterf((float)pm, INFINITY)));
      ipl.push_back(i);
    }
  }
  // the BVH build reorders the spheres so that every leaf is a contiguous run of cull_sph[]
  fa.small_scene = (int)bsph.size() <= RTRB_BVH_MIN_SPHERES && (int)ipl.size() <= RTRB_K_PLANES && s->n_lights <= RTRB_K_LIGHTS;
  if (!fa.small_scene) img.bvh = rtrb_bvh::build_tree(bsph);
  for (const BvhBuildSphere& bs : bsph) {
    float w = (float)bs.r;
    if (bs.bound_only) {  // rounded up, sign bit set
      w = fabsf(w);
      if ((double)w < fabs(bs.r)) w = nextafterf(w, INFINITY);
      w = -w;
      if (w == 0.0f) w = -0.0f;
    }
    csph.push_back(make_float4((float)bs.c[0], (float)bs.c[1], (float)bs.c[2], w));
    isph.push_back(bs.world_index);
  }
  fa.n_sph = (int)isph.size(); fa.n_pl = (int)ipl.size();
  for (const BvhBuildSphere& bs : bsph) { for (int k = 0; k < 3; ++k) img.sph_world.push_back(bs.c[k]); img.sph_world.push_back(bs.r); }
  if (fa.small_scene && !bsph.empty() && s->n_lights > 0) {
    std::vector<float4>& lt = img.light_tab;
    lt.resize((size_t)s->n_lights * bsph.size());
    for (int l = 0; l < s->n_lights; ++l) {
      double lm = fmax(fabs(s->lights[l].position[0]), fmax(fabs(s->lights[l].position[1]), fabs(s->lights[l].position[2])));
      for (size_t k = 0; k < bsph.size(); ++k)
        lt[(size_t)l * bsph.size() + k] = apex_entry(s->lights[l].position, 0.0, bsph[k].c, bsph[k].r, (double)m_scene + lm);
    }
    for (int l = 0; l < RTRB_K_LIGHTS; ++l)
      for (int k = 0; k < RTRB_APEX_MAX; ++k)
        fa.k.light_tab[l][k] = (l < s->n_lights && k < (int)bsph.size()) ? lt[(size_t)l * bsph.size() + k]
                                                                        : make_float4(0.0f, 0.0f, 0.0f, INFINITY);
    fa.k.has_light_tab = 1;
  }
  fa.m_scene = m_scene;
  fa.max_distance_f = nextafterf((float)s->max_distance, INFINITY);
  std::vector<DevLightF>& lf = img.lights_f;
  lf.resize(s->n_lights);
  for (int i = 0; i < s->n_lights; ++i) {
    const rtrb_light_desc& l = s->lights[i];
    double thr = l.high_light_angle / 180.0 * 3.141592653589793;
    lf[i].px = (float)l.position[0]; lf[i].py = (float)l.position[1]; lf[i].pz = (float)l.position[2];
    lf[i].pmax = nextafterf((float)fmax(fabs(l.position[0]), fmax(fabs(l.position[1]), fabs(l.position[2]))), INFINITY);
    lf[i].mode = (thr > 1e-4 && thr < 1.5) ? 1 : 0;
    double c = cos(thr);
    lf[i].cos2_thr = (float)(c * c);
  }
  if (fa.small_scene) {
    for (size_t k = 0; k < csph.size(); ++k) fa.k.cull_sph[k] = csph[k];
    for (size_t k = 0; k < cpl.size(); ++k) fa.k.cull_pl[k] = cpl[k];
    for (size_t k = 0; k < ipl.size(); ++k) fa.k.pl_index[k] = ipl[k];
    for (int l = 0; l < s->n_lights; ++l) { fa.k.lights[l] = lights[l]; fa.k.lights_f[l] = lf[l]; }
  }
  fa.n_boxes = (int)boxes.size();
}

// Calls f(device buffer, host image of it, least element count) for every scene buffer; the textures come before `mat`,
// whose device copy holds their addresses.
template <class F>
void for_each_scene_buffer(rtrb_renderer* r, const SceneImage& img, F&& f) {
  for (size_t i = 0; i < img.textures.size(); ++i) f(r->textures[i], img.textures[i], 1);
  f(r->mat, img.mat, 1);
  f(r->geom, img.geom, 1);
  f(r->lights, img.lights, 1);
  f(r->boxes, img.boxes, 1);
  f(r->cull_sph, img.cull_sph, 1);
  f(r->sph_index, img.sph_index, 1);
  f(r->cull_pl, img.cull_pl, 1);
  f(r->pl_index, img.pl_index, 1);
  f(r->lights_f, img.lights_f, 1);
  f(r->bvh, img.bvh, 1);
  f(r->light_tab, img.light_tab, 0);
}

// The allocations of one apply_scene that replace buffers too small for the new image, in for_each_scene_buffer order
// (nullptr: the current buffer is kept).  What is not handed over is freed.
struct FreshBuffers {
  std::vector<std::pair<void*, size_t>> a;  // (allocation, elements)
  ~FreshBuffers() {
    for (const auto& x : a)
      if (x.first) cudaFree(x.first);
  }
};

// Host image -> the renderer's device buffers, through the pinned staging buffer, asynchronously on `s` (the caller
// orders `s` after every reader of the old contents and has made sure the staging buffer is free).  Then the image
// becomes the renderer's scene.  Every allocation is made first: when one fails, the renderer is left as it was.  A
// buffer that is outgrown is retired, not freed: work queued before the bake may still read it.
int apply_scene(rtrb_renderer* r, SceneImage& img, cudaStream_t s) {
  const size_t kAlign = 256;
  auto padded = [&](size_t bytes) { return (bytes + kAlign - 1) & ~(kAlign - 1); };
  if (r->textures.size() < img.textures.size()) r->textures.resize(img.textures.size());  // empty until committed
  size_t total = 0;
  FreshBuffers fresh;
  cudaError_t e = cudaSuccess;
  for_each_scene_buffer(r, img, [&](auto& buf, const auto& v, size_t min_n) {
    total += padded(v.size() * sizeof(v[0]));
    const size_t want = std::max(min_n, v.size());
    void* q = nullptr;
    if (e == cudaSuccess && want > 0 && (want > buf.n || !buf.p)) e = cudaMalloc(&q, want * sizeof(v[0]));
    fresh.a.emplace_back(q, want);
  });
  if (e != cudaSuccess) return fail(RTRB_ERR_CUDA, "scene buffer allocation failed: %s", cudaGetErrorString(e));
  if (total > r->staging_bytes) {
    if (r->staging) CUDA_TRY(cudaFreeHost(r->staging));
    r->staging = nullptr;
    r->staging_bytes = 0;
    CUDA_TRY(cudaHostAlloc((void**)&r->staging, total, cudaHostAllocDefault));
    r->staging_bytes = total;
  }
  // commit: nothing below allocates
  while (r->textures.size() > img.textures.size()) {
    r->retired.push_back(r->textures.back().detach());
    r->textures.pop_back();
  }
  size_t k = 0;
  for_each_scene_buffer(r, img, [&](auto& buf, const auto&, size_t) {
    const std::pair<void*, size_t> x = fresh.a[k];
    fresh.a[k++].first = nullptr;
    if (!x.first) return;
    if (buf.p) r->retired.push_back(buf.detach());
    buf.adopt((std::remove_reference_t<decltype(*buf.p)>*)x.first, x.second);
  });
  uint8_t* at = r->staging;
  for_each_scene_buffer(r, img, [&](auto& buf, const auto& v, size_t) {
    const size_t bytes = v.size() * sizeof(v[0]);
    if (e != cudaSuccess || bytes == 0) return;
    uint8_t* staged = at;
    at += padded(bytes);
    memcpy(staged, v.data(), bytes);
    if constexpr (std::is_same<std::decay_t<decltype(v)>, std::vector<DevMat>>::value)
      for (size_t i = 0; i < v.size(); ++i)
        if (img.mat_tex[i] >= 0) ((DevMat*)staged)[i].tex = r->textures[img.mat_tex[i]].p;
    e = cudaMemcpyAsync(buf.p, staged, bytes, cudaMemcpyHostToDevice, s);
  });
  r->scene = std::move(img);
  CUDA_TRY(e);
  return RTRB_OK;
}

// Orders scene-reading work about to be queued on `s` after the last rtrb_scene_update: the first such launch on a
// stream since that update waits for the update's copies.  *fresh: this is that first launch (it must not overlap the
// work before it, render_impl).  The bake of rtrb_renderer_create completed before it returned.
int enter_scene_stream(rtrb_renderer* r, cudaStream_t s, bool* fresh) {
  *fresh = false;
  for (cudaStream_t t : r->scene_streams)
    if (t == s) return RTRB_OK;
  r->scene_streams.push_back(s);
  if (r->scene_gen == 0) return RTRB_OK;
  *fresh = true;
  CUDA_TRY(cudaStreamWaitEvent(s, r->scene_ready_ev, 0));
  return RTRB_OK;
}

// Camera#lens_func's per-frame constants in the reference's evaluation order (camera.rb:129-151).
void bake_camera(FrameParams& P, const rtrb_camera_desc* c) {
  H3 pos = h3(c->position), up = h3(c->up), front = h3(c->front);
  H3 left = hnormalize(hcross(up, front));
  H3 front_n = hnormalize(front);
  put(P.pos, pos);
  put(P.front, front);
  put(P.left, left);
  put(P.left_n, hnormalize(left));
  put(P.up_n, hnormalize(up));
  put(P.retina_center, hsub(pos, hmul(front_n, c->image_distance)));
  double object_distance = c->focal_distance * c->image_distance / (c->image_distance - c->focal_distance);
  put(P.focal_point, hadd(pos, hmul(front_n, object_distance)));
  P.retina_width = c->retina_width; P.retina_height = c->retina_height;
  P.aperture_radius = c->aperture_radius;
  P.variant_threshold = c->variant_threshold;
  P.width = c->width; P.height = c->height;
  P.pre = c->pre_sample_times; P.max_samples = c->max_sample_times;
  P.trace_depth = c->trace_depth; P.mc = c->monte_carlo_diffusion_times;
}

// The scene part of FrameParams: baked buffers, FP32 filter view, constant-bank tables of small scenes.  The camera
// apex table is not part of it (it only holds for rays that start at the camera).
void fill_scene_params(const rtrb_renderer* r, FrameParams& P) {
  const SceneImage::Facts& f = r->scene.f;
  P.max_distance = f.max_distance; P.soft_shadow_exponent = f.soft_shadow_exponent;
  P.n_objects = f.n_objects; P.n_lights = f.n_lights;
  P.geom = r->geom.p; P.mat = r->mat.p; P.lights = r->lights.p; P.boxes = r->boxes.p;
  P.cull_sph = r->cull_sph.p; P.sph_index = r->sph_index.p; P.cull_pl = r->cull_pl.p; P.pl_index = r->pl_index.p;
  P.lights_f = r->lights_f.p; P.n_sph = f.n_sph; P.n_pl = f.n_pl; P.bvh = r->bvh.p;
  P.m_scene = f.m_scene; P.max_distance_f = f.max_distance_f;
  P.use_bvh = f.small_scene ? 0 : 1;
  P.scene_class = f.scene_class;
  if (f.small_scene) {
    static_assert(sizeof(f.k.light_tab) == sizeof(P.k_light_tab) && sizeof(f.k.lights) == sizeof(P.k_lights), "table layout");
    memcpy(P.k_light_tab, f.k.light_tab, sizeof(P.k_light_tab));
    memcpy(P.k_cull_sph, f.k.cull_sph, sizeof(P.k_cull_sph));
    memcpy(P.k_cull_pl, f.k.cull_pl, sizeof(P.k_cull_pl));
    memcpy(P.k_lights, f.k.lights, sizeof(P.k_lights));
    memcpy(P.k_lights_f, f.k.lights_f, sizeof(P.k_lights_f));
    memcpy(P.k_pl_index, f.k.pl_index, sizeof(P.k_pl_index));
    P.k_has_light_tab = f.k.has_light_tab;
  }
  P.light_tab = r->scene.light_tab.empty() ? nullptr : r->light_tab.p;  // only scenes that use the linear filter
  P.cam_tab_valid = 0;
}

// Camera and scene of a frame: bake_camera, fill_scene_params and the camera's apex table.
void bake_frame(const rtrb_renderer* r, const rtrb_camera_desc* cam, FrameParams& P) {
  bake_camera(P, cam);
  fill_scene_params(r, P);
  const int n_sph = r->scene.f.n_sph;
  if (!P.use_bvh && n_sph > 0 && n_sph <= RTRB_APEX_MAX) {
    const double cm = fmax(fabs(cam->position[0]), fmax(fabs(cam->position[1]), fabs(cam->position[2])));
    const std::vector<double>& sw = r->scene.sph_world;
    for (int k = 0; k < n_sph; ++k)
      P.cam_tab[k] = apex_entry(cam->position, fabs(cam->aperture_radius), &sw[4 * (size_t)k], sw[4 * (size_t)k + 3],
                                (double)r->scene.f.m_scene + cm + fabs(cam->aperture_radius));
    for (int k = n_sph; k < RTRB_APEX_MAX; ++k) P.cam_tab[k] = make_float4(0.0f, 0.0f, 0.0f, INFINITY);  // never survives
    P.cam_tab_valid = 1;
  }
}

struct FrameTargets {  // where this renderer writes (own buffers, or rank 0's through a peer mapping)
  uint8_t* rgba = nullptr;
  double* rgb = nullptr;
  int32_t* hit = nullptr;
  bool want_rgb = true, want_hit = true;
  bool no_fill = false;  // multi-GPU: the caller pre-fills, ranks must not race on the shared buffer
};

// Own framebuffers for a (w, h) frame.  `rgba` = false when the 8-bit frame goes to a caller-supplied device buffer
// (rgba_device_out, a peer mapping, a pipeline slot).  Once the 8-bit framebuffer's address or IPC handle has been
// handed out (rtrb_framebuffer_device_ptr / _ipc_export) it is pinned: peers may be storing into it, so a frame that
// would need a larger one fails instead of freeing memory other ranks still write to.
int ensure_framebuffers(rtrb_renderer* r, int w, int h, bool rgba, bool rgb, bool hit) {
  size_t px = (size_t)w * h;
  CUDA_TRY(cudaSetDevice(r->device));
  if (rgba && r->rgba.n < px * 4) {
    if (r->fb_exported)
      return fail(RTRB_ERR_INVALID, "the %dx%d frame needs a larger framebuffer than the one whose device pointer / IPC handle "
                                    "was exported (%zu bytes); it cannot be reallocated while peers may write to it", w, h, r->rgba.n);
    CUDA_TRY(r->rgba.ensure(px * 4));
    CUDA_TRY(cudaMemset(r->rgba.p, 0, px * 4));
  }
  if (rgb) CUDA_TRY(r->rgb.ensure(px * 3));
  if (hit) CUDA_TRY(r->hit.ensure(px));
  r->fb_w = w; r->fb_h = h;
  return RTRB_OK;
}

// RTRB_ERR_CUDA without a CUDA device: this library has no CPU fallback.  count_out (optional): the number of devices.
int require_device(int* count_out = nullptr) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();  // not sticky: clear it so that later launch checks do not report it
    return fail(RTRB_ERR_CUDA, "no CUDA device (%s); this library has no CPU fallback", cudaGetErrorString(e));
  }
  if (count_out) *count_out = n;
  return RTRB_OK;
}

// The caller's options, or the defaults (main.rb's Random.srand(1), the default precision) when it passes none.
rtrb_render_opts opts_or_default(const rtrb_render_opts* in) {
  rtrb_render_opts o;
  memset(&o, 0, sizeof(o));
  if (in) o = *in;
  else { o.seed = 1; o.precision = RTRB_PREC_DEFAULT; }
  return o;
}

// Partial frames: the hit ids of pixels outside the window read -3.
void prefill_hits(int32_t* hit, int W, int H, cudaStream_t s) {
  const size_t n = (size_t)W * H;
  fill_i32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(hit, n, -3);
  g_launches++;
}

// Where a launch reports into the control block.
void bind_ctl(FrameParams& P, FrameCtl& fc) {
  CtlBlock* b = fc.blk;
  P.counters = b->counters; P.first_bad = &b->first_bad; P.work_counter = b->work;
  P.status = &b->status; P.extra_count = &b->extra_count; P.hot = b->hot;
}

// Turns a copied-back control block into rtrb_stats (+ RTRB_ERR_RAISED when a status bit is set).
int finish_stats(FrameCtl& fc, rtrb_stats* stats_out) {
  rtrb_stats local;
  if (!stats_out) stats_out = &local;
  const CtlBlock& b = fc.h->blk;
  const unsigned long long* c = b.counters;
  memset(stats_out, 0, sizeof(*stats_out));
  stats_out->rays = c[RTRB_CNT_RAYS]; stats_out->shadow_queries = c[RTRB_CNT_SHADOW];
  for (int sl = 0; sl < RTRB_HOT_SLICES; ++sl) {
    stats_out->rays += b.hot[2 * sl];
    stats_out->shadow_queries += b.hot[2 * sl + 1];
  }
  stats_out->highlight_hits = c[RTRB_CNT_HIGHLIGHT]; stats_out->hits = c[RTRB_CNT_HITS];
  stats_out->local_shaded = c[RTRB_CNT_LOCAL]; stats_out->lit_lights = c[RTRB_CNT_LIT];
  stats_out->mc_rays = c[RTRB_CNT_MC]; stats_out->refractions = c[RTRB_CNT_REFR];
  stats_out->texel_fetches = c[RTRB_CNT_TEXEL];
  stats_out->sphere_tests = c[RTRB_CNT_SPH_TEST]; stats_out->sphere_accepts = c[RTRB_CNT_SPH_ACC];
  stats_out->plane_tests = c[RTRB_CNT_PL_TEST]; stats_out->plane_accepts = c[RTRB_CNT_PL_ACC];
  stats_out->cover_sphere = c[RTRB_CNT_COV_SPH]; stats_out->cover_sphere_full = c[RTRB_CNT_COV_SPH_FULL];
  stats_out->cover_sphere_penumbra = c[RTRB_CNT_COV_SPH_PEN];
  stats_out->cover_plane = c[RTRB_CNT_COV_PL]; stats_out->cover_plane_accepts = c[RTRB_CNT_COV_PL_ACC];
  stats_out->adaptive_pixels = c[RTRB_CNT_ADAPTIVE]; stats_out->exact_tests = c[RTRB_CNT_EXACT];
  stats_out->box_tests = c[RTRB_CNT_BOX_TEST]; stats_out->box_accepts = c[RTRB_CNT_BOX_ACC];
  stats_out->cover_box = c[RTRB_CNT_COV_BOX]; stats_out->cover_box_accepts = c[RTRB_CNT_COV_BOX_ACC];
  // samples: counted on the device with count_detail; otherwise a pure function of the window
  stats_out->samples = fc.detail ? c[RTRB_CNT_SAMPLES]
                                 : (uint64_t)fc.px_count * fc.S + (uint64_t)(fc.E > 0 ? c[RTRB_CNT_ADAPTIVE] * (uint64_t)fc.E : 0);
  stats_out->status = b.status;
  stats_out->max_stack = b.max_stack > 1u ? b.max_stack : (stats_out->rays ? 1u : 0u);  // blocks only report depths > 1
  if (b.status && b.first_bad != 0ull) {  // stored complemented so that an all-zero block means "none"
    const unsigned long long key = ~b.first_bad;
    stats_out->first_bad_x = (int32_t)(key / (unsigned long long)fc.H);
    stats_out->first_bad_y = (int32_t)(key % (unsigned long long)fc.H);
  } else {
    stats_out->first_bad_x = stats_out->first_bad_y = -1;
  }
  float ms = 0;
  if (fc.timed) {
    CUDA_TRY(cudaEventElapsedTime(&ms, fc.ev0, fc.ev1));
    stats_out->device_ms = ms;
  }
  if (fc.timed && fc.n_tiles > 0) {
    CUDA_TRY(cudaEventElapsedTime(&ms, fc.evt0, fc.evt1));
    stats_out->trace_ms = ms;
  }
  if (b.status) {
    fail(RTRB_ERR_RAISED, "the reference would have raised: status 0x%x at pixel (%d, %d)", b.status,
         stats_out->first_bad_x, stats_out->first_bad_y);
    return RTRB_ERR_RAISED;
  }
  return RTRB_OK;
}

// Copies the control block of the work queued on `s` back and finishes its stats.  Synchronises.
int read_stats(FrameCtl& fc, cudaStream_t s, rtrb_stats* stats_out) {
  CUDA_TRY(cudaMemcpyAsync(&fc.h->blk, fc.blk, sizeof(CtlBlock), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  return finish_stats(fc, stats_out);
}

// The trace kernels of a frame or ray batch: their work-stack capacity (rtrb_launch.h, trace_capacity) into *capacity,
// or RTRB_ERR_UNSUPPORTED when none holds the stack; and their counter variant, P.count_detail.  The Box code lives
// only in the full-counter variants (rtrb_trace.cuh, trace_dispatch), so scenes with a box always run those.  Called
// with the other argument checks, before rtrb_trace_rays rejects a NULL renderer.
int pick_trace_kernels(const rtrb_renderer* r, bool strict, int trace_depth, int mc, bool count_detail, FrameParams& P,
                       int* capacity) {
  *capacity = trace_capacity(strict, trace_depth, mc);
  if (*capacity == 0)
    return fail(RTRB_ERR_UNSUPPORTED, "trace_depth*(1+mc)+1 = %lld exceeds the device stack limit %d",
                (long long)trace_depth * (1 + (long long)mc) + 1, kMaxStack);
  P.count_detail = (count_detail || (r && r->scene.f.n_boxes > 0)) ? 1 : 0;
  return RTRB_OK;
}

// The camera checks of a frame (rtrb_render_device and rtrb_progressive_create).
int check_frame_camera(const rtrb_camera_desc* cam) {
  if (cam->width <= 0 || cam->height <= 0) return fail(RTRB_ERR_INVALID, "bad frame size %dx%d", cam->width, cam->height);
  if (cam->pre_sample_times < 1) return fail(RTRB_ERR_INVALID, "pre_sample_times must be >= 1");
  if (cam->max_sample_times < 0 || cam->monte_carlo_diffusion_times < 0 || cam->trace_depth < 0)
    return fail(RTRB_ERR_INVALID, "negative sampling parameter");
  return RTRB_OK;
}

// The option checks of a frame after its RNG mode's: precision, pixel format, window and tile partition.
int check_frame_opts(const rtrb_render_opts& opts, int W, int H, Window& win) {
  if (opts.precision != RTRB_PREC_STRICT && opts.precision != RTRB_PREC_FAST64)
    return fail(RTRB_ERR_INVALID, "unknown precision mode %d", opts.precision);
  if (opts.pixel_format != RTRB_FMT_RGBA8 && opts.pixel_format != RTRB_FMT_RGB8 && opts.pixel_format != RTRB_FMT_PNG_RGB8)
    return fail(RTRB_ERR_INVALID, "unknown pixel format %d", opts.pixel_format);
  return make_window(W, H, opts.x0, opts.y0, opts.x1, opts.y1, opts.tile_rank, opts.tile_world, win);
}

// The per-frame memory budget of the sample buffers: S pre samples per slot (when the frame keeps them) and E extra.
int check_sample_budget(size_t n_slots, int S, int E, bool need_samples) {
  if ((need_samples && n_slots * (size_t)S * 3 * sizeof(double) > ((size_t)96 << 30)) || n_slots * (size_t)E * 3 * sizeof(double) > ((size_t)64 << 30))
    return fail(RTRB_ERR_UNSUPPORTED, "sample buffer would exceed the per-frame memory budget");
  return RTRB_OK;
}

int render_impl(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts_in,
                const FrameTargets* targets, rtrb_stats* stats_out, FrameCtl* ctl = nullptr) {
  if (!r || !cam) return fail(RTRB_ERR_INVALID, "renderer/camera is NULL");
  rtrb_render_opts opts = opts_or_default(opts_in);
  int rc = check_frame_camera(cam);
  if (rc) return rc;
  if (opts.rng_mode != RTRB_RNG_CTR && opts.rng_mode != RTRB_RNG_MT) return fail(RTRB_ERR_INVALID, "unknown rng_mode %d", opts.rng_mode);
  const bool mt_mode = opts.rng_mode == RTRB_RNG_MT;
  if (mt_mode) {
    // stream-exact validation mode: serial by construction (every pixel's first draw depends on how many draws
    // all earlier pixels made), so it is blocking, single-GPU, STRICT arithmetic, and iterates to a fixed point
    if (ctl != nullptr) return fail(RTRB_ERR_UNSUPPORTED, "RTRB_RNG_MT frames cannot be pipelined (rtrb_submit)");
    if (opts.tile_world > 1) return fail(RTRB_ERR_UNSUPPORTED, "RTRB_RNG_MT does not combine with a tile partition");
    if ((opts.seed >> 32) != 0) return fail(RTRB_ERR_UNSUPPORTED, "RTRB_RNG_MT: seeds above 32 bits take Ruby's init_by_array path");
    opts.precision = RTRB_PREC_STRICT;
  }
  const int W = cam->width, H = cam->height;
  Window win;
  if ((rc = check_frame_opts(opts, W, H, win))) return rc;
  const bool strict = opts.precision == RTRB_PREC_STRICT;
  FrameParams P;
  memset(&P, 0, sizeof(P));
  int capacity;
  if ((rc = pick_trace_kernels(r, strict, cam->trace_depth, cam->monte_carlo_diffusion_times, opts.count_detail != 0, P,
                               &capacity)))
    return rc;

  CUDA_TRY(cudaSetDevice(r->device));
  cudaStream_t stream = opts.stream ? (cudaStream_t)opts.stream : r->stream;

  FrameTargets tg;
  if (targets) tg = *targets;
  else {
    tg.want_rgb = !(opts.skip_outputs & RTRB_SKIP_RGB);
    tg.want_hit = !(opts.skip_outputs & RTRB_SKIP_HIT);
  }
  if (!tg.rgba && opts.rgba_device_out) tg.rgba = (uint8_t*)opts.rgba_device_out;
  if ((rc = ensure_framebuffers(r, W, H, tg.rgba == nullptr, tg.want_rgb && !tg.rgb, tg.want_hit && !tg.hit))) return rc;
  if (!tg.rgba) tg.rgba = r->rgba.p;
  if (tg.want_rgb && !tg.rgb) tg.rgb = r->rgb.p;
  if (tg.want_hit && !tg.hit) tg.hit = r->hit.p;
  if (!tg.want_rgb) tg.rgb = nullptr;
  if (!tg.want_hit) tg.hit = nullptr;

  if ((rc = r->tiles.ensure(W, H, win, stream)) || (rc = r->lens.ensure(cam, stream))) return rc;
  const int n_tiles = (int)r->tiles.host.size();
  const size_t n_slots = (size_t)n_tiles * RTRB_SUPER_PIXELS;
  const int S = cam->pre_sample_times;
  const int E = cam->max_sample_times > S ? cam->max_sample_times - S : 0;
  // Who finishes render_at (FrameParams::fuse_resolve).  The FAST64 ray-tree kernels resolve a pixel inside the CTA
  // that traced its samples whenever the sample count divides the CTA size: no FP64 sample buffer (24 B per sample:
  // 12.7 GB for one 4K / 64 spp frame) and no resolve launch.  RTRB_RNG_MT frames always go through the sample
  // buffer: trace_mt_body finishes render_at from it.
  int fuse = (!mt_mode && S == 1 && cam->variant_threshold > 0) ? RTRB_RESOLVE_IN_THREAD : RTRB_RESOLVE_SAMPLE_BUFFER;
  if (!strict && !mt_mode && cam->trace_depth > 1 && S <= RTRB_TREE_MIN_BLOCK && RTRB_TREE_MIN_BLOCK % S == 0)
    fuse = RTRB_RESOLVE_IN_CTA;
  const bool need_samples = fuse == RTRB_RESOLVE_SAMPLE_BUFFER;
  if ((rc = check_sample_budget(n_slots, S, E, need_samples))) return rc;
  if (need_samples) CUDA_TRY(r->samples.ensure(std::max<size_t>(1, n_slots * S * 3)));
  CUDA_TRY(r->extra_list.ensure(std::max<size_t>(1, n_slots)));
  if (E > 0) {
    CUDA_TRY(r->extra_samples.ensure(n_slots * E * 3));
    CUDA_TRY(r->pre_avg.ensure(n_slots * 3));
  }
  FrameCtl& fc = ctl ? *ctl : r->main_ctl;
  // Frame overlap: a frame that is one depth-1 FAST64 launch is launched with programmatic stream serialization, so its
  // kernel traces under the tail of the kernel before it on the stream and waits for it only to write
  // (trace_pre_body).  A synchronous frame takes the next control block of the main_ctl ring; an overlapping one also
  // zeroes the block after it, and the next synchronous frame on the same stream then needs no memset between the
  // two kernels.  Frames written into the same buffer stay ordered: every store waits for the previous grid.
  const bool overlap =
      r->frame_overlap && !strict && !mt_mode && fuse == RTRB_RESOLVE_IN_THREAD && cam->trace_depth <= 1 && n_tiles > 0;
  bool zeroed = false;
  CtlBlock* next_blk = nullptr;
  if (!ctl) {
    fc.blk = fc.d.p + r->ring_next;
    r->ring_next = (r->ring_next + 1) % RTRB_CTL_RING;
    zeroed = r->ring_zeroed && r->ring_stream == stream;
    r->ring_zeroed = false;
    if (overlap) next_blk = fc.d.p + r->ring_next;
  }

  // the first frame on a stream after rtrb_scene_update starts only after the update's copies: no overlap with the
  // kernel before it, which would let it read the scene early
  bool fresh_scene;
  if ((rc = enter_scene_stream(r, stream, &fresh_scene))) return rc;
  bake_frame(r, cam, P);
  P.key0 = (uint32_t)opts.seed; P.key1 = (uint32_t)(opts.seed >> 32);
  P.x0 = win.x0; P.y0 = win.y0; P.x1 = win.x1; P.y1 = win.y1;
  P.n_tiles = n_tiles; P.stx_count = (W + RTRB_SUPER - 1) / RTRB_SUPER; P.tiles = r->tiles.dev.p;
  P.lens_sx = r->lens.tab.p; P.lens_sy = r->lens.tab.p + W;
  P.samples = need_samples ? r->samples.p : nullptr; P.rgb = tg.rgb; P.hit = tg.hit; P.rgba = tg.rgba;
  P.pre_avg = r->pre_avg.p;
  bind_ctl(P, fc);
  P.tiles_magic = win.whole ? r->tiles.magic : 0u;
  P.extra_list = r->extra_list.p; P.extra_samples = r->extra_samples.p;
  P.pixel_format = opts.pixel_format;
  P.fuse_resolve = fuse;
  P.ctl_next = (unsigned long long*)next_blk;
  P.ctl_next_words = next_blk ? (uint32_t)(sizeof(CtlBlock) / sizeof(unsigned long long)) : 0u;

  // timing events only for the blocking calls that return stats (the pipelined frames of rtrb_submit report
  // device_ms = trace_ms = 0); the end-of-frame event only where something waits for it (timing, rtrb_submit's copy
  // stream) or when frames do not overlap
  const bool timed = stats_out != nullptr;
  fc.timed = timed;
  if (timed) CUDA_TRY(cudaEventRecord(fc.ev0, stream));
  if (!zeroed) CUDA_TRY(cudaMemsetAsync(fc.blk, 0, sizeof(CtlBlock), stream));
  if (!win.whole && !tg.no_fill && tg.hit == r->hit.p && tg.hit) prefill_hits(tg.hit, W, H, stream);
  if (n_tiles > 0 && mt_mode) {
    if ((rc = r->mt.trace(P, fc, opts.seed, capacity, stream))) return rc;
  } else if (n_tiles > 0) {
    if (timed) CUDA_TRY(cudaEventRecord(fc.evt0, stream));
    CUDA_TRY(strict ? rtrb_launch_trace_pre_strict(P, capacity, stream)
                    : rtrb_launch_trace_pre_fast(P, capacity, stream, overlap && !fresh_scene));
    if (next_blk) { r->ring_zeroed = true; r->ring_stream = stream; }
    if (timed) CUDA_TRY(cudaEventRecord(fc.evt1, stream));
    g_launches++;
    if (fuse == RTRB_RESOLVE_SAMPLE_BUFFER) {
      resolve_kernel<<<(unsigned)((n_slots + 255) / 256), 256, 0, stream>>>(P);
      CUDA_TRY(cudaGetLastError());
      g_launches++;
    }
    if (E > 0 && fuse != RTRB_RESOLVE_IN_THREAD) {
      CUDA_TRY(strict ? rtrb_launch_trace_extra_strict(P, capacity, stream) : rtrb_launch_trace_extra_fast(P, capacity, stream));
      g_launches++;
      resolve_extra_kernel<<<296, 256, 0, stream>>>(P);
      CUDA_TRY(cudaGetLastError());
      g_launches++;
    }
  }
  if (timed || ctl || !r->frame_overlap) CUDA_TRY(cudaEventRecord(fc.ev1, stream));
  r->last_w = W; r->last_h = H;
  r->last_rgba_own = tg.rgba == r->rgba.p;
  r->last_has_rgb = tg.rgb == r->rgb.p && tg.rgb != nullptr;
  r->last_has_hit = tg.hit == r->hit.p && tg.hit != nullptr;
  r->last_stream = stream;
  r->last_format = opts.pixel_format;

  // facts needed to finish the stats once the control block has been copied back
  fc.W = W; fc.H = H; fc.S = S; fc.E = E; fc.n_tiles = n_tiles; fc.detail = P.count_detail != 0;
  fc.px_count = r->tiles.px_count;
  return stats_out ? read_stats(fc, stream, stats_out) : RTRB_OK;
}

// First half of rtrb_submit / rtrb_submit_png: takes the next pipeline slot and launches the frame into its
// framebuffer on the render stream.
int submit_render(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts, FrameCtl** fc_out,
                  uint8_t** frame_out) {
  CUDA_TRY(cudaSetDevice(r->device));
  if (!r->pipe_ready) {
    for (int i = 0; i < RTRB_PIPE_SLOTS; ++i) {
      cudaError_t e = r->pipe_ctl[i].init();
      if (e != cudaSuccess) return fail(RTRB_ERR_CUDA, "pipeline slot init failed: %s", cudaGetErrorString(e));
    }
    r->pipe_ready = true;
  }
  const unsigned ticket = r->next_ticket;
  FrameCtl& fc = r->pipe_ctl[ticket % RTRB_PIPE_SLOTS];
  if (fc.in_flight) return fail(RTRB_ERR_INVALID, "%d frames are already in flight: call rtrb_wait first", RTRB_PIPE_SLOTS);
  const size_t slot_bytes = (size_t)cam->width * cam->height * 4;
  if (cam->width > 0 && cam->height > 0 && fc.rgba.n < slot_bytes) {
    CUDA_TRY(fc.rgba.ensure(slot_bytes));
    CUDA_TRY(cudaMemsetAsync(fc.rgba.p, 0, slot_bytes, r->stream));
  }
  rtrb_render_opts o = opts_or_default(opts);
  o.stream = nullptr;  // the pipeline owns its streams
  FrameTargets tg;
  tg.rgba = o.rgba_device_out ? (uint8_t*)o.rgba_device_out : fc.rgba.p;
  tg.want_rgb = false; tg.want_hit = false;
  int rc = render_impl(r, cam, &o, &tg, nullptr, &fc);
  if (rc) return rc;
  *fc_out = &fc;
  *frame_out = tg.rgba;
  return RTRB_OK;
}

// Second half: publishes the control block and hands out the ticket (the frame's copy or encode is queued).
int submit_finish(rtrb_renderer* r, FrameCtl& fc, int* ticket_out) {
  // The 1.3 KB control block does not go through the copy engine at all: a one-block kernel behind the frame's kernels
  // stores it straight into the pinned (device-mapped) host mirror.  As a DMA of its own - even on its own stream - it
  // sat between the 6.2 MB frame copies of a PCIe-bound sequence and cost 6 % of the frame rate (8 057 -> 8 540 frames/s
  // on config 2); behind the frame on the copy stream it cost 14 % (round 1).
  publish_ctl_kernel<<<1, 256, 0, r->stream>>>((unsigned long long*)&fc.h_dev->blk, (const unsigned long long*)fc.blk,
                                               (int)(sizeof(CtlBlock) / sizeof(unsigned long long)));
  CUDA_TRY(cudaGetLastError());
  g_launches++;
  CUDA_TRY(cudaEventRecord(fc.ctl_copied, r->stream));
  // (the slot is reused only after rtrb_wait has host-synchronised on `copied`, so no stream wait is needed)
  const unsigned ticket = r->next_ticket;
  fc.in_flight = true;
  fc.ticket = ticket;
  r->next_ticket = ticket + 1;
  *ticket_out = (int)ticket;
  return RTRB_OK;
}

// ---- ray-level calls ---------------------------------------------------------------------------------------------
// Checks every ray call makes before it needs a device.
int ray_args(const rtrb_ray_opts* opts, int n) {
  if (!opts) return fail(RTRB_ERR_INVALID, "opts is NULL");
  if (n < 0) return fail(RTRB_ERR_INVALID, "n = %d < 0", n);
  if (opts->precision != RTRB_PREC_STRICT && opts->precision != RTRB_PREC_FAST64)
    return fail(RTRB_ERR_INVALID, "unknown precision mode %d", opts->precision);
  if (opts->device_buffers != 0 && opts->device_buffers != 1)
    return fail(RTRB_ERR_INVALID, "device_buffers must be 0 or 1, not %d", opts->device_buffers);
  return RTRB_OK;
}

// No device: RTRB_ERR_CUDA, as every computing entry point.  Otherwise selects the renderer's device and sets up the
// ray calls' own control block on first use.
int ray_device(rtrb_renderer* r) {
  int rc = require_device();
  if (rc) return rc;
  if (!r) return fail(RTRB_ERR_INVALID, "renderer is NULL");
  CUDA_TRY(cudaSetDevice(r->device));
  if (!r->ray_ready) {
    cudaError_t e = r->ray_ctl.init();
    if (e != cudaSuccess) return fail(RTRB_ERR_CUDA, "ray control block init failed: %s", cudaGetErrorString(e));
    r->ray_ready = true;
  }
  return RTRB_OK;
}

// device_buffers = 1: `p` (if not NULL) must be device memory of the renderer's device.
int check_device_ptr(const rtrb_renderer* r, const void* p, const char* what) {
  if (!p) return RTRB_OK;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return fail(RTRB_ERR_INVALID, "%s is not a device pointer", what);
  }
  if (a.type != cudaMemoryTypeDevice || a.device != r->device)
    return fail(RTRB_ERR_INVALID, "%s is not device memory of the renderer's device %d", what, r->device);
  return RTRB_OK;
}

// Host-buffer calls stage their k arrays of bytes[i] bytes (0 = absent: nullptr) in ray_scratch.
int ray_stage(rtrb_renderer* r, const size_t* bytes, int k, uint8_t** out) {
  size_t off[8], total = 0;
  for (int i = 0; i < k; ++i) { off[i] = total; total += (bytes[i] + 255) & ~(size_t)255; }
  if (total > RTRB_RAY_SCRATCH_BUDGET)
    return fail(RTRB_ERR_UNSUPPORTED, "the call needs %zu bytes of device scratch, more than RTRB_RAY_SCRATCH_BUDGET (%zu); "
                                      "split it or pass device buffers", total, RTRB_RAY_SCRATCH_BUDGET);
  CUDA_TRY(r->ray_scratch.ensure(std::max<size_t>(1, total)));
  for (int i = 0; i < k; ++i) out[i] = bytes[i] ? r->ray_scratch.p + off[i] : nullptr;
  return RTRB_OK;
}

// Downloads the frame just rendered into host buffers.  A frame that raised (rc == RTRB_ERR_RAISED) keeps its error text.
int download_frame(rtrb_renderer* r, int rc, uint8_t* rgba, double* rgb_or_null, int32_t* hit_or_null) {
  if (rc != RTRB_OK && rc != RTRB_ERR_RAISED) return rc;
  std::string keep = g_last_error;
  int rc2 = rtrb_download(r, rgba, rgb_or_null, hit_or_null);
  if (rc2) return rc2;
  if (rc == RTRB_ERR_RAISED) g_last_error = keep;
  return rc;
}

}  // namespace

// ================================================================================================
extern "C" {
#pragma GCC visibility push(default)

int rtrb_abi_version(void) { return RTRB_ABI_VERSION; }
const char* rtrb_last_error(void) { return g_last_error.c_str(); }
uint64_t rtrb_launch_count(void) { return g_launches.load(); }

int rtrb_device_count(int* count_out) {
  if (!count_out) return fail(RTRB_ERR_INVALID, "count_out is NULL");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) { *count_out = 0; return fail(RTRB_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
  *count_out = n;
  return RTRB_OK;
}

int rtrb_renderer_create(const rtrb_scene_desc* scene, int device, rtrb_renderer** out) {
  if (!out) return fail(RTRB_ERR_INVALID, "out is NULL");
  *out = nullptr;
  int rc = validate_scene(scene);
  if (rc) return rc;
  int n = 0;
  if ((rc = require_device(&n))) return rc;
  if (device < 0 || device >= n) return fail(RTRB_ERR_INVALID, "device %d out of range (%d devices)", device, n);
  CUDA_TRY(cudaSetDevice(device));
  rtrb_renderer* r = new rtrb_renderer();
  r->device = device;
  cudaError_t ce;
  if ((ce = cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (ce = cudaStreamCreateWithFlags(&r->copy_stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (ce = cudaEventCreateWithFlags(&r->push_ev, cudaEventDisableTiming)) != cudaSuccess ||
      (ce = cudaEventCreateWithFlags(&r->push_done_ev, cudaEventDisableTiming)) != cudaSuccess ||
      (ce = r->main_ctl.init(RTRB_CTL_RING)) != cudaSuccess) {
    rtrb_renderer_destroy(r);
    return fail(RTRB_ERR_CUDA, "stream/event creation failed: %s", cudaGetErrorString(ce));
  }
  const char* overlap = getenv("RTRB_FRAME_OVERLAP");
  r->frame_overlap = !(overlap && strcmp(overlap, "0") == 0);
  SceneImage img;
  build_scene_image(scene, img);
  rc = apply_scene(r, img, r->stream);
  if (!rc && cudaStreamSynchronize(r->stream) != cudaSuccess) rc = fail(RTRB_ERR_CUDA, "scene upload failed");
  if (rc) { rtrb_renderer_destroy(r); return rc; }
  // a renderer that is never updated keeps no pinned staging memory
  cudaFreeHost(r->staging);
  r->staging = nullptr;
  r->staging_bytes = 0;
  *out = r;
  return RTRB_OK;
}

int rtrb_scene_update(rtrb_renderer* r, const rtrb_scene_desc* scene, void* stream) {
  int rc = validate_scene(scene);
  if (rc) return rc;
  if (!r) return fail(RTRB_ERR_INVALID, "renderer is NULL");
  SceneImage img;
  build_scene_image(scene, img);
  if (same_image(img, r->scene)) return RTRB_OK;  // nothing queued: frames keep overlapping
  CUDA_TRY(cudaSetDevice(r->device));
  const cudaStream_t s = stream ? (cudaStream_t)stream : r->stream;
  if (!r->scene_ready_ev) {
    CUDA_TRY(cudaEventCreateWithFlags(&r->scene_prior_ev, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&r->scene_ready_ev, cudaEventDisableTiming));
  }
  // The last update's copies are done: its staging buffer is free, and so is every buffer it outgrew (the work that
  // could read those was queued before it, and its copies waited for that work).
  if (r->scene_gen > 0) CUDA_TRY(cudaEventSynchronize(r->scene_ready_ev));
  cudaError_t freed = cudaSuccess;
  for (void* p : r->retired) {
    const cudaError_t e = cudaFree(p);
    if (freed == cudaSuccess) freed = e;
  }
  r->retired.clear();
  CUDA_TRY(freed);
  // Work queued so far reads the old scene: the copies wait for it on every stream that has launched some.  A stream
  // that can no longer be recorded on was destroyed by its owner; the work it had queued still runs, so then the copies
  // wait for the whole device, and the stream is forgotten.
  bool lost_stream = false;
  for (size_t i = 0; i < r->scene_streams.size();) {
    const cudaStream_t t = r->scene_streams[i];
    if (t != s && cudaEventRecord(r->scene_prior_ev, t) != cudaSuccess) {
      cudaGetLastError();  // not sticky: clear it so that later launch checks do not report it
      lost_stream = true;
      r->scene_streams.erase(r->scene_streams.begin() + i);
      continue;
    }
    if (t != s) CUDA_TRY(cudaStreamWaitEvent(s, r->scene_prior_ev, 0));
    ++i;
  }
  if (lost_stream) CUDA_TRY(cudaDeviceSynchronize());
  if ((rc = apply_scene(r, img, s))) return rc;
  CUDA_TRY(cudaEventRecord(r->scene_ready_ev, s));
  r->scene_gen++;
  r->scene_streams.clear();
  return RTRB_OK;
}

int rtrb_renderer_destroy(rtrb_renderer* r) {
  if (!r) return RTRB_OK;
  cudaSetDevice(r->device);
  cudaDeviceSynchronize();
  delete r;
  return RTRB_OK;
}

int rtrb_render_device(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts,
                       rtrb_stats* stats_out) {
  return render_impl(r, cam, opts, nullptr, stats_out);
}

int rtrb_download(rtrb_renderer* r, uint8_t* rgba, double* rgb_or_null, int32_t* hit_or_null) {
  if (!r) return fail(RTRB_ERR_INVALID, "renderer is NULL");
  if (r->last_w == 0) return fail(RTRB_ERR_INVALID, "nothing rendered yet");
  CUDA_TRY(cudaSetDevice(r->device));
  cudaStream_t s = r->last_stream ? r->last_stream : r->stream;
  size_t px = (size_t)r->last_w * r->last_h;
  if (rgba) {
    if (!r->last_rgba_own) return fail(RTRB_ERR_INVALID, "the last frame was written to rgba_device_out, not to the renderer's framebuffer");
    CUDA_TRY(cudaMemcpyAsync(rgba, r->rgba.p, RTRB_FRAME_BYTES(r->last_w, r->last_h, r->last_format), cudaMemcpyDeviceToHost, s));
  }
  if (rgb_or_null) {
    if (!r->last_has_rgb) return fail(RTRB_ERR_INVALID, "the last frame kept no float RGB");
    CUDA_TRY(cudaMemcpyAsync(rgb_or_null, r->rgb.p, px * 3 * sizeof(double), cudaMemcpyDeviceToHost, s));
  }
  if (hit_or_null) {
    if (!r->last_has_hit) return fail(RTRB_ERR_INVALID, "the last frame kept no hit ids");
    CUDA_TRY(cudaMemcpyAsync(hit_or_null, r->hit.p, px * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  return RTRB_OK;
}

int rtrb_render(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts, uint8_t* rgba,
                double* rgb_or_null, int32_t* hit_or_null, rtrb_stats* stats_out) {
  if (!rgba) return fail(RTRB_ERR_INVALID, "rgba is NULL");
  if (opts && opts->rgba_device_out)
    return fail(RTRB_ERR_INVALID, "rgba_device_out does not combine with a host-buffer call (use rtrb_render_device)");
  FrameTargets tg;
  tg.want_rgb = rgb_or_null != nullptr;
  tg.want_hit = hit_or_null != nullptr;
  rtrb_stats local;
  const int rc = render_impl(r, cam, opts, &tg, stats_out ? stats_out : &local);
  return download_frame(r, rc, rgba, rgb_or_null, hit_or_null);
}

int rtrb_submit(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts, uint8_t* rgba_host,
                int* ticket_out) {
  if (!r || !cam || !rgba_host || !ticket_out) return fail(RTRB_ERR_INVALID, "bad argument");
  FrameCtl* fcp = nullptr;
  uint8_t* frame = nullptr;
  int rc = submit_render(r, cam, opts, &fcp, &frame);
  if (rc) return rc;
  FrameCtl& fc = *fcp;
  const size_t bytes = RTRB_FRAME_BYTES(cam->width, cam->height, opts ? opts->pixel_format : RTRB_FMT_RGBA8);
  // the copy stream picks the frame up as soon as its kernels are done; the render stream is free
  // to start the next frame into the other slot meanwhile
  CUDA_TRY(cudaStreamWaitEvent(r->copy_stream, fc.ev1, 0));
  CUDA_TRY(cudaMemcpyAsync(rgba_host, frame, bytes, cudaMemcpyDeviceToHost, r->copy_stream));
  CUDA_TRY(cudaEventRecord(fc.copied, r->copy_stream));
  fc.png_bytes_out = nullptr;
  return submit_finish(r, fc, ticket_out);
}

int rtrb_submit_png(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts, uint8_t* png_host,
                    size_t capacity, size_t* png_bytes_out, int* ticket_out) {
  if (!r || !cam || !png_host || !png_bytes_out || !ticket_out) return fail(RTRB_ERR_INVALID, "bad argument");
  const int fmt = opts ? opts->pixel_format : RTRB_FMT_RGBA8;
  if (fmt != RTRB_FMT_RGBA8 && fmt != RTRB_FMT_RGB8)
    return fail(RTRB_ERR_INVALID, "rtrb_submit_png encodes RTRB_FMT_RGBA8 or RTRB_FMT_RGB8 frames, not format %d", fmt);
  if (opts && opts->rgba_device_out)
    return fail(RTRB_ERR_INVALID, "rgba_device_out does not combine with rtrb_submit_png (the frame stays in its slot)");
  size_t need = 0;
  int rc = rtrb_png_max_bytes(cam->width, cam->height, &need);
  if (rc) return rc;
  if (capacity < need) return fail(RTRB_ERR_INVALID, "png capacity %zu < %zu bytes (rtrb_png_max_bytes)", capacity, need);
  CUDA_TRY(cudaSetDevice(r->device));
  void* host_dev = nullptr;
  if (cudaHostGetDevicePointer(&host_dev, png_host, 0) != cudaSuccess) {
    cudaGetLastError();  // not sticky: clear it so that later launch checks do not report it
    return fail(RTRB_ERR_INVALID, "png_host is not page-locked, device-mapped host memory");
  }
  FrameCtl* fcp = nullptr;
  uint8_t* frame = nullptr;
  rc = submit_render(r, cam, opts, &fcp, &frame);
  if (rc) return rc;
  FrameCtl& fc = *fcp;
  // encoded on the copy stream behind the frame's kernels: the render stream goes on with the next frame, and only the
  // file crosses PCIe (device stores into png_host, the byte count into the slot's mapped control word)
  CUDA_TRY(cudaStreamWaitEvent(r->copy_stream, fc.ev1, 0));
  unsigned long long launches = 0;
  cudaError_t e = rtrb_png_encode(r->png, frame, cam->width, cam->height, fmt, r->copy_stream, (uint8_t*)host_dev,
                                  &fc.h_dev->png_bytes, &launches);
  g_launches += launches;
  if (e != cudaSuccess) return fail(RTRB_ERR_CUDA, "PNG encoder: %s", cudaGetErrorString(e));
  CUDA_TRY(cudaEventRecord(fc.copied, r->copy_stream));
  fc.png_bytes_out = png_bytes_out;
  return submit_finish(r, fc, ticket_out);
}

int rtrb_wait(rtrb_renderer* r, int ticket, rtrb_stats* stats_out) {
  if (!r || !r->pipe_ready) return fail(RTRB_ERR_INVALID, "nothing submitted");
  FrameCtl& fc = r->pipe_ctl[(unsigned)ticket % RTRB_PIPE_SLOTS];
  if (!fc.in_flight || fc.ticket != (unsigned)ticket) return fail(RTRB_ERR_INVALID, "ticket %d is not in flight", ticket);
  CUDA_TRY(cudaSetDevice(r->device));
  CUDA_TRY(cudaEventSynchronize(fc.copied));
  CUDA_TRY(cudaEventSynchronize(fc.ctl_copied));
  fc.in_flight = false;
  if (fc.png_bytes_out) *fc.png_bytes_out = (size_t)fc.h->png_bytes;
  return finish_stats(fc, stats_out);
}

int rtrb_framebuffer_device_ptr(rtrb_renderer* r, int width, int height, void** ptr_out) {
  if (!r || !ptr_out || width <= 0 || height <= 0) return fail(RTRB_ERR_INVALID, "bad argument");
  int rc = ensure_framebuffers(r, width, height, true, false, false);
  if (rc) return rc;
  r->fb_exported = true;
  *ptr_out = r->rgba.p;
  return RTRB_OK;
}

int rtrb_framebuffer_download(rtrb_renderer* r, int width, int height, uint8_t* rgba_host) {
  if (!r || !rgba_host || width <= 0 || height <= 0) return fail(RTRB_ERR_INVALID, "bad argument");
  CUDA_TRY(cudaSetDevice(r->device));
  const size_t bytes = (size_t)width * height * 4;
  if (r->rgba.n < bytes) return fail(RTRB_ERR_INVALID, "framebuffer is smaller than %dx%d", width, height);
  CUDA_TRY(cudaMemcpyAsync(rgba_host, r->rgba.p, bytes, cudaMemcpyDeviceToHost, r->copy_stream));
  CUDA_TRY(cudaStreamSynchronize(r->copy_stream));
  return RTRB_OK;
}

int rtrb_framebuffer_copy_async(rtrb_renderer* r, size_t bytes, uint8_t* host, void* stream) {
  if (!r || !host) return fail(RTRB_ERR_INVALID, "bad argument");
  if (bytes == 0) return RTRB_OK;
  CUDA_TRY(cudaSetDevice(r->device));
  if (r->rgba.n < bytes) return fail(RTRB_ERR_INVALID, "framebuffer is smaller than %zu bytes", bytes);
  CUDA_TRY(cudaMemcpyAsync(host, r->rgba.p, bytes, cudaMemcpyDeviceToHost, stream ? (cudaStream_t)stream : r->stream));
  return RTRB_OK;
}

int rtrb_framebuffer_ipc_export(rtrb_renderer* r, int width, int height, uint8_t handle_out[64]) {
  if (!r || !handle_out) return fail(RTRB_ERR_INVALID, "bad argument");
  int rc = ensure_framebuffers(r, width, height, true, false, false);
  if (rc) return rc;
  r->fb_exported = true;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  CUDA_TRY(cudaIpcGetMemHandle(&h, r->rgba.p));
  memcpy(handle_out, &h, 64);
  return RTRB_OK;
}

int rtrb_ipc_open(int device, const uint8_t handle[64], void** ptr_out) {
  if (!handle || !ptr_out) return fail(RTRB_ERR_INVALID, "bad argument");
  CUDA_TRY(cudaSetDevice(device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  CUDA_TRY(cudaIpcOpenMemHandle(ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
  return RTRB_OK;
}

int rtrb_ipc_close(int device, void* ptr) {
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaIpcCloseMemHandle(ptr));
  return RTRB_OK;
}

int rtrb_peer_push(rtrb_renderer* r, const void* src, void* dst_peer, size_t bytes, void* after_stream) {
  if (!r || !src || !dst_peer) return fail(RTRB_ERR_INVALID, "bad argument");
  if (bytes == 0) return RTRB_OK;
  CUDA_TRY(cudaSetDevice(r->device));
  cudaStream_t after = after_stream ? (cudaStream_t)after_stream : r->stream;
  CUDA_TRY(cudaEventRecord(r->push_ev, after));
  CUDA_TRY(cudaStreamWaitEvent(r->copy_stream, r->push_ev, 0));
  CUDA_TRY(cudaMemcpyAsync(dst_peer, src, bytes, cudaMemcpyDefault, r->copy_stream));  // copy engine over NVLink
  return RTRB_OK;
}

int rtrb_peer_push_join(rtrb_renderer* r, void* stream) {
  if (!r) return fail(RTRB_ERR_INVALID, "renderer is NULL");
  CUDA_TRY(cudaSetDevice(r->device));
  CUDA_TRY(cudaEventRecord(r->push_done_ev, r->copy_stream));
  CUDA_TRY(cudaStreamWaitEvent(stream ? (cudaStream_t)stream : r->stream, r->push_done_ev, 0));
  return RTRB_OK;
}

int rtrb_render_multi(rtrb_renderer* const* renderers, int n, const rtrb_camera_desc* cam,
                      const rtrb_render_opts* opts_in, uint8_t* rgba, double* rgb_or_null, int32_t* hit_or_null,
                      rtrb_stats* stats_out) {
  if (!renderers || n < 1 || !cam || !rgba) return fail(RTRB_ERR_INVALID, "bad argument");
  if (opts_in && opts_in->rgba_device_out)
    return fail(RTRB_ERR_INVALID, "rgba_device_out does not combine with a host-buffer call (use rtrb_render_device)");
  if (n == 1) return rtrb_render(renderers[0], cam, opts_in, rgba, rgb_or_null, hit_or_null, stats_out);
  rtrb_renderer* root = renderers[0];
  const bool want_rgb = rgb_or_null != nullptr, want_hit = hit_or_null != nullptr;
  int rc = ensure_framebuffers(root, cam->width, cam->height, true, want_rgb, want_hit);
  if (rc) return rc;
  // peer access root <- others (writes land in root's framebuffer over NVLink; no collective)
  for (int i = 1; i < n; ++i) {
    int can = 0;
    CUDA_TRY(cudaDeviceCanAccessPeer(&can, renderers[i]->device, root->device));
    if (!can) return fail(RTRB_ERR_CUDA, "device %d cannot access device %d", renderers[i]->device, root->device);
    CUDA_TRY(cudaSetDevice(renderers[i]->device));
    cudaError_t e = cudaDeviceEnablePeerAccess(root->device, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
      return fail(RTRB_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
    cudaGetLastError();
  }
  const rtrb_render_opts base = opts_or_default(opts_in);
  // (a bad window is left to the ranks' render_impl to report)
  Window win;
  if (want_hit && make_window(cam->width, cam->height, base.x0, base.y0, base.x1, base.y1, 0, 1, win) == RTRB_OK &&
      !win.whole) {
    CUDA_TRY(cudaSetDevice(root->device));
    prefill_hits(root->hit.p, cam->width, cam->height, root->stream);
    CUDA_TRY(cudaStreamSynchronize(root->stream));
  }
  std::vector<rtrb_stats> st(n);
  std::vector<int> rcs(n, 0);
  std::vector<std::string> errs(n);
  std::vector<std::thread> th;
  for (int i = 0; i < n; ++i) {
    th.emplace_back([&, i]() {
      rtrb_render_opts o = base;
      o.tile_rank = i; o.tile_world = n; o.stream = nullptr; o.rgba_device_out = nullptr;
      FrameTargets tg;
      tg.rgba = root->rgba.p;
      tg.rgb = want_rgb ? root->rgb.p : nullptr;
      tg.hit = want_hit ? root->hit.p : nullptr;
      tg.want_rgb = want_rgb; tg.want_hit = want_hit; tg.no_fill = true;
      rcs[i] = render_impl(renderers[i], cam, &o, &tg, &st[i]);
      errs[i] = g_last_error;
    });
  }
  for (auto& t : th) t.join();
  int worst = RTRB_OK;
  for (int i = 0; i < n; ++i) {
    if (rcs[i] != RTRB_OK && rcs[i] != RTRB_ERR_RAISED) { g_last_error = errs[i]; return rcs[i]; }
    if (rcs[i] == RTRB_ERR_RAISED) { worst = RTRB_ERR_RAISED; g_last_error = errs[i]; }
  }
  rtrb_stats agg;
  memset(&agg, 0, sizeof(agg));
  agg.first_bad_x = agg.first_bad_y = -1;
  long long best_key = -1;
  {
    // the counters samples .. cover_box_accepts are summed as one array
    static_assert(offsetof(rtrb_stats, status) - offsetof(rtrb_stats, samples) == 25 * sizeof(uint64_t), "rtrb_stats counters");
    uint64_t* a = &agg.samples;
    for (int i = 0; i < n; ++i) {
      const uint64_t* b = &st[i].samples;
      for (int k = 0; k < 25; ++k) a[k] += b[k];
      agg.status |= st[i].status;
      agg.max_stack = std::max(agg.max_stack, st[i].max_stack);
      agg.device_ms = std::max(agg.device_ms, st[i].device_ms);
      agg.trace_ms = std::max(agg.trace_ms, st[i].trace_ms);
      if (st[i].first_bad_x >= 0) {
        long long key = (long long)st[i].first_bad_x * cam->height + st[i].first_bad_y;
        if (best_key < 0 || key < best_key) { best_key = key; agg.first_bad_x = st[i].first_bad_x; agg.first_bad_y = st[i].first_bad_y; }
      }
    }
  }
  if (stats_out) *stats_out = agg;
  return download_frame(root, worst, rgba, rgb_or_null, hit_or_null);  // rank 0's render_impl recorded the frame
}

int rtrb_png_max_bytes(int width, int height, size_t* bytes_out) {
  if (!bytes_out || width <= 0 || height <= 0) return fail(RTRB_ERR_INVALID, "bad argument");
  *bytes_out = rtrb_png_bound(width, height);
  return RTRB_OK;
}

int rtrb_encode_png(rtrb_renderer* r, const void* src_device, int width, int height, int pixel_format, void* stream,
                    uint8_t* png_host, size_t capacity, size_t* bytes_out) {
  if (!png_host || !bytes_out) return fail(RTRB_ERR_INVALID, "bad argument");
  if (pixel_format != RTRB_FMT_RGBA8 && pixel_format != RTRB_FMT_RGB8 && pixel_format != RTRB_FMT_PNG_RGB8)
    return fail(RTRB_ERR_INVALID, "unknown pixel format %d", pixel_format);
  size_t need = 0;
  int rc = rtrb_png_max_bytes(width, height, &need);
  if (rc) return rc;
  if (capacity < need) return fail(RTRB_ERR_INVALID, "png capacity %zu < %zu bytes (rtrb_png_max_bytes)", capacity, need);
  if ((rc = require_device())) return rc;
  if (!r) return fail(RTRB_ERR_INVALID, "renderer is NULL");
  CUDA_TRY(cudaSetDevice(r->device));
  const uint8_t* src = (const uint8_t*)src_device;
  if (!src) {
    if (r->rgba.n < RTRB_FRAME_BYTES(width, height, pixel_format))
      return fail(RTRB_ERR_INVALID, "the framebuffer (%zu bytes) is smaller than a %dx%d frame", r->rgba.n, width, height);
    src = r->rgba.p;
  }
  cudaStream_t s = stream ? (cudaStream_t)stream : r->stream;
  if (!r->png_ev) CUDA_TRY(cudaEventCreateWithFlags(&r->png_ev, cudaEventDisableTiming));
  CUDA_TRY(cudaEventRecord(r->png_ev, r->copy_stream));  // pipelined encodes use the same scratch
  CUDA_TRY(cudaStreamWaitEvent(s, r->png_ev, 0));
  unsigned long long launches = 0;
  cudaError_t e = rtrb_png_encode(r->png, src, width, height, pixel_format, s, nullptr, nullptr, &launches);
  g_launches += launches;
  if (e != cudaSuccess) return fail(RTRB_ERR_CUDA, "PNG encoder: %s", cudaGetErrorString(e));
  unsigned long long total = 0;
  CUDA_TRY(cudaMemcpyAsync(&total, r->png.total.p, sizeof(total), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  if (total > capacity) return fail(RTRB_ERR_CUDA, "PNG encoder produced %llu bytes, more than its bound %zu", total, need);
  CUDA_TRY(cudaMemcpyAsync(png_host, r->png.file.p, total, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  *bytes_out = (size_t)total;
  return RTRB_OK;
}

int rtrb_trace_rays(rtrb_renderer* r, const rtrb_ray_opts* opts, int n, const rtrb_ray* rays, const uint32_t* keys_or_null,
                    double* rgb_out, int32_t* hit_or_null, rtrb_stats* stats_out) {
  int rc = ray_args(opts, n);
  if (rc) return rc;
  if (n > 0 && (!rays || !rgb_out)) return fail(RTRB_ERR_INVALID, "rays / rgb_out is NULL");
  if (opts->trace_depth < 0 || opts->monte_carlo_diffusion_times < 0) return fail(RTRB_ERR_INVALID, "negative trace_depth / mc");
  const bool strict = opts->precision == RTRB_PREC_STRICT;
  FrameParams P;
  memset(&P, 0, sizeof(P));
  int capacity;
  if ((rc = pick_trace_kernels(r, strict, opts->trace_depth, opts->monte_carlo_diffusion_times, opts->count_detail != 0,
                               P, &capacity)))
    return rc;
  if ((rc = ray_device(r))) return rc;
  const bool dev = opts->device_buffers == 1;
  if (dev && ((rc = check_device_ptr(r, rays, "rays")) || (rc = check_device_ptr(r, keys_or_null, "keys")) ||
              (rc = check_device_ptr(r, rgb_out, "rgb_out")) || (rc = check_device_ptr(r, hit_or_null, "hit"))))
    return rc;
  if (stats_out) { memset(stats_out, 0, sizeof(*stats_out)); stats_out->first_bad_x = stats_out->first_bad_y = -1; }
  if (n == 0) return RTRB_OK;
  cudaStream_t s = opts->stream ? (cudaStream_t)opts->stream : r->stream;
  bool fresh_scene;
  if ((rc = enter_scene_stream(r, s, &fresh_scene))) return rc;
  const size_t un = (size_t)n;
  RayBatch B;
  memset(&B, 0, sizeof(B));
  B.n = n;
  if (dev) {
    B.rays = (const double*)rays; B.keys = keys_or_null; B.rgb = rgb_out; B.hit = hit_or_null;
  } else {
    const size_t bytes[4] = {un * sizeof(rtrb_ray), keys_or_null ? un * 2 * sizeof(uint32_t) : 0, un * 3 * sizeof(double),
                             hit_or_null ? un * sizeof(int32_t) : 0};
    uint8_t* p[4];
    if ((rc = ray_stage(r, bytes, 4, p))) return rc;
    CUDA_TRY(cudaMemcpyAsync(p[0], rays, bytes[0], cudaMemcpyHostToDevice, s));
    if (keys_or_null) CUDA_TRY(cudaMemcpyAsync(p[1], keys_or_null, bytes[1], cudaMemcpyHostToDevice, s));
    B.rays = (const double*)p[0]; B.keys = (const uint32_t*)p[1]; B.rgb = (double*)p[2]; B.hit = (int32_t*)p[3];
  }
  fill_scene_params(r, P);
  P.trace_depth = opts->trace_depth; P.mc = opts->monte_carlo_diffusion_times;
  P.width = 1; P.height = 1;  // status reports ray i as pixel (i, 0)
  P.key0 = (uint32_t)opts->seed; P.key1 = (uint32_t)(opts->seed >> 32);
  FrameCtl& fc = r->ray_ctl;
  bind_ctl(P, fc);
  fc.timed = stats_out != nullptr;
  fc.W = 1; fc.H = 1; fc.S = 1; fc.E = 0; fc.n_tiles = 1; fc.px_count = un; fc.detail = P.count_detail != 0;
  if (fc.timed) CUDA_TRY(cudaEventRecord(fc.ev0, s));
  CUDA_TRY(cudaMemsetAsync(fc.blk, 0, sizeof(CtlBlock), s));
  if (fc.timed) CUDA_TRY(cudaEventRecord(fc.evt0, s));
  CUDA_TRY(rtrb_launch_trace_rays(P, B, strict, capacity, s));
  g_launches++;
  if (fc.timed) { CUDA_TRY(cudaEventRecord(fc.evt1, s)); CUDA_TRY(cudaEventRecord(fc.ev1, s)); }
  if (!dev) {
    CUDA_TRY(cudaMemcpyAsync(rgb_out, B.rgb, un * 3 * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (hit_or_null) CUDA_TRY(cudaMemcpyAsync(hit_or_null, B.hit, un * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    return read_stats(fc, s, stats_out);
  }
  return stats_out ? read_stats(fc, s, stats_out) : RTRB_OK;
}

int rtrb_intersect_rays(rtrb_renderer* r, const rtrb_ray_opts* opts, int n, const rtrb_ray* rays, rtrb_ray_hit* hits_out) {
  static_assert(sizeof(rtrb_ray) == 48 && sizeof(rtrb_ray_hit) == 72, "rtrb_ray / rtrb_ray_hit layout");
  int rc = ray_args(opts, n);
  if (rc) return rc;
  if (n > 0 && (!rays || !hits_out)) return fail(RTRB_ERR_INVALID, "rays / hits_out is NULL");
  if ((rc = ray_device(r))) return rc;
  const bool dev = opts->device_buffers == 1;
  if (dev && ((rc = check_device_ptr(r, rays, "rays")) || (rc = check_device_ptr(r, hits_out, "hits_out")))) return rc;
  if (n == 0) return RTRB_OK;
  cudaStream_t s = opts->stream ? (cudaStream_t)opts->stream : r->stream;
  bool fresh_scene;
  if ((rc = enter_scene_stream(r, s, &fresh_scene))) return rc;
  const size_t un = (size_t)n;
  RayBatch B;
  memset(&B, 0, sizeof(B));
  B.n = n;
  if (dev) {
    B.rays = (const double*)rays; B.hits = hits_out;
  } else {
    const size_t bytes[2] = {un * sizeof(rtrb_ray), un * sizeof(rtrb_ray_hit)};
    uint8_t* p[2];
    if ((rc = ray_stage(r, bytes, 2, p))) return rc;
    CUDA_TRY(cudaMemcpyAsync(p[0], rays, bytes[0], cudaMemcpyHostToDevice, s));
    B.rays = (const double*)p[0]; B.hits = (rtrb_ray_hit*)p[1];
  }
  FrameParams P;
  memset(&P, 0, sizeof(P));
  fill_scene_params(r, P);
  CUDA_TRY(rtrb_launch_intersect_rays(P, B, opts->precision == RTRB_PREC_STRICT, s));
  g_launches++;
  if (!dev) {
    CUDA_TRY(cudaMemcpyAsync(hits_out, B.hits, un * sizeof(rtrb_ray_hit), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
  }
  return RTRB_OK;
}

int rtrb_camera_rays(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_ray_opts* opts, int sample_begin,
                     int sample_end, rtrb_ray* rays_out, uint32_t* keys_or_null) {
  int rc = ray_args(opts, 0);
  if (rc) return rc;
  if (!cam) return fail(RTRB_ERR_INVALID, "camera is NULL");
  const int W = cam->width, H = cam->height;
  if (W <= 0 || H <= 0) return fail(RTRB_ERR_INVALID, "bad frame size %dx%d", W, H);
  Window win;
  if ((rc = make_window(W, H, opts->x0, opts->y0, opts->x1, opts->y1, 0, 1, win))) return rc;
  if (sample_begin < 0 || sample_end <= sample_begin)
    return fail(RTRB_ERR_INVALID, "empty sample range [%d, %d)", sample_begin, sample_end);
  if (!rays_out) return fail(RTRB_ERR_INVALID, "rays_out is NULL");
  const unsigned long long n =
      (unsigned long long)(win.x1 - win.x0) * (unsigned long long)(win.y1 - win.y0) * (unsigned long long)(sample_end - sample_begin);
  if (n > 0x7fffffffull) return fail(RTRB_ERR_UNSUPPORTED, "%llu rays: more than one ray call takes", n);
  if ((rc = ray_device(r))) return rc;
  const bool dev = opts->device_buffers == 1;
  if (dev && ((rc = check_device_ptr(r, rays_out, "rays_out")) || (rc = check_device_ptr(r, keys_or_null, "keys")))) return rc;
  cudaStream_t s = opts->stream ? (cudaStream_t)opts->stream : r->stream;
  if ((rc = r->ray_lens.ensure(cam, s))) return rc;  // the frames' lens tables are not touched
  RayBatch B;
  memset(&B, 0, sizeof(B));
  B.n = (long long)n; B.sample_begin = sample_begin; B.sample_end = sample_end;
  if (dev) {
    B.rays_out = (double*)rays_out; B.keys_out = keys_or_null;
  } else {
    const size_t bytes[2] = {(size_t)n * sizeof(rtrb_ray), keys_or_null ? (size_t)n * 2 * sizeof(uint32_t) : 0};
    uint8_t* p[2];
    if ((rc = ray_stage(r, bytes, 2, p))) return rc;
    B.rays_out = (double*)p[0]; B.keys_out = (uint32_t*)p[1];
  }
  FrameParams P;
  memset(&P, 0, sizeof(P));
  bake_camera(P, cam);
  P.x0 = win.x0; P.y0 = win.y0; P.x1 = win.x1; P.y1 = win.y1;
  P.lens_sx = r->ray_lens.tab.p; P.lens_sy = r->ray_lens.tab.p + W;
  P.key0 = (uint32_t)opts->seed; P.key1 = (uint32_t)(opts->seed >> 32);
  CUDA_TRY(rtrb_launch_camera_rays(P, B, s));
  g_launches++;
  if (!dev) {
    CUDA_TRY(cudaMemcpyAsync(rays_out, B.rays_out, (size_t)n * sizeof(rtrb_ray), cudaMemcpyDeviceToHost, s));
    if (keys_or_null) CUDA_TRY(cudaMemcpyAsync(keys_or_null, B.keys_out, (size_t)n * 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
  }
  return RTRB_OK;
}

int rtrb_tile_partition(int width, int height, const int32_t* window, int tile_rank, int tile_world,
                        int32_t* tiles_out, int capacity, int* count_out) {
  if (width <= 0 || height <= 0 || !count_out) return fail(RTRB_ERR_INVALID, "bad argument");
  static const int32_t whole[4] = {0, 0, 0, 0};
  if (!window) window = whole;
  Window win;
  int rc = make_window(width, height, window[0], window[1], window[2], window[3], tile_rank, tile_world, win);
  if (rc) return rc;
  std::vector<int32_t> t;
  enumerate_tiles(width, win, t);
  *count_out = (int)t.size();
  if (tiles_out)
    for (int i = 0; i < (int)t.size() && i < capacity; ++i) tiles_out[i] = t[i];
  return RTRB_OK;
}

int rtrb_progressive_create(rtrb_renderer* r, const rtrb_camera_desc* cam, const rtrb_render_opts* opts_in,
                            rtrb_progressive** out) {
  if (!out) return fail(RTRB_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (!r || !cam) return fail(RTRB_ERR_INVALID, "renderer/camera is NULL");
  int rc = check_frame_camera(cam);
  if (rc) return rc;
  const rtrb_render_opts opts = opts_or_default(opts_in);
  if (opts.rng_mode == RTRB_RNG_MT)
    return fail(RTRB_ERR_UNSUPPORTED, "progressive frames draw from the counter RNG (RTRB_RNG_MT is a blocking validation mode)");
  if (opts.rng_mode != RTRB_RNG_CTR) return fail(RTRB_ERR_INVALID, "unknown rng_mode %d", opts.rng_mode);
  const int W = cam->width, H = cam->height;
  Window win;
  if ((rc = check_frame_opts(opts, W, H, win))) return rc;
  if ((rc = require_device())) return rc;
  CUDA_TRY(cudaSetDevice(r->device));
  std::unique_ptr<rtrb_progressive> p(new rtrb_progressive());
  FrameParams& P = p->P;
  memset(&P, 0, sizeof(P));
  const bool strict = opts.precision == RTRB_PREC_STRICT;
  if ((rc = pick_trace_kernels(r, strict, cam->trace_depth, cam->monte_carlo_diffusion_times, opts.count_detail != 0, P,
                               &p->capacity)))
    return rc;
  const cudaStream_t s = opts.stream ? (cudaStream_t)opts.stream : r->stream;
  const int S = cam->pre_sample_times, E = cam->max_sample_times > S ? cam->max_sample_times - S : 0;
  p->r = r; p->stream = s; p->strict = strict; p->S = S; p->E = E;
  p->W = W; p->H = H; p->format = opts.pixel_format;
  const cudaError_t ce = p->fc.init();
  if (ce != cudaSuccess) return fail(RTRB_ERR_CUDA, "control block init failed: %s", cudaGetErrorString(ce));
  if ((rc = p->tiles.ensure(W, H, win, s)) || (rc = p->lens.ensure(cam, s))) return rc;
  const int n_tiles = (int)p->tiles.host.size();
  const size_t n_slots = (size_t)n_tiles * RTRB_SUPER_PIXELS, px = (size_t)W * H;
  if ((rc = check_sample_budget(n_slots, S, E, true))) return rc;
  CUDA_TRY(p->samples.ensure(std::max<size_t>(1, n_slots * S * 3)));
  CUDA_TRY(p->extra_list.ensure(std::max<size_t>(1, n_slots)));
  if (E > 0) {
    CUDA_TRY(p->extra_samples.ensure(n_slots * E * 3));
    CUDA_TRY(p->pre_avg.ensure(n_slots * 3));
  }
  // its outputs: pixels outside the window or the rank's tiles read 0, hit id -3
  p->frame_bytes = RTRB_FRAME_BYTES(W, H, opts.pixel_format);
  p->own_frame = opts.rgba_device_out == nullptr;
  if (p->own_frame) {
    CUDA_TRY(p->frame.ensure(p->frame_bytes));
    CUDA_TRY(cudaMemsetAsync(p->frame.p, 0, p->frame_bytes, s));
  }
  if (!(opts.skip_outputs & RTRB_SKIP_RGB)) {
    CUDA_TRY(p->rgb.ensure(px * 3));
    CUDA_TRY(cudaMemsetAsync(p->rgb.p, 0, px * 3 * sizeof(double), s));
  }
  if (!(opts.skip_outputs & RTRB_SKIP_HIT)) {
    CUDA_TRY(p->hit.ensure(px));
    if (!win.whole) prefill_hits(p->hit.p, W, H, s);
  }
  bake_frame(r, cam, P);
  P.key0 = (uint32_t)opts.seed; P.key1 = (uint32_t)(opts.seed >> 32);
  P.x0 = win.x0; P.y0 = win.y0; P.x1 = win.x1; P.y1 = win.y1;
  P.n_tiles = n_tiles; P.stx_count = (W + RTRB_SUPER - 1) / RTRB_SUPER; P.tiles = p->tiles.dev.p;
  P.tiles_magic = win.whole ? p->tiles.magic : 0u;
  P.lens_sx = p->lens.tab.p; P.lens_sy = p->lens.tab.p + W;
  P.samples = p->samples.p; P.rgb = p->rgb.p; P.hit = p->hit.p;
  P.rgba = p->own_frame ? p->frame.p : (uint8_t*)opts.rgba_device_out;
  P.pre_avg = p->pre_avg.p; P.extra_list = p->extra_list.p; P.extra_samples = p->extra_samples.p;
  P.pixel_format = opts.pixel_format;
  P.fuse_resolve = RTRB_RESOLVE_SAMPLE_BUFFER;
  bind_ctl(P, p->fc);
  CUDA_TRY(cudaMemsetAsync(p->fc.blk, 0, sizeof(CtlBlock), s));
  FrameCtl& fc = p->fc;
  fc.W = W; fc.H = H; fc.n_tiles = n_tiles; fc.detail = P.count_detail != 0; fc.px_count = p->tiles.px_count;
  p->scene_gen = r->scene_gen;
  *out = p.release();
  return RTRB_OK;
}

int rtrb_progressive_pass(rtrb_progressive* p, int sample_end, rtrb_stats* stats_out) {
  if (!p) return fail(RTRB_ERR_INVALID, "progressive frame is NULL");
  if (p->done >= p->S) return fail(RTRB_ERR_INVALID, "the frame is final: its last pass has run");
  if (sample_end <= p->done || sample_end > p->S)
    return fail(RTRB_ERR_INVALID, "sample_end %d outside (%d, %d]", sample_end, p->done, p->S);
  rtrb_renderer* r = p->r;
  if (r->scene_gen != p->scene_gen)
    return fail(RTRB_ERR_INVALID, "scene changed: rtrb_scene_update replaced the scene after the frame was created");
  CUDA_TRY(cudaSetDevice(r->device));
  const cudaStream_t s = p->stream;
  bool fresh_scene;
  int rc = enter_scene_stream(r, s, &fresh_scene);
  if (rc) return rc;
  FrameCtl& fc = p->fc;
  FrameParams& P = p->P;
  P.pass_begin = p->done; P.pass_end = sample_end;
  const bool final = sample_end == p->S;
  const size_t n_slots = (size_t)P.n_tiles * RTRB_SUPER_PIXELS;
  const unsigned grid = (unsigned)((n_slots + 255) / 256);
  fc.timed = stats_out != nullptr;
  if (fc.timed) CUDA_TRY(cudaEventRecord(fc.ev0, s));
  // the counters accumulate over the passes, except adaptive_pixels: each resolve counts the frame it resolves
  CUDA_TRY(cudaMemsetAsync(&fc.blk->counters[RTRB_CNT_ADAPTIVE], 0, sizeof(unsigned long long), s));
  if (P.n_tiles > 0) {
    if (fc.timed) CUDA_TRY(cudaEventRecord(fc.evt0, s));
    CUDA_TRY(p->strict ? rtrb_launch_trace_pass_strict(P, p->capacity, s) : rtrb_launch_trace_pass_fast(P, p->capacity, s));
    g_launches++;
    if (fc.timed) CUDA_TRY(cudaEventRecord(fc.evt1, s));
    if (!final) {
      // the preview is the frame of pre = max = sample_end samples
      FrameParams Q = P;
      Q.pre = sample_end; Q.max_samples = sample_end;
      resolve_prefix_kernel<<<grid, 256, 0, s>>>(Q, p->S);
      CUDA_TRY(cudaGetLastError());
      g_launches++;
    } else {
      // render_at's tail as a one-shot sample-buffer frame runs it
      resolve_kernel<<<grid, 256, 0, s>>>(P);
      CUDA_TRY(cudaGetLastError());
      g_launches++;
      if (p->E > 0) {
        CUDA_TRY(p->strict ? rtrb_launch_trace_extra_strict(P, p->capacity, s) : rtrb_launch_trace_extra_fast(P, p->capacity, s));
        g_launches++;
        resolve_extra_kernel<<<296, 256, 0, s>>>(P);
        CUDA_TRY(cudaGetLastError());
        g_launches++;
      }
    }
  }
  if (fc.timed) CUDA_TRY(cudaEventRecord(fc.ev1, s));
  p->done = sample_end;
  fc.S = sample_end; fc.E = final ? p->E : 0;
  return stats_out ? read_stats(fc, s, stats_out) : RTRB_OK;
}

int rtrb_progressive_download(rtrb_progressive* p, uint8_t* frame, double* rgb_or_null, int32_t* hit_or_null) {
  if (!p) return fail(RTRB_ERR_INVALID, "progressive frame is NULL");
  if (p->done == 0) return fail(RTRB_ERR_INVALID, "no pass has run yet");
  CUDA_TRY(cudaSetDevice(p->r->device));
  const cudaStream_t s = p->stream;
  const size_t px = (size_t)p->W * p->H;
  if (frame) {
    if (!p->own_frame) return fail(RTRB_ERR_INVALID, "the frame is written to rgba_device_out, not to its own buffer");
    CUDA_TRY(cudaMemcpyAsync(frame, p->frame.p, p->frame_bytes, cudaMemcpyDeviceToHost, s));
  }
  if (rgb_or_null) {
    if (!p->rgb.p) return fail(RTRB_ERR_INVALID, "the frame keeps no float RGB (RTRB_SKIP_RGB)");
    CUDA_TRY(cudaMemcpyAsync(rgb_or_null, p->rgb.p, px * 3 * sizeof(double), cudaMemcpyDeviceToHost, s));
  }
  if (hit_or_null) {
    if (!p->hit.p) return fail(RTRB_ERR_INVALID, "the frame keeps no hit ids (RTRB_SKIP_HIT)");
    CUDA_TRY(cudaMemcpyAsync(hit_or_null, p->hit.p, px * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  return RTRB_OK;
}

int rtrb_progressive_frame_ptr(rtrb_progressive* p, void** ptr_out) {
  if (!p || !ptr_out) return fail(RTRB_ERR_INVALID, "bad argument");
  *ptr_out = p->P.rgba;
  return RTRB_OK;
}

int rtrb_progressive_destroy(rtrb_progressive* p) {
  if (!p) return RTRB_OK;
  cudaSetDevice(p->r->device);
  cudaDeviceSynchronize();  // its passes may still be writing its buffers
  delete p;
  return RTRB_OK;
}

int rtrb_last_mt_passes(rtrb_renderer* r) { return r ? r->mt.iterations : 0; }

int rtrb_measure_fma_peak(int device, int which, double* tflops_out) {
  if (!tflops_out) return fail(RTRB_ERR_INVALID, "tflops_out is NULL");
  return which == 0 ? measure_fma<float>(device, tflops_out) : measure_fma<double>(device, tflops_out);
}

#pragma GCC visibility pop
}  // extern "C"
