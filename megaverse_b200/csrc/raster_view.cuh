// K4: batched first-person rasteriser -- ONE persistent kernel, one CTA per (view, row band), everything between the
// instance list and the finished pixels lives in shared memory.
//
//   The persistent grid (2 CTAs per SM) draws the envs in the order of what their views cost in the previous launch, most expensive
//   first (the last CTA to leave counting-sorts them; the step kernel steps the envs in the same order).
//   per work item (view, band), 256 threads:
//     1. the env's instance list (MvInstance, 80 B each, draw order) arrives in chunks of 128 by TMA bulk copies
//        (cp.async.bulk + mbarrier, double-buffered: chunk c+1 flies while chunk c is processed)
//     2. instance pass, one thread per instance: model-view product, conservative frustum test of the bounding sphere,
//        normal matrix, per-face back-face test of boxes -> struct-of-arrays transform table in shared memory
//     3. item pass, one thread per (visible box face | mesh triangle): object-space back-face test of mesh triangles, vertices,
//        near/far clip, projection, 8-bit sub-pixel
//        snap, integer edge set-up with the top-left rule folded into the constants -> TriCover / TriShade records appended
//        to the CTA's triangle list IN SHARED MEMORY (no global scratch, no global atomics)
//     4. binning, once per batch, all threads: every (tile, triangle) pair of a triangle's pixel box is tested edge by edge against
//        the tile's samples (exact integers, conservative) -> one bit per list entry in the tile's bin (shared memory)
//     5. tile pass, warps pull 32x4-pixel tiles of the band from a shared-memory counter and walk the tile's bin in list order: the
//        whole warp evaluates each triangle (lane = 4 adjacent pixels, best fragment in registers); exact integer edge functions,
//        nearest depth wins, later draw wins ties (LESS_OR_EQUAL); the single winner per pixel is shaded (deferred) and
//        each lane stores its 4 pixels with one 128-bit store -- 8 lanes cover one full 128-byte line of the obs tensor
//   A view with more triangles than the list holds is drawn in several batches: the per-pixel best fragment of earlier
//   batches is parked in a per-CTA global spill slab, already shaded pixels are marked and only repainted when a later
//   batch wins them.  Nothing is ever dropped (the r1 MV_FAULT_TRI_OVERFLOW cannot occur).
//
// Replaces (file:line under /root/reference):
//   V4R CommandStreamState::render        src/3rdparty/v4r/src/vulkan_state.inl:10-160
//   vertex / fragment shaders             src/3rdparty/v4r/src/pipelines/shaders/uber.vert:53-110, uber.frag:112-141
//   projection                            src/3rdparty/v4r/src/v4r.cpp:35-45
//   raster + depth state                  src/3rdparty/v4r/src/vulkan_state.cpp:588-606
//   image -> linear buffer copy           src/3rdparty/v4r/src/vulkan_state.cpp:909-957 (obs layout uint8[N][H][W][4])
//   instance lists, draw order            src/libs/v4r_rendering/src/v4r_env_renderer.cpp:267-279
#pragma once
#include "dev_math.cuh"
#include "mesh_tables.inc"
#include "mv_types.h"

namespace mvr {
using namespace dm;

struct __align__(16) TriCover {  // what the coverage / depth loop reads (broadcast loads)
    long long C[3];     // edge constant terms, top-left bias already applied
    int32_t A[3], B[3];
    float z[3];
    float invArea;
    uint32_t key;       // draw order + 1 (later wins depth ties: LESS_OR_EQUAL)
    int32_t flags;      // bits 0..2: edge e is top-left (no bias was applied); bit 3: every edge function fits int32 in the viewport;
                        // bit 4: the three vertex normals are identical (box faces, cone and cylinder caps)
    uint32_t bx, by;    // pixel box, inclusive: x0 | x1 << 16, y0 | y1 << 16
};
struct __align__(16) TriShade {  // what deferred shading reads for the winning fragment
    float rw[3];
    float p[9];
    float n[9];        // fast shading, flat triangle (flags bit 4): n[0..2] is the UNIT normal
    float diffuse[3];  // the material colour (palette entry), looked up once per triangle
};
static_assert(sizeof(TriCover) == 80 && sizeof(TriShade) == 96, "triangle record layout");

#ifndef MV_VIEW_THREADS
#define MV_VIEW_THREADS 256
#endif
#ifndef MV_VIEW_MIN_CTAS
#define MV_VIEW_MIN_CTAS 2
#endif
constexpr int kThreads = MV_VIEW_THREADS;     // per CTA
constexpr int kWarps = kThreads / 32;
#ifndef MV_VIEW_INST_CHUNK
#define MV_VIEW_INST_CHUNK 128
#endif
constexpr int kInstChunk = MV_VIEW_INST_CHUNK;   // instances per TMA chunk (one thread each in the instance pass)
static_assert(kInstChunk <= kThreads && kInstChunk <= 128, "one thread per instance of a chunk; slow-list entries keep 7 bits of it");
constexpr int kXfWords = 23;      // per instance: model-view (12: three rows of each column), normal matrix (9), colour, mesh | face mask << 8
constexpr int kClipVerts = 6;     // a triangle clipped by two planes has at most 5 vertices
constexpr int kMaxBandTiles = 128;  // 32x4 tiles of one (view, band) work item (the host keeps to it)
constexpr uint32_t kSmemOptin = 232448u;  // shared memory one CTA may opt in to on sm_100 (227 KB)
// a fragment is (~depth bits << 32) | (draw-order key << kIdxBits) | index in the CTA's triangle list
constexpr int kIdxBits = 10;
constexpr uint32_t kStaleIdx = (1u << kIdxBits) - 1u;  // "already shaded in an earlier batch"
constexpr int kMaxTriCap = int(kStaleIdx);             // list indices 0 .. kStaleIdx - 1
constexpr int kKeyBits = 32 - kIdxBits;                // key = instance * 128 + triangle-in-mesh + 1
constexpr int kMaxInstancesPerEnv = (1 << (kKeyBits - 7)) - 1;
static_assert(MV_CAPSULE_TRIS <= 128 && MV_SPHERE_TRIS <= 128 && MV_CONE_TRIS <= 128 && MV_CYLINDER_TRIS <= 128, "triangle-in-mesh index needs 7 bits");

// mesh tables staged in shared memory (divergent indexing would serialise in the constant cache)
constexpr int kVBox = 0, kVCapsule = kVBox + MV_BOX_VERTS, kVSphere = kVCapsule + MV_CAPSULE_VERTS, kVCone = kVSphere + MV_SPHERE_VERTS,
              kVCylinder = kVCone + MV_CONE_VERTS, kMeshVerts = kVCylinder + MV_CYLINDER_VERTS;
constexpr int kICapsule = 0, kISphere = kICapsule + MV_CAPSULE_TRIS * 3, kICone = kISphere + MV_SPHERE_TRIS * 3, kICylinder = kICone + MV_CONE_TRIS * 3,
              kMeshIdx = kICylinder + MV_CYLINDER_TRIS * 3;

struct ViewParams {
    const MvInstance *instances; // [E][instStride] drawables in draw order (boxes first)
    const int32_t *instCounts;   // [E][8] {boxes, total, capsules, spheres, cones, cylinders, -, -}
    const float *views;          // [E*A][16]
    int instStride;
    uint8_t *obs;                // [N][H][W][4]
    float *depth;                // [N][H][W] or nullptr
    uint32_t *workCounter;       // persistent work queue: claim = atomicAdd(counter, 1) - counterBase (never reset: the host advances the base)
    uint32_t counterBase;
    const uint32_t *ready;       // [E] step-kernel completion stamps (nullptr: plain stream order)
    uint32_t readyStamp;         // value ready[env] holds once this step's state, instances and views of env are written
    uint32_t *consumed;          // optional [E]: += 1 when a work item of env has read the env's instance list and view (step/raster overlap)
    unsigned long long *stats;   // optional [16]: work items, instances, visible instances, items, clipped items, triangles, batches, item
                                 // sub-passes, then thread-0 cycles: head (claim, stamp, view), TMA waits, instance passes, item passes, final
                                 // binning + tile pass, whole item; then (tile, triangle) pairs: kept by the binning (evaluated), in the pixel boxes
    unsigned long long *spill;   // [gridDim.x][spillStride] per-CTA fragment slab for views drawn in several batches
    int spillStride;             // >= W * bandRows
    // cost-ordered work queue (optional; viewBase == 0, N = E * A): claim c draws item c % (A * bands) of env order[c / (A * bands)].  Every
    // CTA writes the SM cycles a work item took into viewCost; the last CTA to leave sorts the ENVS by the cost of their items, descending
    // (counting sort over 256 cost classes), into `order` for the next launch -- so the persistent CTAs do not run dry at very different
    // times (an expensive view started last is the kernel's tail).  The step kernel steps the envs in the same order, so that the envs
    // this grid asks for first are also the first to be ready.
    uint32_t *viewCost;          // [N * bands] (indexed like the work items: view * bands + band) or nullptr
    uint32_t *order;             // [E] a permutation of the envs
    uint32_t *exitCounter;       // CTAs that have left (the last one sorts)
    // progressive host delivery (optional): sliceDone[env / envsPerSlice] += 1 when a work item is completely drawn (frames visible device-wide),
    // so that a copy stream blocked on the counter can start downloading a slice of whole envs while the rest of the batch is still being
    // drawn; the cost order is then slice-major (slices complete one after the other)
    uint32_t *sliceDone;
    int envsPerSlice;
    int viewBase, N;             // this launch draws views [viewBase, viewBase + N)
    int A, W, H;
    int bands, bandRows;         // bandRows: multiple of 4; bands * bandRows >= H
    int triCap;                  // triangle list capacity of a CTA (shared memory), <= kMaxTriCap
    float p00, p11, p22, p32;
};

struct SmemLayout { uint32_t stage, cover, shade, xf, off, meshV, meshI, slow, sched, misc, bins, clip, binTiles, total; };
struct ViewMisc {
    float view[16];
    int32_t counts[8];
    int32_t nTris;      // append counter of the current batch (may run past triCap: the excess is retried in the next batch)
    int32_t nValid;     // first refused list index of the current batch (INT_MAX: none)
    int32_t tileCtr;    // next tile of the band (binTris sets it to the first tile of its round)
    uint32_t claim;     // this work item; claimed (and, when its env was ready, its view / counts / first chunk fetched) during the previous tile pass
    int32_t prefetched;
    int32_t lastCta;    // cost-ordered queue: this CTA is the last one to leave the grid (it sorts the views for the next launch)
    int32_t wsum[kWarps];
    int32_t nSlow[2];   // entries of the two slow-item lists (alternating per item sub-pass)
    uint32_t stat[10];  // debug counters of the current work item (stats slots 0..7, then 14, 15)
    alignas(8) unsigned long long bar[2];
    unsigned long long itemStart;  // clock64 when thread 0 started the current work item (after the wait for its env)
};
// per-tile bins: one bit per list entry, `binWords` words per tile
__host__ __device__ inline int binWords(int triCap) { return (triCap + 31) >> 5; }
__host__ __device__ inline SmemLayout smemLayout(int triCap) {
    SmemLayout L;
    uint32_t o = 0;
    L.stage = o; o += 2u * kInstChunk * uint32_t(sizeof(MvInstance));
    L.cover = o; o += uint32_t(triCap) * uint32_t(sizeof(TriCover));
    L.shade = o; o += uint32_t(triCap) * uint32_t(sizeof(TriShade));
    L.xf = o; o += uint32_t(kXfWords) * kInstChunk * 4u;
    L.off = o; o += (kInstChunk + 4u) * 4u;
    L.meshV = o; o += uint32_t(kMeshVerts) * 6u * 4u;
    L.meshI = o; o += (uint32_t(kMeshIdx) + 15u) & ~15u;
    L.slow = o; o += 2u * kThreads * 2u;                        // two lists of at most one entry per thread
    L.sched = o; o += 256u * 4u;                                // cost classes of the counting sort (last CTA of a cost-ordered launch)
    L.misc = o; o += (uint32_t(sizeof(ViewMisc)) + 15u) & ~15u;
    // the tile bins of the current batch (binning + tile pass) -- the same bytes hold the warps' clip polygons during the item pass (per
    // warp 4 x kClipVerts x 40 B = 960 B <= 1024 B): neither keeps state across the other (the bins are rebuilt per batch once the item
    // pass has finished the list, the polygons per clipped item).  Bins for kMaxBandTiles tiles where shared memory allows (up to
    // tri_cap 640 that is no more than the clip polygons take); at the largest lists only what fits, and the tile pass then bins and
    // draws a band in several rounds of binTiles tiles.
    const uint32_t clipBytes = uint32_t(kWarps) * 1024u, tileBytes = uint32_t(binWords(triCap)) * 4u;
    uint32_t binBytes = uint32_t(kMaxBandTiles) * tileBytes;
    if (o + binBytes > kSmemOptin) binBytes = o + clipBytes < kSmemOptin ? (kSmemOptin - o) / tileBytes * tileBytes : 0u;
    binBytes = binBytes > clipBytes ? binBytes : clipBytes;
    L.bins = o; o += binBytes;
    L.clip = L.bins;
    L.binTiles = binBytes / tileBytes;
    L.total = o;
    return L;
}

// ---------------------------------------------------------------- TMA (1-D bulk async copy) helpers
__device__ __forceinline__ uint32_t smemAddrOf(const void *p) { return uint32_t(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbarInit(unsigned long long *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smemAddrOf(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbarExpectTx(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smemAddrOf(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulkG2S(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smemAddrOf(dst)), "l"(src), "r"(bytes),
                 "r"(smemAddrOf(bar))
                 : "memory");
}
__device__ __forceinline__ void mbarWait(unsigned long long *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smemAddrOf(bar)), "r"(parity)
            : "memory");
    } while (!done);
}

__constant__ float c_palette[22][3];

struct ClipVert { float cx, cy, cz, cw, px, py, pz, nx, ny, nz; };  // clipNearFar indexes it as float[10]
static_assert(sizeof(ClipVert) == 40, "ClipVert is ten floats");

__device__ __forceinline__ ClipVert lerpVert(const ClipVert &a, const ClipVert &b, float t) {
    ClipVert o;
    o.cx = a.cx + t * (b.cx - a.cx); o.cy = a.cy + t * (b.cy - a.cy); o.cz = a.cz + t * (b.cz - a.cz); o.cw = a.cw + t * (b.cw - a.cw);
    o.px = a.px + t * (b.px - a.px); o.py = a.py + t * (b.py - a.py); o.pz = a.pz + t * (b.pz - a.pz);
    o.nx = a.nx + t * (b.nx - a.nx); o.ny = a.ny + t * (b.ny - a.ny); o.nz = a.nz + t * (b.nz - a.nz);
    return o;
}
__device__ __forceinline__ int32_t snapSub(float v) { return int32_t(floorf(v * 256.0f + 0.5f)); }

struct SetupCtx {
    TriCover *cover;      // shared memory
    TriShade *shade;
    int32_t *nTris;       // shared-memory append counter (runs past triCap when the list is full)
    int32_t *nValid;      // shared memory: first list index that was refused in this batch (min over refusals)
    int triCap;
    int W, H;
    int rowLo, rowHi;     // the band's pixel rows, inclusive
};
// All triangles of one item are appended with ONE reservation (all or nothing), so an item that does not fit leaves nothing behind and is
// simply retried in the next batch; the first reservation of a batch always fits.  (The context travels by value, so the compiler no
// longer sees that the counters live in shared memory: say it.)  Returns the first slot or -1.
// index of the n-th (0-based) set bit of a six-bit face mask (__fns is a long software loop)
__device__ __forceinline__ int nthFace(unsigned mask, int n) {
    int face = 0, seen = 0;
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        const int bit = int(mask >> f) & 1;
        if (bit && seen == n) face = f;
        seen += bit;
    }
    return face;
}
__device__ __forceinline__ int reserveTris(const SetupCtx &cx, int n) {
    int base;
    asm volatile("atom.shared.add.s32 %0, [%1], %2;" : "=r"(base) : "r"(smemAddrOf(cx.nTris)), "r"(n) : "memory");
    if (base + n <= cx.triCap) return base;
    asm volatile("red.shared.min.s32 [%0], %1;" ::"r"(smemAddrOf(cx.nValid)), "r"(base) : "memory");
    return -1;
}

struct ScreenVert { int32_t sx, sy; float sz, rw; };
__device__ __forceinline__ ScreenVert projectVert(const ClipVert &v, float hw, float hh) {
    ScreenVert o;
    const float r = 1.0f / v.cw;
    o.rw = r;
    o.sx = snapSub((v.cx * r) * hw + hw);
    o.sy = snapSub((v.cy * r) * hh + hh);
    o.sz = v.cz * r;
    return o;
}
// winding, pixel box: does the projected triangle touch a pixel centre of this band at all?
struct TriBox { long long area2; uint32_t bx, by; };
__device__ __forceinline__ bool triBox(const SetupCtx &cx, const ScreenVert &a, const ScreenVert &b, const ScreenVert &c, TriBox &o) {
    o.area2 = (long long)(b.sx - a.sx) * (long long)(c.sy - a.sy) - (long long)(b.sy - a.sy) * (long long)(c.sx - a.sx);
    if (o.area2 >= 0) return false;  // back-facing (visually clockwise with y down) or degenerate
    const int32_t minx = min(a.sx, min(b.sx, c.sx)), maxx = max(a.sx, max(b.sx, c.sx));
    const int32_t miny = min(a.sy, min(b.sy, c.sy)), maxy = max(a.sy, max(b.sy, c.sy));
    const int px0 = max(0, (minx - 128 + 255) >> 8), px1 = min(cx.W - 1, (maxx - 128) >> 8);
    const int py0 = max(0, (miny - 128 + 255) >> 8), py1 = min(cx.H - 1, (maxy - 128) >> 8);
    if (px0 > px1 || py0 > py1) return false;            // covers no pixel centre of the viewport
    if (py0 > cx.rowHi || py1 < cx.rowLo) return false;  // ... or none of this band
    o.bx = uint32_t(px0) | (uint32_t(px1) << 16);
    o.by = uint32_t(py0) | (uint32_t(py1) << 16);
    return true;
}
// edge / plane set-up of one visible triangle into list slot `slot`
template <bool FAST>
__device__ __forceinline__ void writeTri(const SetupCtx &cx, int slot, const ClipVert &va, const ClipVert &vb, const ClipVert &vc, const ScreenVert &a,
                                         const ScreenVert &b, const ScreenVert &c, const TriBox &tb, int color, uint32_t key) {
    TriCover cv;
    TriShade s;
    const int32_t sxs[3] = {a.sx, b.sx, c.sx}, sys[3] = {a.sy, b.sy, c.sy};
    int tl = 0;
    long long worst = 0;
    const long long wsub = (long long)cx.W * 256, hsub = (long long)cx.H * 256;
#pragma unroll
    for (int e = 0; e < 3; ++e) {
        const int ia = (e + 1) % 3, ib = (e + 2) % 3;
        const long long dx = (long long)sxs[ib] - sxs[ia], dy = (long long)sys[ib] - sys[ia];
        const bool topleft = (dy == 0 && dx < 0) || dy > 0;
        cv.A[e] = int32_t(dy);
        cv.B[e] = int32_t(-dx);
        cv.C[e] = dx * sys[ia] - dy * sxs[ia] - (topleft ? 0 : 1);
        tl |= topleft ? (1 << e) : 0;
        const long long bound = llabs(dy) * wsub + llabs(dx) * hsub + llabs(cv.C[e]);
        worst = bound > worst ? bound : worst;
    }
    cv.z[0] = a.sz; cv.z[1] = b.sz; cv.z[2] = c.sz;
    s.rw[0] = a.rw; s.rw[1] = b.rw; s.rw[2] = c.rw;
    s.p[0] = va.px; s.p[1] = va.py; s.p[2] = va.pz; s.p[3] = vb.px; s.p[4] = vb.py; s.p[5] = vb.pz; s.p[6] = vc.px; s.p[7] = vc.py; s.p[8] = vc.pz;
    s.n[0] = va.nx; s.n[1] = va.ny; s.n[2] = va.nz; s.n[3] = vb.nx; s.n[4] = vb.ny; s.n[5] = vb.nz; s.n[6] = vc.nx; s.n[7] = vc.ny; s.n[8] = vc.nz;
    const bool flat = va.nx == vb.nx && va.ny == vb.ny && va.nz == vb.nz && va.nx == vc.nx && va.ny == vc.ny && va.nz == vc.nz;
    if (FAST && flat) {  // the fast fragment stage takes the unit normal as is (the exact one normalises the interpolated normal per pixel)
        const float inv = rsqrtf(va.nx * va.nx + va.ny * va.ny + va.nz * va.nz);
        s.n[0] = va.nx * inv; s.n[1] = va.ny * inv; s.n[2] = va.nz * inv;
    }
    cv.invArea = 1.0f / float(-tb.area2);
    cv.key = key;
    cv.flags = tl | (worst < (1ll << 30) ? 8 : 0) | (flat ? 16 : 0);
    cv.bx = tb.bx;
    cv.by = tb.by;
    s.diffuse[0] = c_palette[color][0]; s.diffuse[1] = c_palette[color][1]; s.diffuse[2] = c_palette[color][2];
    cx.cover[slot] = cv;
    cx.shade[slot] = s;
}

// uber.vert:53-110 for one vertex, in two halves: position (camera space + clip space) and normal.  mv = rows 0..2 of the model-view
// matrix's four columns, nm = inverse transpose of its 3x3.  The item pass computes the positions first and the normals only for
// what survives the screen-space tests (most mesh triangles face away or cover no pixel centre).
__device__ __forceinline__ void vertPosition(ClipVert &cv, const float mv[12], const float *vp, float p00, float p11, float p22, float p32) {
    // Matrix4::transformPoint: accumulate from 0 over the four columns, the translation column times 1 last
    { float acc = 0.0f; acc += mv[0] * vp[0]; acc += mv[3] * vp[1]; acc += mv[6] * vp[2]; acc += mv[9] * 1.0f; cv.px = acc; }
    { float acc = 0.0f; acc += mv[1] * vp[0]; acc += mv[4] * vp[1]; acc += mv[7] * vp[2]; acc += mv[10] * 1.0f; cv.py = acc; }
    { float acc = 0.0f; acc += mv[2] * vp[0]; acc += mv[5] * vp[1]; acc += mv[8] * vp[2]; acc += mv[11] * 1.0f; cv.pz = acc; }
    cv.cx = cv.px * p00;
    cv.cy = cv.py * p11;
    cv.cz = cv.pz * p22 + p32;
    cv.cw = -cv.pz;
}
__device__ __forceinline__ void vertNormal(ClipVert &cv, const float nm[9], const float *vp) {
    cv.nx = nm[0] * vp[3] + nm[3] * vp[4] + nm[6] * vp[5];
    cv.ny = nm[1] * vp[3] + nm[4] * vp[4] + nm[7] * vp[5];
    cv.nz = nm[2] * vp[3] + nm[5] * vp[4] + nm[8] * vp[5];
}
__device__ __forceinline__ ClipVert makeVert(const float mv[12], const float nm[9], const float *vp, float p00, float p11, float p22, float p32) {
    ClipVert cv;
    vertPosition(cv, mv, vp, p00, p11, p22, p32);
    vertNormal(cv, nm, vp);
    return cv;
}

__device__ __forceinline__ bool insideNearFar(const ClipVert &v) { return v.cz >= 0.0f && (v.cw - v.cz) >= 0.0f; }
// Bits of the four side planes a vertex is strictly outside of, in homogeneous clip space (x > w, x < -w, y > w, y < -w; the linear
// inequalities hold for w <= 0 too).  A polygon whose vertices share a bit lies wholly beyond that plane -- clipped against near /
// far or not -- and covers no pixel of the viewport: the reference's rasteriser scissors it away.
__device__ __forceinline__ unsigned sideOutcode(const ClipVert &v) {
    return (v.cx > v.cw ? 1u : 0u) | (v.cx < -v.cw ? 2u : 0u) | (v.cy > v.cw ? 4u : 0u) | (v.cy < -v.cw ? 8u : 0u);
}

enum SetupResult { kSetupDone = 0, kSetupFull = 1, kSetupClip = 2 };  // appended (or invisible) / the list is full / crosses the near or far plane

// One item: a box face -- four vertices, triangles (0,1,2) and (0,2,3) (Magnum cubeSolid index pattern), nTri = 2 -- or a mesh
// triangle (nTri = 1, v3 repeats v2).  v0..v3 carry positions only; vp0..vp3 = the mesh vertices (six floats each) for the normals,
// which are only computed for what survives the screen-space tests.  One copy of the set-up code serves both (code size: the kernel's
// hot loops have to stay inside the instruction cache).
template <bool FAST>
__device__ __forceinline__ SetupResult setupItem(const SetupCtx &cx, ClipVert &v0, ClipVert &v1, ClipVert &v2, ClipVert &v3, int nTri, const float nm[9], const float *vp0,
                                                 const float *vp1, const float *vp2, const float *vp3, int color, uint32_t keyBase) {
    if (sideOutcode(v0) & sideOutcode(v1) & sideOutcode(v2) & sideOutcode(v3)) return kSetupDone;
    if (!(insideNearFar(v0) && insideNearFar(v1) && insideNearFar(v2) && insideNearFar(v3))) {
        // wholly behind the near plane or wholly beyond the far plane: clipping would leave nothing
        if (v0.cz < 0.0f && v1.cz < 0.0f && v2.cz < 0.0f && v3.cz < 0.0f) return kSetupDone;
        if ((v0.cw - v0.cz) < 0.0f && (v1.cw - v1.cz) < 0.0f && (v2.cw - v2.cz) < 0.0f && (v3.cw - v3.cz) < 0.0f) return kSetupDone;
        return kSetupClip;
    }
    const float hw = float(cx.W) * 0.5f, hh = float(cx.H) * 0.5f;
    const ScreenVert s0 = projectVert(v0, hw, hh), s1 = projectVert(v1, hw, hh), s2 = projectVert(v2, hw, hh);
    ScreenVert s3 = s2;
    if (nTri == 2) s3 = projectVert(v3, hw, hh);
    TriBox b0, b1;
    const bool vis0 = triBox(cx, s0, s1, s2, b0), vis1 = nTri == 2 && triBox(cx, s0, s2, s3, b1);
    const int n = (vis0 ? 1 : 0) + (vis1 ? 1 : 0);
    if (!n) return kSetupDone;
    int slot = reserveTris(cx, n);
    if (slot < 0) return kSetupFull;
    vertNormal(v0, nm, vp0); vertNormal(v1, nm, vp1); vertNormal(v2, nm, vp2); vertNormal(v3, nm, vp3);
#pragma unroll 1
    for (int t = 0; t < 2; ++t) {
        if (!(t ? vis1 : vis0)) continue;
        const ClipVert vb = t ? v2 : v1, vc = t ? v3 : v2;
        const ScreenVert sb = t ? s2 : s1, sc = t ? s3 : s2;
        const TriBox tb = t ? b1 : b0;
        writeTri<FAST>(cx, slot++, v0, vb, vc, s0, sb, sc, tb, color, keyBase + uint32_t(t));
    }
    return kSetupDone;
}

// Sutherland-Hodgman of one triangle against z >= 0 and z <= w by a group of 16 lanes: lane c < 10 owns component c of every vertex
// (ClipVert is ten floats), the in/out decisions are the same for all lanes of the group (broadcast reads of the z and w components).
// Polygon and scratch live in SHARED memory (ten floats per vertex, kClipVerts vertices each).  The input triangle is in bufA, so is
// the result; returns the vertex count (0: nothing left).
__device__ __forceinline__ int clipNearFar(float *bufA, float *bufB, int c, unsigned groupMask) {
    float *src = bufA, *dst = bufB;
    int n = 3;
    for (int plane = 0; plane < 2; ++plane) {
        int m = 0;
        for (int i = 0; i < n; ++i) {
            const int i1 = i + 1 == n ? 0 : i + 1;
            const float az = src[i * 10 + 2], aw = src[i * 10 + 3], bz = src[i1 * 10 + 2], bw = src[i1 * 10 + 3];
            const float da = plane == 0 ? az : aw - az;
            const float db = plane == 0 ? bz : bw - bz;
            const bool ina = da >= 0.0f, inb = db >= 0.0f;
            float a = 0.0f, b = 0.0f;
            if (c < 10) { a = src[i * 10 + c]; b = src[i1 * 10 + c]; }
            if (ina) { if (c < 10) dst[m * 10 + c] = a; ++m; }
            if (ina != inb) {  // always interpolate from the inside vertex so that shared edges clip identically (lerpVert)
                float val;
                if (ina) { const float t = da / (da - db); val = a + t * (b - a); }
                else { const float t = db / (db - da); val = b + t * (a - b); }
                if (c < 10) dst[m * 10 + c] = val;
                ++m;
            }
        }
        __syncwarp(groupMask);
        n = m;
        float *sw = src; src = dst; dst = sw;
        if (n < 3) return 0;
    }
    return n;
}

// Conservative instance-level frustum test: the bounding sphere of the instance's mesh in view space against the near plane and the
// four side planes.  Unit meshes span |x|,|z| <= 1 and |y| <= 1 (capsule: 2), so a vertex lies within |col0| + by*|col1| + |col2| of
// the instance origin.  An instance that fails contributes no fragment (every one of its triangles would be clipped or scissored away).
__device__ __forceinline__ bool instanceMayBeVisible(const M4 &mv, float by, float p00, float p11) {
    const float l0 = sqrtf(mv.c[0] * mv.c[0] + mv.c[1] * mv.c[1] + mv.c[2] * mv.c[2]);
    const float l1 = sqrtf(mv.c[4] * mv.c[4] + mv.c[5] * mv.c[5] + mv.c[6] * mv.c[6]);
    const float l2 = sqrtf(mv.c[8] * mv.c[8] + mv.c[9] * mv.c[9] + mv.c[10] * mv.c[10]);
    const float r = (l0 + by * l1 + l2) * 1.001f + 1e-3f;
    const float x = mv.c[12], y = mv.c[13], z = mv.c[14];
    if (-z - 0.01f < -r) return false;  // wholly in front of the near plane (camera looks down -z)
    // side planes x_clip = +-w_clip, y_clip = +-w_clip with x_clip = p00 * x, y_clip = p11 * y, w_clip = -z: inward unit normals
    const float ix = rsqrtf(p00 * p00 + 1.0f), iy = rsqrtf(p11 * p11 + 1.0f);
    const float ax = fabsf(p00), ay = fabsf(p11);
    if ((-ax * x - z) * ix < -r || (ax * x - z) * ix < -r) return false;
    if ((-ay * y - z) * iy < -r || (ay * y - z) * iy < -r) return false;
    return true;
}

// ---------------------------------------------------------------------------------------------------- shading
__device__ __forceinline__ float pow300(float x) {
    const float x2 = x * x, x4 = x2 * x2, x8 = x4 * x4, x16 = x8 * x8, x32 = x16 * x16, x64 = x32 * x32, x128 = x64 * x64, x256 = x128 * x128;
    return ((x256 * x32) * x8) * x4;
}
__device__ __forceinline__ uint32_t toUnorm8(float c) {
    c = c < 0.0f ? 0.0f : (c > 1.0f ? 1.0f : c);
    return uint32_t(floorf(c * 255.0f + 0.5f));
}

template <bool FAST> __device__ __forceinline__ float invLen3(float x, float y, float z) {
    if (FAST) return rsqrtf(__fmaf_rn(z, z, __fmaf_rn(y, y, x * x)));
    return 1.0f / sqrtf((x * x + y * y) + z * z);
}
template <bool FAST> __device__ __forceinline__ float dot3(float ax, float ay, float az, float bx, float by, float bz) {
    if (FAST) return __fmaf_rn(az, bz, __fmaf_rn(ay, by, ax * bx));
    return (ax * bx + ay * by) + az * bz;
}

// uber.frag:112-141.  FAST keeps the structure but uses rsqrt.approx + FMA: colours move by at most 1 LSB (the tolerance the
// north star grants for RGB); the exact variant reproduces the oracle byte for byte.  The depth output is exact in both.
struct ShadeRec { float4 a0, a1, a2, a3, a4, a5; };
__device__ __forceinline__ ShadeRec loadShade(const TriShade *tp) {  // shared memory, 96-byte record as six 128-bit loads
    const float4 *q = reinterpret_cast<const float4 *>(tp);
    ShadeRec r;
    r.a0 = q[0]; r.a1 = q[1]; r.a2 = q[2]; r.a3 = q[3]; r.a4 = q[4]; r.a5 = q[5];
    return r;
}
// The fast variant skips the normal interpolation on flat triangles (the record holds the unit normal) and the highlight where it
// cannot reach a tenth of an LSB.  (Taking the camera-space position from the interpolated w instead of interpolating the vertex
// positions was tried and dropped: the sub-pixel snap of the vertices moves ~0.5 % of the bytes by one LSB.)
template <bool FAST> __device__ __forceinline__ uint32_t shadePixel(const ShadeRec &rec, float l0, float l1, float l2, bool flat, float &wOut) {
    const float4 a0 = rec.a0, a1 = rec.a1, a2 = rec.a2, a3 = rec.a3, a4 = rec.a4, a5 = rec.a5;
    const float rw0 = a0.x, rw1 = a0.y, rw2 = a0.z;
    const float k0 = l0 * rw0, k1 = l1 * rw1, k2 = l2 * rw2;
    const float s = (k0 + k1) + k2;
    const float r = 1.0f / s;
    wOut = r;
    float Pc[3], nn0, nn1, nn2;
    if (FAST) {
        const float p[9] = {a0.w, a1.x, a1.y, a1.z, a1.w, a2.x, a2.y, a2.z, a2.w};
        const float q0 = k0 * r, q1 = k1 * r, q2 = k2 * r;
#pragma unroll
        for (int c = 0; c < 3; ++c) Pc[c] = dot3<true>(q0, q1, q2, p[c], p[3 + c], p[6 + c]);
        if (flat) {
            nn0 = a3.x; nn1 = a3.y; nn2 = a3.z;
        } else {
            const float n[9] = {a3.x, a3.y, a3.z, a3.w, a4.x, a4.y, a4.z, a4.w, a5.x};
            const float N0 = dot3<true>(q0, q1, q2, n[0], n[3], n[6]), N1 = dot3<true>(q0, q1, q2, n[1], n[4], n[7]), N2 = dot3<true>(q0, q1, q2, n[2], n[5], n[8]);
            const float nni = invLen3<true>(N0, N1, N2);
            nn0 = N0 * nni; nn1 = N1 * nni; nn2 = N2 * nni;
        }
    } else {
        const float p[9] = {a0.w, a1.x, a1.y, a1.z, a1.w, a2.x, a2.y, a2.z, a2.w};
        const float n[9] = {a3.x, a3.y, a3.z, a3.w, a4.x, a4.y, a4.z, a4.w, a5.x};
        const float q0 = k0 * r, q1 = k1 * r, q2 = k2 * r;
        float N[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            Pc[c] = dot3<false>(q0, q1, q2, p[c], p[3 + c], p[6 + c]);
            N[c] = dot3<false>(q0, q1, q2, n[c], n[3 + c], n[6 + c]);
        }
        const float nni = invLen3<false>(N[0], N[1], N[2]);
        nn0 = N[0] * nni; nn1 = N[1] * nni; nn2 = N[2] * nni;
    }
    const float cd0 = -Pc[0], cd1 = -Pc[1], cd2 = -Pc[2];
    const float ld0 = 0.0f + cd0, ld1 = 4.0f + cd1, ld2 = 2.0f + cd2;
    const float ldi = invLen3<FAST>(ld0, ld1, ld2);
    const float nl0 = ld0 * ldi, nl1 = ld1 * ldi, nl2 = ld2 * ldi;
    const float ndl = dot3<FAST>(nn0, nn1, nn2, nl0, nl1, nl2);
    const float intensity = ndl > 0.0f ? ndl : 0.0f;
    float spec = 0.0f;
    if (intensity > 0.001f) {
        const float dni = -ndl;
        const float r0 = -nl0 - (2.0f * dni) * nn0, r1 = -nl1 - (2.0f * dni) * nn1, r2 = -nl2 - (2.0f * dni) * nn2;
        const float cdi = invLen3<FAST>(cd0, cd1, cd2);
        const float vdr = dot3<FAST>(cd0 * cdi, cd1 * cdi, cd2 * cdi, r0, r1, r2);
        const float base = vdr > 0.0f ? vdr : 0.0f;
        if (!FAST || base > 0.97f) {  // 0.97^300 = 1.1e-4: three hundredths of an LSB
            spec = pow300(base);
            spec = spec < 0.0f ? 0.0f : (spec > 1.0f ? 1.0f : spec);
        }
    }
    const float diffuse[3] = {a5.y, a5.z, a5.w};
    uint32_t out = 0xff000000u;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float Lo;
        if (FAST) {
            Lo = __fmaf_rn((0.73f * diffuse[c]) * 0.66f, intensity, 0.33f * diffuse[c]) + spec;
            out |= __float2uint_rn(__saturatef(Lo) * 255.0f) << (8 * c);
        } else {
            Lo = 0.33f * diffuse[c];
            Lo = Lo + ((0.73f * diffuse[c]) * 0.66f) * intensity;
            Lo = Lo + 1.0f * spec;
            out |= toUnorm8(Lo) << (8 * c);
        }
    }
    return out;
}

// ---------------------------------------------------------------------------------------------------- coverage
struct EdgeEval {  // one triangle's edge functions
    int A0, A1, A2, B0, B1, B2, u0, u1, u2, small, flat;
    long long C0, C1, C2;
    float z0, z1, z2, invArea;
    uint32_t key;
};
__device__ __forceinline__ EdgeEval unpackCover(const int4 q0, const int4 q1, const int4 q2, const int4 q3, const int4 q4) {
    EdgeEval e;
    e.C0 = (long long)(((unsigned long long)(unsigned)q0.y << 32) | (unsigned)q0.x);
    e.C1 = (long long)(((unsigned long long)(unsigned)q0.w << 32) | (unsigned)q0.z);
    e.C2 = (long long)(((unsigned long long)(unsigned)q1.y << 32) | (unsigned)q1.x);
    e.A0 = q1.z; e.A1 = q1.w; e.A2 = q2.x; e.B0 = q2.y; e.B1 = q2.z; e.B2 = q2.w;
    e.z0 = __int_as_float(q3.x); e.z1 = __int_as_float(q3.y); e.z2 = __int_as_float(q3.z); e.invArea = __int_as_float(q3.w);
    e.key = uint32_t(q4.x);
    const int fl = q4.y;
    e.u0 = (fl & 1) ? 0 : 1; e.u1 = (fl & 2) ? 0 : 1; e.u2 = (fl & 4) ? 0 : 1;  // undo the top-left bias for the barycentrics
    e.small = (fl >> 3) & 1;
    e.flat = (fl >> 4) & 1;
    return e;
}
__device__ __forceinline__ EdgeEval loadCover(const TriCover *c) {  // shared memory
    const int4 *cq = reinterpret_cast<const int4 *>(c);
    return unpackCover(cq[0], cq[1], cq[2], cq[3], cq[4]);
}
__device__ __forceinline__ unsigned long long packFrag(float z, uint32_t key, int idx) {
    const uint32_t b = __float_as_uint(z);
    const uint32_t asc = b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);  // monotonic in z over all floats (tiny negative z can come out of the clipper)
    return ((unsigned long long)(~asc) << 32) | (unsigned long long)((key << kIdxBits) | uint32_t(idx));
}

// Out of line on purpose: the tile pass (with the binning) is called from two places (a full triangle list in mid-view, the end of the
// view) and two inlined copies of it pushed the kernel's hot code out of the instruction cache (Collect 1024 x 4: 2.65 ms inlined, 1.70 ms called)
#ifdef MV_TILE_FORCEINLINE
#define MV_TILE_INLINE __forceinline__
#else
#define MV_TILE_INLINE __noinline__
#endif
extern __shared__ __align__(128) unsigned char g_viewSmem[];  // the CTA's dynamic shared memory (carved up by smemLayout)

// ---------------------------------------------------------------------------------------------------- work queue
// Next work item of the CTA (called by one thread): an index into [0, total), or >= total when the queue is empty.  Natural order: the
// claim itself; cost-ordered: the view the previous launch's sort put at that position.
__device__ __forceinline__ uint32_t claimWork(const ViewParams &P, uint32_t total) {
    const uint32_t c = atomicAdd(P.workCounter, 1u) - P.counterBase;
    if (P.viewCost && c < total) {
        const uint32_t perEnv = uint32_t(P.A) * uint32_t(P.bands);
        return __ldcg(P.order + c / perEnv) * perEnv + c % perEnv;
    }
    return c;
}

// Claim the next work item now and, if its env's state is already published, fetch its view matrix, its counts and its first instance
// chunk while this item's tiles are drawn (the stage buffers, M.view and M.counts are idle during the tile pass): the global round trips
// of the item head then cost nothing.  One thread (thread 0, after the binning); its warp joins the tile pass a little later.
__device__ __forceinline__ void claimNext(const ViewParams &P) {
    const SmemLayout L = smemLayout(P.triCap);
    MvInstance *stage = reinterpret_cast<MvInstance *>(g_viewSmem + L.stage);
    ViewMisc &M = *reinterpret_cast<ViewMisc *>(g_viewSmem + L.misc);
    const int bands = P.bands;
    const uint32_t total = uint32_t(P.N) * uint32_t(bands);
    const uint32_t nc = claimWork(P, total);
    int pre = 0;
    if (nc < total) {
        const int nview = P.viewBase + int(nc / uint32_t(bands)), nenv = nview / P.A;
        bool ready = true;
        if (P.ready) {
            uint32_t v;
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(P.ready + nenv) : "memory");
            ready = v == P.readyStamp;
            if (ready) asm volatile("fence.proxy.async;" ::: "memory");
        }
        if (ready) {
            float vm[16];
            int32_t cn[8];
#pragma unroll
            for (int q = 0; q < 16; ++q) vm[q] = __ldcg(P.views + size_t(nview) * 16 + q);
#pragma unroll
            for (int q = 0; q < 8; ++q) cn[q] = __ldcg(P.instCounts + nenv * 8 + q);
#pragma unroll
            for (int q = 0; q < 16; ++q) M.view[q] = vm[q];
#pragma unroll
            for (int q = 0; q < 8; ++q) M.counts[q] = cn[q];
            if (cn[1] > 0) {
                const uint32_t bytes = uint32_t(min(cn[1], kInstChunk)) * uint32_t(sizeof(MvInstance));
                mbarExpectTx(&M.bar[0], bytes);
                bulkG2S(stage, P.instances + size_t(nenv) * size_t(P.instStride), bytes, &M.bar[0]);
            }
            pre = 1;
        }
    }
    M.claim = nc; M.prefetched = pre;
}

// Bins of the current batch of `count` triangles for the band's tiles [t0, t1): bit j % 32 of bins[(tile - t0) * binWords + j / 32] is
// set when list entry j may cover a sample of the tile.  Each (tile, triangle) pair of a triangle's pixel box is tested against the tile: every edge function at the
// sample of (tile & box) where it is largest -- exact 64-bit integers, the top-left bias already in C -- and the pair is dropped only
// when one edge is negative there, i.e. at every sample of the tile (a kept pair may still cover nothing; a covered sample is never
// lost).  The pairs are spread over the lanes: a warp takes 32 list entries, scans their box tile counts and then tests one pair per
// lane, so a floor triangle spanning the whole band does not hold up one thread.  Called by all threads, once the list is complete; also
// points the tile counter at t0.
__device__ __forceinline__ void binTris(const ViewParams &P, int count, int rowLo, int t0, int t1) {
    const SmemLayout L = smemLayout(P.triCap);
    const TriCover *cover = reinterpret_cast<const TriCover *>(g_viewSmem + L.cover);
    uint32_t *bins = reinterpret_cast<uint32_t *>(g_viewSmem + L.bins);
    ViewMisc &M = *reinterpret_cast<ViewMisc *>(g_viewSmem + L.misc);
    const int words = binWords(P.triCap), tilesX = P.W >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < (t1 - t0) * words; i += kThreads) bins[i] = 0u;
    if (threadIdx.x == 0) M.tileCtr = t0;
    const int yLo = rowLo + (t0 / tilesX) * 4, yHi = rowLo + ((t1 - 1) / tilesX) * 4 + 3;  // the rows of [t0, t1)
    __syncthreads();
    uint32_t nBox = 0, nKept = 0;
    for (int base = (threadIdx.x >> 5) * 32; base < count; base += kThreads) {
        int n = 0;
        if (base + lane < count) {
            const uint2 bb = *reinterpret_cast<const uint2 *>(&cover[base + lane].bx);
            const int y0 = max(int(bb.y & 0xffffu), yLo), y1 = min(int(bb.y >> 16), yHi);
            if (y0 <= y1) n = ((int(bb.x >> 16) >> 5) - (int(bb.x & 0xffffu) >> 5) + 1) * (((y1 - rowLo) >> 2) - ((y0 - rowLo) >> 2) + 1);
        }
        int incl = n;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += up;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        for (int p0 = 0; p0 < total; p0 += 32) {
            const int p = p0 + lane;
            int o = 0;  // the entry pair p belongs to: the first lane whose inclusive count exceeds p
#pragma unroll
            for (int s = 16; s; s >>= 1)
                if (__shfl_sync(0xffffffffu, incl, o + s - 1) <= p) o += s;
            const int r = p - __shfl_sync(0xffffffffu, incl - n, o);
            bool inRange = false, keep = false;
            if (p < total) {
                const TriCover *c = cover + base + o;
                const uint2 bb = *reinterpret_cast<const uint2 *>(&c->bx);
                const int x0 = int(bb.x & 0xffffu), x1 = int(bb.x >> 16);
                const int y0 = max(int(bb.y & 0xffffu), yLo), y1 = min(int(bb.y >> 16), yHi);
                const int ntx = (x1 >> 5) - (x0 >> 5) + 1, rq = r / ntx;
                const int tx = (x0 >> 5) + (r - rq * ntx), ty = ((y0 - rowLo) >> 2) + rq, tile = ty * tilesX + tx;
                inRange = tile >= t0 && tile < t1;  // (whole tile rows but the first and last of a round)
                // sample centres of the tile inside the box, in 1/256 pixel
                const long long sx0 = max(x0, tx * 32) * 256 + 128, sx1 = min(x1, tx * 32 + 31) * 256 + 128;
                const long long sy0 = max(y0, rowLo + ty * 4) * 256 + 128, sy1 = min(y1, rowLo + ty * 4 + 3) * 256 + 128;
                keep = inRange;
#pragma unroll
                for (int e = 0; e < 3; ++e) {
                    const int A = c->A[e], B = c->B[e];
                    keep = keep && c->C[e] + A * (A > 0 ? sx1 : sx0) + B * (B > 0 ? sy1 : sy0) >= 0;
                }
                if (keep) atomicOr(&bins[(tile - t0) * words + (base >> 5)], 1u << o);
            }
            nKept += uint32_t(__popc(__ballot_sync(0xffffffffu, keep)));
            nBox += uint32_t(__popc(__ballot_sync(0xffffffffu, inRange)));
        }
    }
    if (P.stats && lane == 0) { atomicAdd(&M.stat[8], nKept); atomicAdd(&M.stat[9], nBox); }
    __syncthreads();
}

// All tiles of the band against the current batch of `count` triangles: the batch is binned first (all threads), then the warps draw
// the tiles -- in one round unless the list is so long that shared memory holds the bins of fewer tiles than the band has.  batch 0
// paints every pixel (background included); later batches repaint only the pixels they win.  Unless `final`, the per-pixel best
// fragment is parked in the CTA's spill slab with its list index replaced by kStaleIdx (the list is about to be overwritten); if
// `final`, thread 0 claims the next work item once the first round is binned.
template <bool FAST>
__device__ MV_TILE_INLINE void tilePass(const ViewParams &P, int count, unsigned long long *spill, int view, int rowLo, int bandTiles, int batch, bool final) {
    // addresses derived from the shared-memory symbol itself, so that this out-of-line function keeps shared-space loads
    const SmemLayout L = smemLayout(P.triCap);
    const TriCover *cover = reinterpret_cast<const TriCover *>(g_viewSmem + L.cover);
    const TriShade *shade = reinterpret_cast<const TriShade *>(g_viewSmem + L.shade);
    const uint32_t *bins = reinterpret_cast<const uint32_t *>(g_viewSmem + L.bins);
    int32_t *tileCtr = &reinterpret_cast<ViewMisc *>(g_viewSmem + L.misc)->tileCtr;
    const int lane = threadIdx.x & 31;
    const int tilesX = P.W >> 5, words = binWords(P.triCap), nWords = (count + 31) >> 5;
    for (int t0 = 0; t0 < bandTiles; t0 += int(L.binTiles)) {
        const int t1 = min(bandTiles, t0 + int(L.binTiles));
        if (t0) __syncthreads();  // the previous round's bins and tile counter are no longer read
        binTris(P, count, rowLo, t0, t1);
        if (final && t0 == 0 && threadIdx.x == 0) claimNext(P);
        for (;;) {
            int tile = 0;
            if (lane == 0) tile = atomicAdd(tileCtr, 1);
            tile = __shfl_sync(0xffffffffu, tile, 0);
            if (tile >= t1) break;
            const int tk = tile / tilesX, ty = tk;  // (drawing the tile rows from the middle outwards -- horizon first, sky and floor last -- was measured: no effect)
            const int tx0 = (tile - tk * tilesX) * 32, ty0 = rowLo + ty * 4;
            const int px = tx0 + (lane & 7) * 4, py = ty0 + (lane >> 3);
            const int sx32 = px * 256 + 128, sy32 = py * 256 + 128;
            unsigned long long best[4] = {0ull, 0ull, 0ull, 0ull};
            // the tile's triangles in list order (the result does not depend on it: a max), whole warp, lane = 4 pixels, the record is
            // broadcast from shared memory
            const uint32_t *bin = bins + (tile - t0) * words;
            for (int w = 0; w < nWords; ++w) {
                unsigned bits = bin[w];
                while (bits) {
                    const int ti = w * 32 + __ffs(bits) - 1;
                    bits &= bits - 1;
                    const EdgeEval e2 = loadCover(cover + ti);
                    if (e2.small) {
                        int F0 = int(e2.C0) + e2.A0 * sx32 + e2.B0 * sy32, F1 = int(e2.C1) + e2.A1 * sx32 + e2.B1 * sy32, F2 = int(e2.C2) + e2.A2 * sx32 + e2.B2 * sy32;
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if ((F0 | F1 | F2) >= 0) {
                                const float l0 = float(F0 + e2.u0) * e2.invArea, l1 = float(F1 + e2.u1) * e2.invArea, l2 = float(F2 + e2.u2) * e2.invArea;
                                const float z = (l0 * e2.z0 + l1 * e2.z1) + l2 * e2.z2;
                                if (z <= 1.0f) { const unsigned long long f = packFrag(z, e2.key, ti); best[k] = f > best[k] ? f : best[k]; }
                            }
                            F0 += e2.A0 * 256; F1 += e2.A1 * 256; F2 += e2.A2 * 256;
                        }
                    } else {
                        long long F0 = e2.C0 + (long long)e2.A0 * sx32 + (long long)e2.B0 * sy32, F1 = e2.C1 + (long long)e2.A1 * sx32 + (long long)e2.B1 * sy32,
                                  F2 = e2.C2 + (long long)e2.A2 * sx32 + (long long)e2.B2 * sy32;
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if ((F0 | F1 | F2) >= 0) {
                                const float l0 = float(F0 + e2.u0) * e2.invArea, l1 = float(F1 + e2.u1) * e2.invArea, l2 = float(F2 + e2.u2) * e2.invArea;
                                const float z = (l0 * e2.z0 + l1 * e2.z1) + l2 * e2.z2;
                                if (z <= 1.0f) { const unsigned long long f = packFrag(z, e2.key, ti); best[k] = f > best[k] ? f : best[k]; }
                            }
                            F0 += (long long)e2.A0 * 256; F1 += (long long)e2.A1 * 256; F2 += (long long)e2.A2 * 256;
                        }
                    }
                }
            }
            // ---- merge with the earlier batches, recompute the winner's barycentrics, shade, store
            const int pixInTile = (lane >> 3) * 32 + (lane & 7) * 4;
            unsigned long long *sp = spill + size_t(tile) * 128 + pixInTile;
            unsigned long long f4[4];
            if (batch > 0) {
                const ulonglong2 s01 = *reinterpret_cast<const ulonglong2 *>(sp), s23 = *reinterpret_cast<const ulonglong2 *>(sp + 2);
                f4[0] = s01.x; f4[1] = s01.y; f4[2] = s23.x; f4[3] = s23.y;
            } else {
                f4[0] = f4[1] = f4[2] = f4[3] = 0ull;
            }
            // winners of the lane's four pixels (list index, 0xffff = nothing new to shade), then ONE copy of the fragment stage in a rolled
            // loop: the kernel's hot code has to stay inside the instruction cache (unrolled four times it did not)
            unsigned long long winners = 0ull;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const unsigned long long f = best[k] > f4[k] ? best[k] : f4[k];
                f4[k] = f;
                const uint32_t ti = uint32_t(f) & kStaleIdx;
                const bool fresh = f != 0ull && ti != kStaleIdx;
                winners |= (unsigned long long)(fresh ? ti : 0xffffu) << (16 * k);
            }
            uint32_t o0 = 0xff000000u, o1 = 0xff000000u, o2 = 0xff000000u, o3 = 0xff000000u;
            float w0 = 0.0f, w1 = 0.0f, w2 = 0.0f, w3 = 0.0f;
            // (keeping the records of the previous pixel's triangle in registers across the iterations -- the lane's four pixels mostly belong
            // to one triangle -- was measured: 20 % SLOWER, the loop then spills)
#pragma unroll 1
            for (int k = 0; k < 4; ++k) {
                const uint32_t ti = uint32_t(winners >> (16 * k)) & 0xffffu;
                if (ti == 0xffffu) continue;
                const ShadeRec rec = loadShade(shade + ti);
                const EdgeEval e = loadCover(cover + ti);
                const int sx = sx32 + k * 256;
                float l0, l1, l2;
                if (e.small) {
                    l0 = float(int(e.C0) + e.A0 * sx + e.B0 * sy32 + e.u0) * e.invArea;
                    l1 = float(int(e.C1) + e.A1 * sx + e.B1 * sy32 + e.u1) * e.invArea;
                    l2 = float(int(e.C2) + e.A2 * sx + e.B2 * sy32 + e.u2) * e.invArea;
                } else {
                    l0 = float(e.C0 + (long long)e.A0 * sx + (long long)e.B0 * sy32 + e.u0) * e.invArea;
                    l1 = float(e.C1 + (long long)e.A1 * sx + (long long)e.B1 * sy32 + e.u1) * e.invArea;
                    l2 = float(e.C2 + (long long)e.A2 * sx + (long long)e.B2 * sy32 + e.u2) * e.invArea;
                }
                float w;
                const uint32_t c = shadePixel<FAST>(rec, l0, l1, l2, e.flat != 0, w);
                if (k == 0) { o0 = c; w0 = w; } else if (k == 1) { o1 = c; w1 = w; } else if (k == 2) { o2 = c; w2 = w; } else { o3 = c; w3 = w; }
            }
            const bool fr0 = (winners & 0xffffull) != 0xffffull, fr1 = ((winners >> 16) & 0xffffull) != 0xffffull, fr2 = ((winners >> 32) & 0xffffull) != 0xffffull,
                       fr3 = (winners >> 48) != 0xffffull;
            uint8_t *obsPix = P.obs + ((size_t(view) * P.H + size_t(py)) * P.W + px) * 4;
            float *depthPix = P.depth ? P.depth + (size_t(view) * P.H + size_t(py)) * P.W + px : nullptr;
            if (batch == 0) {
                *reinterpret_cast<uint4 *>(obsPix) = make_uint4(o0, o1, o2, o3);
                if (depthPix) *reinterpret_cast<float4 *>(depthPix) = make_float4(w0, w1, w2, w3);
            } else if (fr0 || fr1 || fr2 || fr3) {  // a later batch won some of this lane's pixels: this lane wrote the others itself, earlier
                uint4 old = *reinterpret_cast<const uint4 *>(obsPix);
                if (fr0) old.x = o0;
                if (fr1) old.y = o1;
                if (fr2) old.z = o2;
                if (fr3) old.w = o3;
                *reinterpret_cast<uint4 *>(obsPix) = old;
                if (depthPix) {
                    float4 od = *reinterpret_cast<const float4 *>(depthPix);
                    if (fr0) od.x = w0;
                    if (fr1) od.y = w1;
                    if (fr2) od.z = w2;
                    if (fr3) od.w = w3;
                    *reinterpret_cast<float4 *>(depthPix) = od;
                }
            }
            if (!final) {
#pragma unroll
                for (int k = 0; k < 4; ++k) f4[k] = f4[k] ? (f4[k] | (unsigned long long)kStaleIdx) : 0ull;
                *reinterpret_cast<ulonglong2 *>(sp) = make_ulonglong2(f4[0], f4[1]);
                *reinterpret_cast<ulonglong2 *>(sp + 2) = make_ulonglong2(f4[2], f4[3]);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------- the kernel
#ifdef MV_VIEW_MAXNREG  // a register cap below what two CTAs per SM allow leaves room for a step-kernel CTA beside them
#define MV_VIEW_BOUNDS __maxnreg__(MV_VIEW_MAXNREG)
#else
#define MV_VIEW_BOUNDS __launch_bounds__(kThreads, MV_VIEW_MIN_CTAS)
#endif
template <bool FAST> __global__ void MV_VIEW_BOUNDS viewKernel(const __grid_constant__ ViewParams P) {
    unsigned char *smem = g_viewSmem;
    const SmemLayout L = smemLayout(P.triCap);
    MvInstance *stage = reinterpret_cast<MvInstance *>(smem + L.stage);
    TriCover *cover = reinterpret_cast<TriCover *>(smem + L.cover);
    TriShade *shade = reinterpret_cast<TriShade *>(smem + L.shade);
    float *xf = reinterpret_cast<float *>(smem + L.xf);          // [kXfWords][kInstChunk]
    int32_t *off = reinterpret_cast<int32_t *>(smem + L.off);    // exclusive item offsets of the chunk's instances, off[n] = total
    float *meshV = reinterpret_cast<float *>(smem + L.meshV);    // [kMeshVerts][6]
    uint8_t *meshI = smem + L.meshI;
    uint16_t *slowAll = reinterpret_cast<uint16_t *>(smem + L.slow);  // [2][kThreads]: instance-in-chunk | item << 7 | done << 15
    ClipVert *clipScratch = reinterpret_cast<ClipVert *>(smem + L.clip + (threadIdx.x >> 5) * 1024u);
    static_assert(4 * kClipVerts * sizeof(ClipVert) <= 1024, "a warp's clip polygons fit its 1 KB of the bin region");
    ViewMisc &M = *reinterpret_cast<ViewMisc *>(smem + L.misc);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // once per CTA: mesh tables, barriers
    for (int i = tid; i < kMeshVerts * 6; i += kThreads) {
        const int v = i / 6, c = i - v * 6;
        float val;
        if (v < kVCapsule) val = c_boxVerts[v][c];
        else if (v < kVSphere) val = c_capsuleVerts[v - kVCapsule][c];
        else if (v < kVCone) val = c_sphereVerts[v - kVSphere][c];
        else if (v < kVCylinder) val = c_coneVerts[v - kVCone][c];
        else val = c_cylinderVerts[v - kVCylinder][c];
        meshV[i] = val;
    }
    for (int i = tid; i < kMeshIdx; i += kThreads) {
        uint8_t val;
        if (i < kISphere) val = c_capsuleIdx[i];
        else if (i < kICone) val = c_sphereIdx[i - kISphere];
        else if (i < kICylinder) val = c_coneIdx[i - kICone];
        else val = c_cylinderIdx[i - kICylinder];
        meshI[i] = val;
    }
    if (tid == 0) { mbarInit(&M.bar[0], 1); mbarInit(&M.bar[1], 1); }
    __syncthreads();
    uint32_t phase[2] = {0u, 0u};

    const int bands = P.bands;
    const uint32_t total = uint32_t(P.N) * uint32_t(bands);
    const int tilesX = P.W >> 5;
    unsigned long long *spill = P.spill + size_t(blockIdx.x) * size_t(P.spillStride);

    if (tid == 0) { M.claim = claimWork(P, total); M.prefetched = 0; }
    for (;;) {
        const long long tc0 = P.stats ? clock64() : 0;
        long long tcWait = 0, tcInst = 0, tcItem = 0;
        __syncthreads();
        const uint32_t claim = M.claim;
        const bool prefetched = M.prefetched != 0;
        if (claim >= total) break;
        const int vrel = int(claim / uint32_t(bands)), band = int(claim - uint32_t(vrel) * uint32_t(bands));
        const int view = P.viewBase + vrel;
        const int env = view / P.A;
        const int rowLo = band * P.bandRows, rowHi = min(P.H, rowLo + P.bandRows) - 1;
        const int bandTiles = tilesX * ((rowHi - rowLo + 1) >> 2);
        const MvInstance *inst = P.instances + size_t(env) * size_t(P.instStride);

        // Launched with programmatic stream serialisation this grid starts while the step kernel is still running: a CTA waits for
        // its env's completion stamp (release/acquire through L2) instead of for the whole step grid.  What the step kernel
        // produced is then read with L2-coherent loads (ld.global.cg) or by the TMA unit (which reads L2), never through L1.
        if (tid == 0) {
            if (P.ready && !prefetched) {
                const uint32_t *flag = P.ready + env;
                uint32_t v;
                while (true) {
                    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
                    if (v == P.readyStamp) break;
                    __nanosleep(200);
                }
                asm volatile("fence.proxy.async;" ::: "memory");  // the acquire orders generic-proxy reads; the bulk copies below go through the async proxy
            }
            M.itemStart = (unsigned long long)clock64();
            M.nTris = 0;
            M.nValid = 0x7fffffff;
            M.nSlow[0] = 0; M.nSlow[1] = 0;
            for (int q = 0; q < 10; ++q) M.stat[q] = 0;
        }
        __syncthreads();
        if (!prefetched) {
            if (tid < 16) M.view[tid] = __ldcg(P.views + size_t(view) * 16 + tid);
            else if (tid < 24) M.counts[tid - 16] = __ldcg(P.instCounts + env * 8 + (tid - 16));
            __syncthreads();
        }
        const int nInst = M.counts[1];
        const int nChunks = (nInst + kInstChunk - 1) / kInstChunk;
        if (tid == 0 && nChunks > 0 && !prefetched) {
            const uint32_t bytes = uint32_t(min(nInst, kInstChunk)) * uint32_t(sizeof(MvInstance));
            mbarExpectTx(&M.bar[0], bytes);
            bulkG2S(stage, inst, bytes, &M.bar[0]);
        }
        M4 viewM;
#pragma unroll
        for (int i = 0; i < 16; ++i) viewM.c[i] = M.view[i];

        SetupCtx cx;
        cx.cover = cover; cx.shade = shade; cx.nTris = &M.nTris; cx.nValid = &M.nValid; cx.triCap = P.triCap; cx.W = P.W; cx.H = P.H; cx.rowLo = rowLo; cx.rowHi = rowHi;
        int batch = 0, parity = 0;
        const long long tc1 = P.stats ? clock64() : 0;

        for (int c = 0; c < nChunks; ++c) {
            const int buf = c & 1;
            const int cBase = c * kInstChunk, cCnt = min(kInstChunk, nInst - cBase);
            const long long tw0 = P.stats ? clock64() : 0;
            mbarWait(&M.bar[buf], phase[buf]);
            phase[buf] ^= 1u;
            const long long tw1 = P.stats ? clock64() : 0;
            tcWait += tw1 - tw0;
            if (tid == 0 && c + 1 < nChunks) {  // the other buffer was last read before the barrier that closed chunk c-1's instance pass
                const int nCnt = min(kInstChunk, nInst - (cBase + kInstChunk));
                const uint32_t bytes = uint32_t(nCnt) * uint32_t(sizeof(MvInstance));
                mbarExpectTx(&M.bar[buf ^ 1], bytes);
                bulkG2S(stage + (buf ^ 1) * kInstChunk, inst + cBase + kInstChunk, bytes, &M.bar[buf ^ 1]);
            }
            // ---- instance pass: one thread per instance of the chunk
            int items = 0;
            if (tid < cCnt) {
                const float4 *src = reinterpret_cast<const float4 *>(stage + buf * kInstChunk + tid);
                const float4 c0 = src[0], c1 = src[1], c2 = src[2], c3 = src[3], c4 = src[4];
                M4 model;
                model.c[0] = c0.x; model.c[1] = c0.y; model.c[2] = c0.z; model.c[3] = c0.w;
                model.c[4] = c1.x; model.c[5] = c1.y; model.c[6] = c1.z; model.c[7] = c1.w;
                model.c[8] = c2.x; model.c[9] = c2.y; model.c[10] = c2.z; model.c[11] = c2.w;
                model.c[12] = c3.x; model.c[13] = c3.y; model.c[14] = c3.z; model.c[15] = c3.w;
                const int mesh = __float_as_int(c4.x), color = __float_as_int(c4.y);
                const M4 mv = mul4(viewM, model);
                int meta = mesh;
                if (instanceMayBeVisible(mv, mesh == 1 ? 2.0f : 1.0f, P.p00, P.p11)) {
                    float nm[9];
                    const float det = normalMatrix(mv, nm);
                    if (!(det > 0.0f)) meta |= 1 << 16;  // a mirroring transform turns the winding round: no object-space face test for its triangles
                    if (mesh == 0) {
                        // a box face whose plane clearly faces away from the eye (the view-space origin) only yields triangles the
                        // winding test drops: outward normal n, face centre = origin + n (unit cube), cull when n_view . c_view > 0
                        int mask = 0;
#pragma unroll
                        for (int face = 0; face < 6; ++face) {
                            const float *fn = meshV + (face * 4) * 6 + 3;
                            const float cxv = mv.c[12] + (fn[0] * mv.c[0] + fn[1] * mv.c[4] + fn[2] * mv.c[8]);
                            const float cyv = mv.c[13] + (fn[0] * mv.c[1] + fn[1] * mv.c[5] + fn[2] * mv.c[9]);
                            const float czv = mv.c[14] + (fn[0] * mv.c[2] + fn[1] * mv.c[6] + fn[2] * mv.c[10]);
                            const float nxv = nm[0] * fn[0] + nm[3] * fn[1] + nm[6] * fn[2];
                            const float nyv = nm[1] * fn[0] + nm[4] * fn[1] + nm[7] * fn[2];
                            const float nzv = nm[2] * fn[0] + nm[5] * fn[1] + nm[8] * fn[2];
                            const float d = nxv * cxv + nyv * cyv + nzv * czv;
                            if (!(d > 1e-3f * sqrtf((nxv * nxv + nyv * nyv + nzv * nzv) * (cxv * cxv + cyv * cyv + czv * czv)))) mask |= 1 << face;
                        }
                        items = __popc(mask);
                        meta |= mask << 8;
                    } else {
                        items = mesh == 1 ? MV_CAPSULE_TRIS : (mesh == 2 ? MV_SPHERE_TRIS : (mesh == 3 ? MV_CONE_TRIS : MV_CYLINDER_TRIS));
                    }
                    if (items) {
#pragma unroll
                        for (int col = 0; col < 4; ++col)
#pragma unroll
                            for (int row = 0; row < 3; ++row) xf[(col * 3 + row) * kInstChunk + tid] = mv.c[col * 4 + row];
#pragma unroll
                        for (int q = 0; q < 9; ++q) xf[(12 + q) * kInstChunk + tid] = nm[q];
                        xf[21 * kInstChunk + tid] = __int_as_float(color);
                    }
                }
                xf[22 * kInstChunk + tid] = __int_as_float(meta);
                if (P.stats && items) atomicAdd(&M.stat[2], 1u);
            }
            // exclusive scan of the item counts over the chunk
            {
                int incl = items;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int up = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += up;
                }
                if (lane == 31) M.wsum[warp] = incl;
                __syncthreads();
                int prefix = 0, totalItems = 0;
#pragma unroll
                for (int w = 0; w < kWarps; ++w) { const int s = M.wsum[w]; if (w < warp) prefix += s; totalItems += s; }
                if (tid < kInstChunk) off[tid] = prefix + incl - items;
                if (tid == 0) off[kInstChunk] = totalItems;
                __syncthreads();
            }
            const int totalItems = off[kInstChunk];
            const long long tw2 = P.stats ? clock64() : 0;
            tcInst += tw2 - tw1;
            if (P.stats && tid == 0) { M.stat[1] += uint32_t(cCnt); M.stat[3] += uint32_t(totalItems); }
            // ---- item pass: one thread per visible box face / mesh triangle.  Items that do not fit the list wait for the next batch;
            // items crossing the near / far plane go to a short list that the warps then clip co-operatively (see slowItem)
            for (int ibase = 0; ibase < totalItems; ibase += kThreads, parity ^= 1) {
                const int j = ibase + tid;
                uint16_t *slowList = slowAll + parity * kThreads;
                if (tid == 0) { M.nSlow[parity ^ 1] = 0; if (P.stats) M.stat[7] += 1; }  // the other list: last read before the barrier that closed the previous sub-pass
                bool pending = j < totalItems, pushed = false, again = false;
                for (;;) {
                    if (pending) {
                        int lo = 0, hi = cCnt - 1;  // largest i with off[i] <= j (instances without items share their successor's offset)
                        while (lo < hi) {
                            const int mid = (lo + hi + 1) >> 1;
                            if (off[mid] <= j) lo = mid; else hi = mid - 1;
                        }
                        const int i = lo, sub = j - off[i];
                        float mv[12], nm[9];
#pragma unroll
                        for (int q = 0; q < 12; ++q) mv[q] = xf[q * kInstChunk + i];
#pragma unroll
                        for (int q = 0; q < 9; ++q) nm[q] = xf[(12 + q) * kInstChunk + i];
                        const int color = __float_as_int(xf[21 * kInstChunk + i]);
                        const int meta = __float_as_int(xf[22 * kInstChunk + i]);
                        const int mesh = meta & 255;
                        const uint32_t ii = uint32_t(cBase + i);
                        ClipVert cvt[4];
                        const float *vpn[4];
                        int nTri;
                        uint32_t keyBase;
                        bool facesAway = false;
                        if (mesh == 0) {
                            const int face = nthFace(unsigned(meta >> 8) & 63u, sub);
#pragma unroll
                            for (int k = 0; k < 4; ++k) vpn[k] = meshV + (face * 4 + k) * 6;
                            nTri = 2; keyBase = ii * 128u + uint32_t(face) * 2u + 1u;
                        } else {
                            const int vBase = mesh == 1 ? kVCapsule : (mesh == 2 ? kVSphere : (mesh == 3 ? kVCone : kVCylinder));
                            const int iBase = mesh == 1 ? kICapsule : (mesh == 2 ? kISphere : (mesh == 3 ? kICone : kICylinder));
#pragma unroll
                            for (int k = 0; k < 3; ++k) vpn[k] = meshV + (vBase + int(meshI[iBase + sub * 3 + k])) * 6;
                            vpn[3] = vpn[2];
                            nTri = 1; keyBase = ii * 128u + uint32_t(sub) + 1u;
#ifndef MV_NO_MESH_PRECULL
                            // Half of a closed mesh faces away.  Those triangles would be dropped by the winding test after three vertex
                            // transforms, three divisions and the 64-bit area; the same decision is available in object space for a
                            // fraction: the eye there is -inverse(M3) t = -(normal matrix)^T t, and the triangle faces away when its plane
                            // has the eye behind it.  Only CLEAR cases are skipped (sine of the angle to the plane beyond 0.02); the
                            // rest take the exact path.
                            if (!(meta & (1 << 16))) {
                                const float t0 = mv[9], t1 = mv[10], t2 = mv[11];
                                const float ex = -(nm[0] * t0 + nm[1] * t1 + nm[2] * t2), ey = -(nm[3] * t0 + nm[4] * t1 + nm[5] * t2), ez = -(nm[6] * t0 + nm[7] * t1 + nm[8] * t2);
                                const float *pa = vpn[0], *pb = vpn[1], *pc = vpn[2];
                                const float ux = pb[0] - pa[0], uy = pb[1] - pa[1], uz = pb[2] - pa[2], vx = pc[0] - pa[0], vy = pc[1] - pa[1], vz = pc[2] - pa[2];
                                const float nx = uy * vz - uz * vy, ny = uz * vx - ux * vz, nz = ux * vy - uy * vx;
                                const float dx = ex - pa[0], dy = ey - pa[1], dz = ez - pa[2];
                                const float sd = nx * dx + ny * dy + nz * dz;
                                facesAway = sd < 0.0f && sd * sd > 4e-4f * ((nx * nx + ny * ny + nz * nz) * (dx * dx + dy * dy + dz * dz));
                            }
#endif
                        }
                        SetupResult res = kSetupDone;
                        if (!facesAway) {
#pragma unroll
                            for (int k = 0; k < 4; ++k) vertPosition(cvt[k], mv, vpn[k], P.p00, P.p11, P.p22, P.p32);
                            res = setupItem<FAST>(cx, cvt[0], cvt[1], cvt[2], cvt[3], nTri, nm, vpn[0], vpn[1], vpn[2], vpn[3], color, keyBase);
                        }
                        pending = res == kSetupFull;
                        if (res == kSetupClip) {
                            int at;
                            asm volatile("atom.shared.add.s32 %0, [%1], 1;" : "=r"(at) : "r"(smemAddrOf(&M.nSlow[parity])) : "memory");
                            slowList[at] = uint16_t(i | (sub << 7));
                            pushed = true;
                        }
                    }
                    const bool any = __syncthreads_or((pending || pushed) ? 1 : 0) || again;
                    pushed = false;
                    if (!any) break;
                    // ---- clipped items, one warp each
                    bool slowFull = false;
                    const int nSlow = M.nSlow[parity];
                    if (P.stats && tid == 0 && !again) M.stat[4] += uint32_t(nSlow);
                    for (int sidx = warp; sidx < nSlow; sidx += kWarps) {
                        const int e = slowList[sidx];
                        if (e & 0x8000) continue;  // done in an earlier round
                        const int i = e & 127, sub = (e >> 7) & 127;
                        float mv[12], nm[9];
#pragma unroll
                        for (int q = 0; q < 12; ++q) mv[q] = xf[q * kInstChunk + i];
#pragma unroll
                        for (int q = 0; q < 9; ++q) nm[q] = xf[(12 + q) * kInstChunk + i];
                        const int color = __float_as_int(xf[21 * kInstChunk + i]);
                        const int meta = __float_as_int(xf[22 * kInstChunk + i]);
                        const int mesh = meta & 255;
                        const uint32_t ii = uint32_t(cBase + i);
                        ClipVert *poly0 = clipScratch, *poly1 = clipScratch + kClipVerts, *tmp0 = clipScratch + 2 * kClipVerts, *tmp1 = clipScratch + 3 * kClipVerts;
                        int nSrc;
                        uint32_t keyBase;
                        if (mesh == 0) {  // lanes 0..3: the face's vertices; source triangles (0,1,2) and (0,2,3)
                            const int face = nthFace(unsigned(meta >> 8) & 63u, sub);
                            nSrc = 2; keyBase = ii * 128u + uint32_t(face) * 2u + 1u;
                            if (lane < 4) {
                                const ClipVert v = makeVert(mv, nm, meshV + (face * 4 + lane) * 6, P.p00, P.p11, P.p22, P.p32);
                                if (lane == 0) { poly0[0] = v; poly1[0] = v; }
                                else if (lane == 1) poly0[1] = v;
                                else if (lane == 2) { poly0[2] = v; poly1[1] = v; }
                                else poly1[2] = v;
                            }
                        } else {
                            const int vBase = mesh == 1 ? kVCapsule : (mesh == 2 ? kVSphere : (mesh == 3 ? kVCone : kVCylinder));
                            const int iBase = mesh == 1 ? kICapsule : (mesh == 2 ? kISphere : (mesh == 3 ? kICone : kICylinder));
                            nSrc = 1; keyBase = ii * 128u + uint32_t(sub) + 1u;
                            if (lane < 3) poly0[lane] = makeVert(mv, nm, meshV + (vBase + int(meshI[iBase + sub * 3 + lane])) * 6, P.p00, P.p11, P.p22, P.p32);
                        }
                        __syncwarp();
                        int nv = 0;  // sixteen lanes per source triangle
                        if ((lane >> 4) < nSrc)
                            nv = clipNearFar(reinterpret_cast<float *>(lane >> 4 ? poly1 : poly0), reinterpret_cast<float *>(lane >> 4 ? tmp1 : tmp0), lane & 15,
                                             0xffffu << (lane & 16));
                        __syncwarp();
                        const int n0 = __shfl_sync(0xffffffffu, nv, 0), n1 = __shfl_sync(0xffffffffu, nv, 16);
                        // fan pieces (0, k, k+1), at most three per source triangle: one lane each; the pieces of one source triangle share
                        // its key (coplanar and disjoint, they never tie on a pixel)
                        const int t = lane / 3, k = lane - t * 3 + 1;
                        const ClipVert *pp = t ? poly1 : poly0;
                        bool vis = false;
                        TriBox tb;
                        ScreenVert sa, sb, sc;
                        if (lane < 6 && k + 1 < (t ? n1 : n0)) {
                            const float hw = float(P.W) * 0.5f, hh = float(P.H) * 0.5f;
                            sa = projectVert(pp[0], hw, hh); sb = projectVert(pp[k], hw, hh); sc = projectVert(pp[k + 1], hw, hh);
                            vis = triBox(cx, sa, sb, sc, tb);
                        }
                        const unsigned vm = __ballot_sync(0xffffffffu, vis);
                        bool done = true;
                        if (vm) {
                            int base = 0;
                            if (lane == 0) base = reserveTris(cx, __popc(vm));
                            base = __shfl_sync(0xffffffffu, base, 0);
                            if (base < 0) done = false;
                            else if (vis) writeTri<FAST>(cx, base + __popc(vm & ((1u << lane) - 1u)), pp[0], pp[k], pp[k + 1], sa, sb, sc, tb, color, keyBase + uint32_t(t));
                        }
                        if (done) { if (lane == 0) slowList[sidx] = uint16_t(e | 0x8000); }
                        else slowFull = true;
                        __syncwarp();  // the scratch polygons are rewritten by the warp's next entry
                    }
                    if (!__syncthreads_or((pending || slowFull) ? 1 : 0)) break;
                    // the list is full: draw what it holds, then retry what did not fit
                    tilePass<FAST>(P, min(M.nTris, M.nValid), spill, view, rowLo, bandTiles, batch, false);
                    if (P.stats && tid == 0) M.stat[5] += uint32_t(min(M.nTris, M.nValid));
                    ++batch;
                    again = true;
                    __syncthreads();
                    if (tid == 0) { M.nTris = 0; M.nValid = 0x7fffffff; }
                    __syncthreads();
                }
            }
            __syncthreads();  // the transform table and the stage buffer are rewritten by the next chunk
            if (P.stats) tcItem += clock64() - tw2;
        }
        if (P.consumed && tid == 0) {  // this item no longer needs the env's instance list or view matrix
            __threadfence();
            atomicAdd(P.consumed + env, 1u);
        }
        const long long tc2 = P.stats ? clock64() : 0;
        tilePass<FAST>(P, min(M.nTris, M.nValid), spill, view, rowLo, bandTiles, batch, true);
        __syncthreads();
        if (P.sliceDone && tid == 0) { __threadfence(); atomicAdd(P.sliceDone + env / P.envsPerSlice, 1u); }
        if (P.viewCost && tid == 0) P.viewCost[claim] = uint32_t(min((unsigned long long)clock64() - M.itemStart, 0xffffffffull * 16ull) >> 4);
        if (P.stats && tid < 10) {
            unsigned long long v = M.stat[tid];
            if (tid == 0) v = 1;
            if (tid == 5) v += (unsigned long long)min(M.nTris, M.nValid);
            if (tid == 6) v = (unsigned long long)(batch + 1);
            atomicAdd(P.stats + (tid < 8 ? tid : tid + 6), v);
            if (tid == 0) {
                const long long tc3 = clock64();
                atomicAdd(P.stats + 8, (unsigned long long)(tc1 - tc0)); atomicAdd(P.stats + 9, (unsigned long long)tcWait);
                atomicAdd(P.stats + 10, (unsigned long long)tcInst); atomicAdd(P.stats + 11, (unsigned long long)tcItem);
                atomicAdd(P.stats + 12, (unsigned long long)(tc3 - tc2)); atomicAdd(P.stats + 13, (unsigned long long)(tc3 - tc0));
            }
        }
    }
    // cost-ordered queue: the last CTA to leave knows every view's cost and sorts the views for the next launch, most expensive first -- a
    // counting sort over 256 linear cost classes (order within a class is arbitrary: it cannot change a frame).  The next launch on the
    // stream cannot start before this grid has drained, so `order` is never read while it is rewritten.
    if (P.viewCost) {
        if (tid == 0) {
            __threadfence();
            M.lastCta = atomicAdd(P.exitCounter, 1u) == gridDim.x - 1u ? 1 : 0;
        }
        __syncthreads();
        if (M.lastCta) {
            __threadfence();
            uint32_t *bins = reinterpret_cast<uint32_t *>(smem + L.sched);
            // per-env cost = sum over its views, gathered once into shared memory (the triangle list is free now); independent loads, four in flight
            const int E = P.N / P.A;
            uint32_t *costS = reinterpret_cast<uint32_t *>(smem + L.cover);
            const int capS = int((L.xf - L.cover) / 4u);
            const bool inSmem = E <= capS;
            if (inSmem) {
                for (int e = tid; e < E; e += kThreads) costS[e] = 0u;
                __syncthreads();
                const uint32_t perEnv = uint32_t(P.A) * uint32_t(P.bands);
                const int items = int(total);
                for (int v0 = tid; v0 < items; v0 += 4 * kThreads) {
                    uint32_t c[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) { const int v = v0 + q * kThreads; c[q] = v < items ? __ldcg(P.viewCost + v) : 0u; }
#pragma unroll
                    for (int q = 0; q < 4; ++q) { const int v = v0 + q * kThreads; if (v < items) atomicAdd(&costS[uint32_t(v) / perEnv], c[q]); }
                }
                __syncthreads();
            }
            auto envCost = [&](int e) {
                if (inSmem) return costS[e];
                uint32_t c = 0u;
                const int perEnv = P.A * P.bands;
                for (int a = 0; a < perEnv; ++a) c += __ldcg(P.viewCost + e * perEnv + a);
                return c;
            };
            uint32_t mx = 1u;
            for (int e = tid; e < E; e += kThreads) mx = max(mx, envCost(e));
#pragma unroll
            for (int d = 16; d; d >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, d));
            if (lane == 0) M.wsum[warp] = int32_t(mx);
            // sort key: (slice of the progressive host delivery, if any) major, cost class descending minor
            int nSlices = P.sliceDone ? (E + P.envsPerSlice - 1) / P.envsPerSlice : 1;
            if (!inSmem || E + nSlices * 256 > capS) nSlices = 1;  // no room for the classes of every slice: plain cost order
            const int envsPerSlice = nSlices > 1 ? P.envsPerSlice : E;
            const int nBins = nSlices * 256;
            uint32_t *kbins = nSlices > 1 ? costS + E : bins;
            for (int b = tid; b < nBins; b += kThreads) kbins[b] = 0u;
            __syncthreads();
#pragma unroll
            for (int w = 0; w < kWarps; ++w) mx = max(mx, uint32_t(M.wsum[w]));
            const float scale = 255.0f / float(mx);
            auto keyOf = [&](int e) { return (e / envsPerSlice) * 256 + 255 - min(255, int(float(envCost(e)) * scale)); };
            for (int e = tid; e < E; e += kThreads) atomicAdd(&kbins[keyOf(e)], 1u);
            __syncthreads();
            {   // exclusive scan of the class counts: a run of consecutive classes per thread, then a scan over the threads
                const int per = (nBins + kThreads - 1) / kThreads, b0 = min(nBins, tid * per), b1 = min(nBins, b0 + per);
                uint32_t sum = 0u;
                for (int b = b0; b < b1; ++b) sum += kbins[b];
                uint32_t incl = sum;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const uint32_t up = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += up; }
                __syncthreads();  // (M.wsum still holds the maxima some warp may be reading)
                if (lane == 31) M.wsum[warp] = int32_t(incl);
                __syncthreads();
                uint32_t run = incl - sum;
#pragma unroll
                for (int w = 0; w < kWarps; ++w) if (w < warp) run += uint32_t(M.wsum[w]);
                for (int b = b0; b < b1; ++b) { const uint32_t c = kbins[b]; kbins[b] = run; run += c; }
            }
            __syncthreads();
            for (int e = tid; e < E; e += kThreads) {
                const uint32_t at = atomicAdd(&kbins[keyOf(e)], 1u);
                P.order[at] = uint32_t(e);
            }
            if (tid == 0) *P.exitCounter = 0u;
        }
    }
}

}  // namespace mvr
