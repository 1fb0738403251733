// simplify.cu -- quadric edge-collapse mesh simplification (K10)
//
// Replaces the simplifier inside zmesh.Mesher.get(id, reduction_factor,
// max_error) (igneous/tasks/mesh/mesh.py:376-381) for ALL labels of a task at
// once.  zmesh's simplifier is a sequential heap-ordered collapse per label; a
// GPU needs a data-parallel formulation, so this is a round-based variant:
//
//   init    per-vertex Garland-Heckbert plane quadrics (unit normals, summed in
//           face order), boundary vertices locked (chunk borders must stitch),
//           per-vertex incident-face arrays (half-edge nodes, fixed capacity,
//           merged and compacted on collapse).
//   round   E  every edge of a label still above its face target computes the cheap
//              quadric cost (min over {u, v, midpoint} of p^T (Qu+Qv) p) and, if
//              cost <= max_error^2, posts a (cost, per-round hash of the label-local
//              half-edge id) key to both endpoints (atomic min); labels with at most
//              65536 half-edges use a 32-bit key (16 cost bits | 16-bit id permutation);
//           K2 per vertex: is its key the minimum over its face neighbours' keys?
//           C  an edge WINS iff its key is the minimum of both endpoints' keys and of
//              all their neighbours' -> winners are two edges apart, never touch each
//              other's faces or vertices and are processed concurrently: a winner
//              collapses iff the link condition holds and no incident face flips,
//              otherwise it is parked until one of its endpoints' rings changes.
//   stop    per label: faces <= target, or a round without winners, or four
//           consecutive rounds that each remove < 0.2% of the label's faces.
//   compact scans renumber surviving vertices / faces per label.
//
// Labels are independent, so all rounds of one label run inside ONE CTA with the
// label's topology in shared memory (k_simp_labels below: one launch per MeshTask, one
// CTA per label).
//
// All arithmetic is double precision WITHOUT fused multiply-add (this file is
// compiled with -fmad=false) so that oracle/igneous_oracle.c::orc_simplify
// reproduces it bit for bit.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <stdlib.h>

#include <algorithm>
#include <type_traits>

#include "mesher.h"

namespace ign {

constexpr uint64_t S_KEYMAX = 0xFFFFFFFFFFFFFFFFull;
constexpr int S_MAXV = 32;
constexpr int S_VCAP = 64;  // two rings of < S_MAXV alive faces always fit after a collapse
constexpr int VB = 11;  // vertex key coordinate bits (mesh.cu V_COORD_BITS)

struct Simp {
  uint64_t U, T;
  double* pos;      // 3U
  double* Q;        // 10U
  uint32_t* face;   // 3T global vertex ids
  uint32_t* flabel; // T dense labels
  uint8_t* falive;
  uint8_t* valive;
  uint8_t* vbound;
  // incident half-edge nodes (3f+c) of every vertex as a fixed-capacity array: ring
  // enumeration is a set of independent loads instead of a linked-list pointer chase
  uint32_t* vf;   // [U * S_VCAP]
  uint32_t* vn;   // [U] entries in use (dead faces are skipped, compacted when the vertex is kept)
  const uint32_t* tri_off;  // [K+2] first face of each label
};

__device__ __forceinline__ uint32_t s_mix(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
__device__ __forceinline__ uint32_t s_unmix(uint32_t x) {
  x ^= x >> 16; x *= 0x43021123U; x ^= x >> 15 ^ x >> 30; x *= 0x1d69e2a5U; x ^= x >> 16;
  return x;
}
// 16-bit variant for labels whose half-edge ids fit 16 bits (oracle: simp_mix16 / simp_unmix16)
__device__ __forceinline__ uint32_t s_mix16(uint32_t x) {
  x &= 0xFFFFu;
  x = (x * 0x2F35u) & 0xFFFFu; x ^= x >> 7;
  x = (x * 0x4A6Bu) & 0xFFFFu; x ^= x >> 9;
  x = (x * 0x9E37u) & 0xFFFFu; x ^= x >> 8;
  return x;
}
__device__ __forceinline__ uint32_t s_unmix16(uint32_t x) {
  x &= 0xFFFFu;
  x ^= x >> 8; x = (x * 0x7787u) & 0xFFFFu;
  x ^= x >> 9; x = (x * 0x1243u) & 0xFFFFu;
  x ^= x >> 7; x ^= x >> 14; x = (x * 0xEB1Du) & 0xFFFFu;
  return x;
}
__device__ __forceinline__ unsigned long long s_key(double cost, uint32_t h, uint32_t salt) {
  const float c = __double2float_rn(cost);
  return ((unsigned long long)__float_as_uint(c) << 32) | s_mix(h ^ salt);
}

__device__ __forceinline__ double s_qeval(const double* q, const double* p) {
  const double x = p[0], y = p[1], z = p[2];
  return q[0] * x * x + 2.0 * q[1] * x * y + 2.0 * q[2] * x * z + 2.0 * q[3] * x + q[4] * y * y +
         2.0 * q[5] * y * z + 2.0 * q[6] * y + q[7] * z * z + 2.0 * q[8] * z + q[9];
}

__device__ int s_twins(const Simp& s, uint32_t f, uint32_t u, uint32_t v, uint32_t* twin) {
  int cnt = 0;
  const uint32_t* lu = s.vf + (uint64_t)u * S_VCAP;
  const uint32_t cu = s.vn[u];
  for (uint32_t j = 0; j < cu; j++) {
    const uint32_t h = lu[j];
    const uint32_t g = h / 3;
    if (g == f || !s.falive[g]) continue;
    const uint32_t* fv = s.face + 3 * (uint64_t)g;
    if (fv[0] == v || fv[1] == v || fv[2] == v) {
      if (cnt == 0) *twin = h;
      cnt++;
    }
  }
  return cnt;
}

struct SEval {
  bool valid;
  double cost;
  uint32_t keep, remove;
  double p[3];
};

// ------------------------------------------------------------------ kernels
__global__ void __launch_bounds__(256)
    k_simp_init_verts(const uint64_t* __restrict__ vkeys, uint64_t U, double rx, double ry, double rz,
                      double* __restrict__ pos, uint8_t* __restrict__ valive,
                      uint8_t* __restrict__ vbound, uint32_t* __restrict__ vn) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= U) return;
  const uint64_t k = vkeys[i];
  const double x = (double)(k & ((1u << VB) - 1));
  const double y = (double)((k >> VB) & ((1u << VB) - 1));
  const double z = (double)((k >> (2 * VB)) & ((1u << VB) - 1));
  pos[3 * i + 0] = x * 0.5 * rx;
  pos[3 * i + 1] = y * 0.5 * ry;
  pos[3 * i + 2] = z * 0.5 * rz;
  valive[i] = 1;
  vbound[i] = 0;
  vn[i] = 0;
}

// faces: local ids + per-label vertex base -> global ids; flabel by offsets search
__global__ void __launch_bounds__(256)
    k_simp_init_faces(const uint32_t* __restrict__ faces_local, const uint32_t* __restrict__ tri_off,
                      const uint32_t* __restrict__ vert_off, uint32_t K, uint64_t T,
                      uint32_t* __restrict__ face, uint32_t* __restrict__ flabel,
                      uint8_t* __restrict__ falive, uint32_t* __restrict__ node_vertex,
                      uint32_t* __restrict__ node_id) {
  const uint64_t f = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (f >= T) return;
  // largest l in [1,K] with tri_off[l] <= f
  uint32_t lo = 1, hi = K;
  while (lo < hi) {
    const uint32_t mid = (lo + hi + 1) >> 1;
    if (tri_off[mid] <= f) lo = mid;
    else hi = mid - 1;
  }
  flabel[f] = lo;
  falive[f] = 1;
  for (int k = 0; k < 3; k++) {
    const uint32_t g = faces_local[3 * f + k] + vert_off[lo];
    face[3 * f + k] = g;
    node_vertex[3 * f + k] = g;
    node_id[3 * f + k] = (uint32_t)(3 * f + k);
  }
}

// sorted (vertex, node) pairs -> per-vertex arrays in ascending node order
__global__ void __launch_bounds__(256)
    k_simp_link(const uint32_t* __restrict__ sv, const uint32_t* __restrict__ sh, uint64_t n,
                uint32_t* __restrict__ vf, uint32_t* __restrict__ vn, uint32_t* overflow) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t v = sv[i];
  if (i > 0 && sv[i - 1] == v) return;  // the first pair of a run writes the whole run
  uint32_t c = 0;
  for (uint64_t j = i; j < n && sv[j] == v; j++) {
    if (c < S_VCAP) vf[(uint64_t)v * S_VCAP + c] = sh[j];
    c++;
  }
  if (c > S_VCAP) {
    *overflow = 1;
    c = S_VCAP;
  }
  vn[v] = c;
}

__global__ void __launch_bounds__(128) k_simp_quadrics(Simp s) {
  const uint64_t v = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (v >= s.U) return;
  double q[10];
  for (int i = 0; i < 10; i++) q[i] = 0.0;
  for (uint32_t j = 0; j < s.vn[v]; j++) {
    const uint32_t h = s.vf[(uint64_t)v * S_VCAP + j];
    const uint32_t* fv = s.face + 3 * (uint64_t)(h / 3);
    const double* a = s.pos + 3 * (uint64_t)fv[0];
    const double* b = s.pos + 3 * (uint64_t)fv[1];
    const double* c = s.pos + 3 * (uint64_t)fv[2];
    const double ux = b[0] - a[0], uy = b[1] - a[1], uz = b[2] - a[2];
    const double vx = c[0] - a[0], vy = c[1] - a[1], vz = c[2] - a[2];
    double nx = uy * vz - uz * vy, ny = uz * vx - ux * vz, nz = ux * vy - uy * vx;
    const double len = sqrt(nx * nx + ny * ny + nz * nz);
    if (!(len > 0.0)) continue;
    nx = nx / len; ny = ny / len; nz = nz / len;
    const double d = -(nx * a[0] + ny * a[1] + nz * a[2]);
    q[0] += nx * nx; q[1] += nx * ny; q[2] += nx * nz; q[3] += nx * d;
    q[4] += ny * ny; q[5] += ny * nz; q[6] += ny * d;
    q[7] += nz * nz; q[8] += nz * d; q[9] += d * d;
  }
  for (int i = 0; i < 10; i++) s.Q[10 * v + i] = q[i];
}

__global__ void __launch_bounds__(256) k_simp_boundary(Simp s) {
  const uint64_t h = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (h >= 3 * s.T) return;
  const uint32_t f = (uint32_t)(h / 3), c = (uint32_t)(h % 3);
  const uint32_t u = s.face[3 * (uint64_t)f + c], v = s.face[3 * (uint64_t)f + (c + 1) % 3];
  uint32_t tw;
  if (s_twins(s, f, u, v, &tw) != 1) {
    s.vbound[u] = 1;
    s.vbound[v] = 1;
  }
}

// ------------------------------------------------------------------ per-label rounds
// One CTA owns one label for ALL of its rounds (labels are independent: keys use
// label-local half-edge ids and the stop rules are per label).  The topology of the
// label -- faces as label-local vertex ids (u16 SoA), one state byte per face (alive bit
// + a 2-bit memo per half-edge), a flag byte and a "lose" byte per vertex, the 32-bit round
// keys and the ring lists of the round's winners -- lives in SHARED MEMORY for the whole
// run; only the double-precision data that a round touches sparsely (positions, quadrics,
// cached float costs) stays in global memory (L2).  A round is a handful of
// __syncthreads() phases instead of five launches and a host round trip:
//
//   P1  key1[v] = MAX, lose[v] = 0                             (vertex parallel)
//   P2  every canonical half-edge (u < v) of an alive face posts its key to both
//       endpoints with a shared-memory min reduction; the float cost is memoised until
//       an endpoint moves (CDIRTY); dropped memos are re-evaluated by per-warp queues on
//       dense lanes while other warps keep posting                (face parallel)
//   P3  a vertex LOSEs if a face neighbour holds a smaller key1 (== key2 test of the
//       round formulation: key2[w] == key1[w] <=> !LOSE[w]); plain byte stores
//                                                               (face parallel)
//   P4  a vertex a WINs iff its key's half-edge starts at a, both endpoints hold that
//       key and neither LOSEs; at most SL_WCAP winners per pass  (vertex parallel)
//   E1  the faces that touch a winner's endpoints append themselves to the winner's
//       two ring lists; the first warps compute the winners' placement and cost (E2a)
//       at the same time                                         (face parallel)
//   E2b one flip test per (winner, side, ring face)              (item parallel)
//   E2c link condition by ballots / shuffles over the ring lists and the collapse
//       itself, one HALF warp per winner (whole warps for rings over 16 faces)
//
// Labels that do not fit (more than 16384 faces, or 6U + 9T + 28 KB over the CTA's shared
// memory) keep faces and lists in global memory, with keys / flags / states still in
// shared memory when those fit ("hybrid"), else everything global (SM = false, 64-bit
// key slots).
// vertex flags: CDIRTY the vertex moved (cached costs of its edges are stale), RDIRTY its ring
// changed (parked edges around it may be valid now)
constexpr uint32_t VF_ALIVE = 1, VF_BOUND = 2, VF_CDIRTY = 4, VF_DONE = 16, VF_END = 32, VF_RDIRTY = 64;
constexpr int SL_THREADS = 1024;
constexpr int SL_WCAP = 128;  // winners validated per selection pass (a round runs as many passes as it needs)
constexpr uint32_t WF_BAD = 1, WF_OK = 2;  // winner flags: failed validation / validated
constexpr int SL_EQ = 96;      // per-warp queue of faces with half-edges whose cost must be (re)computed
constexpr int SL_LIST_PER = 16;  // list entries per thread held in registers while a list is compacted in place

struct SlArgs {
  double* pos;            // 3U
  double* Q;              // 10U
  uint32_t* face;         // 3T global vertex ids
  uint8_t* falive;        // T   (out)
  uint8_t* valive;        // U   (out)
  const uint8_t* vbound;  // U
  float* ecost;           // 3T  memoised float cost per half-edge
  // global-memory class only (labels that do not fit shared memory)
  unsigned long long* key1;  // U
  uint8_t* fstate;           // T
  uint8_t* vflag;            // U
  uint8_t* vlose;            // U  LOSE marks of the round (plain byte stores)
  uint32_t *flist, *flist2;  // T  alive-face lists (ping-pong)
  uint32_t *vlist, *vlist2;  // U
  const uint32_t* tri_off;   // [K+2]
  const uint32_t* vert_off;  // [K+2]
  const uint32_t* target;    // [K+2]
  const uint32_t* order;     // [K] dense labels, largest first
  uint32_t K;
  uint32_t* counters;  // [0] next work item  [1] max rounds  [2] labels run in shared memory  [3] in global memory
  double max_err2;
  int max_rounds;
  uint32_t smem_bytes;  // dynamic shared memory of the launch
  int persist;          // 1: a CTA keeps taking labels until the list is empty (IGN_SIMP_PERSIST=1)
  uint32_t* lrec;       // IGN_SIMP_TRACE=1: [work item][4] = faces, rounds, kilocycles, face visits (sum of list lengths)
  uint32_t* trace;      // IGN_SIMP_TRACE=1: [round][4] = winners, collapses, alive faces, list length of the largest label
};

struct SlWin {
  uint32_t u, v, h, cnt[2], keep, flags, pad;
};

struct SlShared {
  uint32_t work, alive, progress, ncol, nwin, stop, slow, counter, nbig;
  unsigned long long visits, wins;  // IGN_SIMP_TRACE
  long long t_label;
  unsigned long long ph[10];  // phase timers (IGN_SIMP_TRACE)
  long long t_prev;
  SlWin win[SL_WCAP];
  double wbest[SL_WCAP * 3];  // placement of the round's winners
};

template <bool SM>
struct SlLab {
  typedef typename std::conditional<SM, uint16_t, uint32_t>::type idx_t;
  uint32_t T, U, tbase, vbase, target;
  idx_t *fc0, *fc1, *fc2;  // SM: label-local ids, SoA in shared memory
  uint32_t* gface;         // !SM: AoS global ids in place
  uint8_t* fstate;         // bit 7 alive, bits 2c..2c+1 memo of half-edge c
  uint8_t* vflag;
  uint8_t* vlose;  // a face neighbour holds a smaller key this round (written with plain byte stores: every writer stores 1)
  // key format (oracle: simp_key): labels with 3T <= 65536 use 32-bit keys (bf16-like cost | 16-bit id
  // permutation).  The shared-memory class only takes such labels and stores them in 32 bits (native
  // shared-memory min); the other classes keep 64-bit slots for both formats.
  typedef typename std::conditional<SM, uint32_t, unsigned long long>::type key_t;
  key_t* key1;
  bool fmt16;
  uint32_t* wq;    // [warps][SL_EQ] per-warp cost queues of the key pass (shared memory)
  idx_t* ring;     // [SL_WCAP][2][S_MAXV] face ids of the winners' rings (shared memory)
  idx_t *flist, *flist2, *vlist, *vlist2;  // alive lists (flist2 / vlist2: global-memory class only)
};

template <bool SM>
__device__ __forceinline__ uint32_t sl_fget(const SlLab<SM>& L, uint32_t f, int c) {
  if (SM) return c == 0 ? L.fc0[f] : (c == 1 ? L.fc1[f] : L.fc2[f]);
  return L.gface[3 * (uint64_t)f + c] - L.vbase;
}
template <bool SM>
__device__ __forceinline__ void sl_fset(const SlLab<SM>& L, uint32_t f, int c, uint32_t x) {
  typedef typename SlLab<SM>::idx_t idx_t;
  if (SM) {
    if (c == 0) L.fc0[f] = (idx_t)x;
    else if (c == 1) L.fc1[f] = (idx_t)x;
    else L.fc2[f] = (idx_t)x;
  } else {
    L.gface[3 * (uint64_t)f + c] = x + L.vbase;
  }
}
// flag bytes are modified with word atomics whenever two threads may touch the same word
// (SM: the flags are in shared memory for sure -> shared-space reductions instead of generic atomics)
template <bool SM>
__device__ __forceinline__ void sl_vor(uint8_t* vflag, uint32_t v, uint32_t bits) {
  const uintptr_t a = (uintptr_t)(vflag + v);
  if ((*(volatile uint8_t*)a & bits) == bits) return;
  const uint32_t word = bits << (8 * (a & 3));
  if (SM) {
    asm volatile("red.shared.or.b32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared((void*)(a & ~(uintptr_t)3))), "r"(word) : "memory");
  } else {
    atomicOr((uint32_t*)(a & ~(uintptr_t)3), word);
  }
}
template <bool SM>
__device__ __forceinline__ void sl_vclear(uint8_t* vflag, uint32_t v, uint32_t bits) {
  const uintptr_t a = (uintptr_t)(vflag + v);
  const uint32_t word = ~(bits << (8 * (a & 3)));
  if (SM) {
    asm volatile("red.shared.and.b32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared((void*)(a & ~(uintptr_t)3))), "r"(word) : "memory");
  } else {
    atomicAnd((uint32_t*)(a & ~(uintptr_t)3), word);
  }
}
__device__ __forceinline__ void sl_post(unsigned long long* key1, uint32_t u, uint32_t v, unsigned long long key) {
  if (key < *(volatile unsigned long long*)&key1[u]) atomicMin(&key1[u], key);
  if (key < *(volatile unsigned long long*)&key1[v]) atomicMin(&key1[v], key);
}
__device__ __forceinline__ void sl_post(uint32_t* key1, uint32_t u, uint32_t v, uint32_t key) {  // shared memory only
  if (key < *(volatile uint32_t*)&key1[u])
    asm volatile("red.shared.min.u32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(key1 + u)), "r"(key) : "memory");
  if (key < *(volatile uint32_t*)&key1[v])
    asm volatile("red.shared.min.u32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(key1 + v)), "r"(key) : "memory");
}
template <bool SM>
__device__ __forceinline__ typename SlLab<SM>::key_t sl_key(const SlLab<SM>& L, float cost, uint32_t hl, uint32_t salt) {
  typedef typename SlLab<SM>::key_t key_t;
  const uint32_t bits = __float_as_uint(cost);
  if (SM || L.fmt16) return (key_t)((((bits >> 15) & 0xFFFFu) << 16) | s_mix16((hl ^ salt) & 0xFFFFu));
  return (key_t)(((unsigned long long)bits << 32) | s_mix(hl ^ salt));
}
template <bool SM>
__device__ __forceinline__ uint32_t sl_key_edge(const SlLab<SM>& L, typename SlLab<SM>::key_t key, uint32_t salt) {
  if (SM || L.fmt16) return s_unmix16((uint32_t)key & 0xFFFFu) ^ (salt & 0xFFFFu);
  return s_unmix((uint32_t)((unsigned long long)key & 0xFFFFFFFFull)) ^ salt;
}

// s_cost on label-local ids (same arithmetic, same order)
template <bool SM>
__device__ __forceinline__ void sl_cost(const SlArgs& A, const SlLab<SM>& L, uint32_t u, uint32_t v, SEval* e) {
  e->valid = false;
  const bool bu = L.vflag[u] & VF_BOUND, bv = L.vflag[v] & VF_BOUND;
  if (bu && bv) return;
  const double* Qu = A.Q + 10 * (uint64_t)(L.vbase + u);
  const double* Qv = A.Q + 10 * (uint64_t)(L.vbase + v);
  double q[10];
#pragma unroll
  for (int i = 0; i < 10; i++) q[i] = Qu[i] + Qv[i];
  const double* pu = A.pos + 3 * (uint64_t)(L.vbase + u);
  const double* pv = A.pos + 3 * (uint64_t)(L.vbase + v);
  double best[3], cost;
  if (bu) {
    e->keep = u;
    e->remove = v;
    best[0] = pu[0]; best[1] = pu[1]; best[2] = pu[2];
    cost = s_qeval(q, best);
  } else if (bv) {
    e->keep = v;
    e->remove = u;
    best[0] = pv[0]; best[1] = pv[1]; best[2] = pv[2];
    cost = s_qeval(q, best);
  } else {
    e->keep = u < v ? u : v;
    e->remove = u < v ? v : u;
    const double* pk = u < v ? pu : pv;
    const double* pr = u < v ? pv : pu;
    const double kk[3] = {pk[0], pk[1], pk[2]}, rr[3] = {pr[0], pr[1], pr[2]};
    const double mid[3] = {(kk[0] + rr[0]) * 0.5, (kk[1] + rr[1]) * 0.5, (kk[2] + rr[2]) * 0.5};
    const double ck = s_qeval(q, kk), cr = s_qeval(q, rr), cm = s_qeval(q, mid);
    cost = ck;
    best[0] = kk[0]; best[1] = kk[1]; best[2] = kk[2];
    if (cr < cost) { cost = cr; best[0] = rr[0]; best[1] = rr[1]; best[2] = rr[2]; }
    if (cm < cost) { cost = cm; best[0] = mid[0]; best[1] = mid[1]; best[2] = mid[2]; }
  }
  if (cost < 0.0) cost = 0.0;
  if (!(cost <= A.max_err2)) return;
  e->valid = true;
  e->cost = cost;
  e->p[0] = best[0]; e->p[1] = best[1]; e->p[2] = best[2];
}

// does face (a0,a1,a2) flip when vertex w moves to `best`?  (the validation's flip test)
template <bool SM>
__device__ __forceinline__ bool sl_flips(const SlArgs& A, const SlLab<SM>& L, const uint32_t* a, uint32_t w,
                                         const double* best) {
  double P[3][3], N[3][3];
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const double* p = A.pos + 3 * (uint64_t)(L.vbase + a[k]);
    P[k][0] = p[0]; P[k][1] = p[1]; P[k][2] = p[2];
  }
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const bool mv = (a[k] == w);
    N[k][0] = mv ? best[0] : P[k][0];
    N[k][1] = mv ? best[1] : P[k][1];
    N[k][2] = mv ? best[2] : P[k][2];
  }
  const double ax = P[1][0] - P[0][0], ay = P[1][1] - P[0][1], az = P[1][2] - P[0][2];
  const double bx = P[2][0] - P[0][0], by = P[2][1] - P[0][1], bz = P[2][2] - P[0][2];
  const double n0x = ay * bz - az * by, n0y = az * bx - ax * bz, n0z = ax * by - ay * bx;
  const double cx = N[1][0] - N[0][0], cy = N[1][1] - N[0][1], cz = N[1][2] - N[0][2];
  const double dx = N[2][0] - N[0][0], dy = N[2][1] - N[0][1], dz = N[2][2] - N[0][2];
  const double n1x = cy * dz - cz * dy, n1y = cz * dx - cx * dz, n1z = cx * dy - cy * dx;
  const double dot = n0x * n1x + n0y * n1y + n0z * n1z;
  return !(dot > 0.0);
}

// the two corners of a ring face other than w, in cyclic order after w
__device__ __forceinline__ void sl_others(const uint32_t* a, uint32_t w, uint32_t* o1, uint32_t* o2) {
  if (a[0] == w) { *o1 = a[1]; *o2 = a[2]; }
  else if (a[1] == w) { *o1 = a[2]; *o2 = a[0]; }
  else { *o1 = a[0]; *o2 = a[1]; }
}

// distinct values among the (x1, x2) of the first n lanes; f1 / f2 flag the first occurrences
__device__ __forceinline__ uint32_t sl_distinct(uint32_t x1, uint32_t x2, uint32_t n, uint32_t lane, bool* f1,
                                                bool* f2) {
  const uint32_t FULL = 0xFFFFFFFFu;
  const bool have = lane < n;
  const uint32_t m1 = __match_any_sync(FULL, x1);
  const uint32_t m2 = __match_any_sync(FULL, x2);
  *f1 = have && ((int)lane == __ffs(m1) - 1);
  bool in1 = false;
  for (uint32_t j = 0; j < n; j++) in1 |= (__shfl_sync(FULL, x1, j) == x2);
  *f2 = have && ((int)lane == __ffs(m2) - 1) && !in1;
  return __popc(__ballot_sync(FULL, *f1)) + __popc(__ballot_sync(FULL, *f2));
}

// drop the dead entries of an alive list (order is irrelevant).  SM: in place, the entries
// pass through registers; global-memory class: into the second buffer, then swap.
template <bool SM, typename IDX, typename PRED>
__device__ __forceinline__ uint32_t sl_compact(IDX*& list, IDX*& list2, uint32_t n, uint32_t* counter, PRED alive) {
  const uint32_t FULL = 0xFFFFFFFFu;
  const uint32_t tid = threadIdx.x, lane = tid & 31u;
  if (tid == 0) *counter = 0;
  __syncthreads();
  if (SM) {
    IDX keep[SL_LIST_PER];
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < SL_LIST_PER; k++) {
      const uint32_t i = tid + k * blockDim.x;
      keep[k] = 0;
      if (i < n) {
        const IDX e = list[i];
        keep[k] = e;
        if (alive((uint32_t)e)) m |= 1u << k;
      }
    }
    __syncthreads();
    const uint32_t cnt = __popc(m);
    uint32_t inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t o = __shfl_up_sync(FULL, inc, d);
      if ((int)lane >= d) inc += o;
    }
    uint32_t base = 0;
    if (lane == 31 && inc) base = atomicAdd(counter, inc);
    base = __shfl_sync(FULL, base, 31) + inc - cnt;
#pragma unroll
    for (int k = 0; k < SL_LIST_PER; k++)
      if ((m >> k) & 1u) list[base++] = keep[k];
  } else {
    for (uint32_t i0 = (tid & ~31u); i0 < n; i0 += blockDim.x) {
      const uint32_t i = i0 + lane;
      IDX e = 0;
      bool al = false;
      if (i < n) {
        e = list[i];
        al = alive((uint32_t)e);
      }
      const uint32_t bal = __ballot_sync(FULL, al);
      if (!bal) continue;
      uint32_t base = 0;
      const int leader = __ffs(bal) - 1;
      if ((int)lane == leader) base = atomicAdd(counter, (uint32_t)__popc(bal));
      base = __shfl_sync(FULL, base, leader);
      if (al) list2[base + __popc(bal & ((1u << lane) - 1u))] = e;
    }
    IDX* t = list;
    list = list2;
    list2 = t;
  }
  __syncthreads();
  const uint32_t kept = *counter;
  __syncthreads();  // everyone has read the count: the counter may be reused by the next call
  return kept;
}

// phase timers (IGN_SIMP_TRACE=1): thread 0 attributes the cycles since the previous mark to a phase
#define SL_MARK(id)                                   \
  do {                                                \
    if (A.trace != nullptr && tid == 0) {             \
      const long long _t = clock64();                 \
      sh.ph[id] += (unsigned long long)(_t - sh.t_prev); \
      sh.t_prev = _t;                                 \
    }                                                 \
  } while (0)

// One pass of E2c with groups of W lanes (16: two winners per warp side by side, only winners whose
// rings fit 16 lanes; 32: the winners left over).  Both halves of a warp run the same instructions;
// everything that differs between them is predicated and loop counts are made warp uniform.
template <bool SM, int W>
__device__ __forceinline__ void sl_collapse_pass(const SlArgs& A, const SlLab<SM>& L, SlShared& sh, uint32_t nb) {
  const uint32_t FULL = 0xFFFFFFFFu;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5, NW = blockDim.x >> 5;
  constexpr uint32_t G = 32 / W;                       // groups per warp
  const uint32_t gl = lane & (W - 1), goff = lane & ~(uint32_t)(W - 1);
  const uint32_t wmask = W == 32 ? FULL : 0xFFFFu;
  const uint32_t gmask = wmask << goff;
  const uint32_t gidx = lane / W;
  for (uint32_t base = warp * G; base < nb; base += NW * G) {  // warp uniform
    const uint32_t slot = base + gidx;
    bool act = slot < nb;
    uint32_t nfu = 0, nfv = 0;
    if (act) { nfu = sh.win[slot].cnt[0]; nfv = sh.win[slot].cnt[1]; }
    const bool big = nfu > 16u || nfv > 16u;
    if (W == 16) {
      if (act && big && gl == 0) atomicAdd(&sh.nbig, 1u);
      act = act && !big;
    } else {
      act = act && big;
    }
    uint32_t fu = 0, fv = 0, u = 0, v = 0, hl = 0, k = 0;
    bool ok = false;
    if (act) {
      if (gl < nfu && gl < (uint32_t)S_MAXV) fu = L.ring[(2 * slot) * S_MAXV + gl];
      if (gl < nfv && gl < (uint32_t)S_MAXV) fv = L.ring[(2 * slot + 1) * S_MAXV + gl];
      u = sh.win[slot].u; v = sh.win[slot].v; hl = sh.win[slot].h; k = sh.win[slot].keep;
      ok = !(sh.win[slot].flags & WF_BAD) && nfu <= (uint32_t)S_MAXV && nfv <= (uint32_t)S_MAXV;
    }
    const uint32_t rm = (k == u) ? v : u;
    // the quadrics of the two endpoints are needed only if the collapse happens, but the L2 round
    // trip is as long as the whole link test: request them now
    double* Qk = A.Q + 10 * (uint64_t)(L.vbase + k);
    const double* Qr = A.Q + 10 * (uint64_t)(L.vbase + rm);
    double qk = 0.0, qr = 0.0;
    if (ok && gl < 10) { qk = Qk[gl]; qr = Qr[gl]; }
    const bool hu = ok && gl < nfu, hv = ok && gl < nfv;
    uint32_t au[3] = {0, 0, 0}, av[3] = {0, 0, 0};
    uint32_t x1 = 0xF0000000u + lane, x2 = 0xF1000000u + lane, y1 = 0xF2000000u + lane, y2 = 0xF3000000u + lane;
    if (hu) {
      au[0] = sl_fget<SM>(L, fu, 0); au[1] = sl_fget<SM>(L, fu, 1); au[2] = sl_fget<SM>(L, fu, 2);
      sl_others(au, u, &x1, &x2);
    }
    if (hv) {
      av[0] = sl_fget<SM>(L, fv, 0); av[1] = sl_fget<SM>(L, fv, 1); av[2] = sl_fget<SM>(L, fv, 2);
      sl_others(av, v, &y1, &y2);
    }
    // (every lane of the warp takes part in the collectives below; n = 0 for groups without a winner)
    const uint32_t nu = ok ? nfu : 0u, nv = ok ? nfv : 0u;
    uint32_t nmax = nu > nv ? nu : nv;
    if (W == 16) {
      const uint32_t o = __shfl_xor_sync(FULL, nmax, 16);
      nmax = o > nmax ? o : nmax;
    }
    // distinct neighbours of u (first occurrences f1 among x1, f2 among x2 not in x1), same for v
    const uint32_t mu1 = __match_any_sync(FULL, x1) & gmask, mu2 = __match_any_sync(FULL, x2) & gmask;
    const uint32_t mv1 = __match_any_sync(FULL, y1) & gmask, mv2 = __match_any_sync(FULL, y2) & gmask;
    bool inu = false, inv = false, c1 = false, c2 = false;
    for (uint32_t j = 0; j < nmax; j++) {
      const uint32_t sx1 = __shfl_sync(FULL, x1, j, W), sy1 = __shfl_sync(FULL, y1, j, W), sy2 = __shfl_sync(FULL, y2, j, W);
      if (j < nu) inu |= (sx1 == x2);
      if (j < nv) {
        inv |= (sy1 == y2);
        c1 |= (x1 == sy1) | (x1 == sy2);
        c2 |= (x2 == sy1) | (x2 == sy2);
      }
    }
    const bool f1 = hu && ((int)lane == __ffs(mu1) - 1);
    const bool f2 = hu && ((int)lane == __ffs(mu2) - 1) && !inu;
    const bool g1 = hv && ((int)lane == __ffs(mv1) - 1);
    const bool g2 = hv && ((int)lane == __ffs(mv2) - 1) && !inv;
    const uint32_t b_f1 = __ballot_sync(FULL, f1), b_f2 = __ballot_sync(FULL, f2);
    const uint32_t b_g1 = __ballot_sync(FULL, g1), b_g2 = __ballot_sync(FULL, g2);
    const uint32_t b_c1 = __ballot_sync(FULL, f1 && c1), b_c2 = __ballot_sync(FULL, f2 && c2);
    const uint32_t b_sh = __ballot_sync(FULL, hu && (x1 == v || x2 == v));
    const uint32_t nnu = __popc(b_f1 & gmask) + __popc(b_f2 & gmask), nnv = __popc(b_g1 & gmask) + __popc(b_g2 & gmask);
    const uint32_t common = __popc(b_c1 & gmask) + __popc(b_c2 & gmask), shared = __popc(b_sh & gmask);
    const bool go = ok && nnu <= (uint32_t)S_MAXV && nnv <= (uint32_t)S_MAXV && shared == 2 && common == 2;
    if (act && !go && gl == 0) {  // park the edge until one of its endpoints' rings changes
      const uint32_t f = hl / 3, c = hl - 3 * f;
      const uint32_t st = L.fstate[f];  // (winners of one pass never share a face: byte accesses are disjoint)
      L.fstate[f] = (uint8_t)((st & ~(3u << (2 * c))) | (1u << (2 * c)));
      sl_vclear<SM>(L.vflag, u, VF_END);
      sl_vclear<SM>(L.vflag, v, VF_END);
      atomicOr(&sh.progress, 1u);
    }
    const bool rm_is_u = (rm == u);
    const bool hr = go && (rm_is_u ? hu : hv);
    const uint32_t rf = rm_is_u ? fu : fv;
    const uint32_t r0 = rm_is_u ? au[0] : av[0], r1 = rm_is_u ? au[1] : av[1], r2 = rm_is_u ? au[2] : av[2];
    // faces of rm: those that also hold k die, the others get k in rm's corner
    const bool dies = hr && (r0 == k || r1 == k || r2 == k);
    if (hr) {
      if (dies) L.fstate[rf] = (uint8_t)(L.fstate[rf] & 0x7Fu);
      else sl_fset<SM>(L, rf, r0 == rm ? 0 : (r1 == rm ? 1 : 2), k);
    }
    const uint32_t dead = __popc(__ballot_sync(FULL, dies) & gmask);
    if (go) {
      // the new ring of k: parked edges around it may be valid now
      if (hu && x1 != v && x2 != v) { sl_vor<SM>(L.vflag, x1, VF_RDIRTY); sl_vor<SM>(L.vflag, x2, VF_RDIRTY); }
      if (hv && y1 != u && y2 != u) { sl_vor<SM>(L.vflag, y1, VF_RDIRTY); sl_vor<SM>(L.vflag, y2, VF_RDIRTY); }
      if (gl < 10) Qk[gl] = qk + qr;
      if (gl >= 10 && gl < 13) A.pos[3 * (uint64_t)(L.vbase + k) + (gl - 10)] = sh.wbest[3 * slot + (gl - 10)];
      if (gl == 0) {
        sl_vor<SM>(L.vflag, k, VF_CDIRTY | VF_RDIRTY);  // k moved: cached costs of its edges are stale
        sl_vclear<SM>(L.vflag, k, VF_END);
        sl_vclear<SM>(L.vflag, rm, 0xFFu);
        atomicSub(&sh.alive, dead);
        atomicAdd(&sh.ncol, 1u);
        atomicOr(&sh.progress, 1u);
      }
    }
  }
}

template <bool SM>
__device__ void sl_run(const SlArgs& A, const SlLab<SM>& L, SlShared& sh) {
  if (A.trace != nullptr && threadIdx.x == 0) {
    for (int q = 0; q < 10; q++) sh.ph[q] = 0;
    sh.t_prev = clock64();
    sh.t_label = sh.t_prev;
    sh.visits = 0;
    sh.wins = 0;
  }
  typedef typename SlLab<SM>::idx_t idx_t;
  typedef typename SlLab<SM>::key_t key_t;
  const uint32_t FULL = 0xFFFFFFFFu;
  const uint32_t tid = threadIdx.x, NT = blockDim.x, lane = tid & 31u, warp = tid >> 5, NW = NT >> 5;
  const uint32_t T = L.T, U = L.U;
  idx_t *flist = L.flist, *flist2 = L.flist2, *vlist = L.vlist, *vlist2 = L.vlist2;
  // ---- load the label
  for (uint32_t f = tid; f < T; f += NT) {
    if (SM) {
      const uint32_t* g = A.face + 3 * (uint64_t)(L.tbase + f);
      sl_fset<SM>(L, f, 0, g[0] - L.vbase);
      sl_fset<SM>(L, f, 1, g[1] - L.vbase);
      sl_fset<SM>(L, f, 2, g[2] - L.vbase);
    }
    L.fstate[f] = 0x80;
    flist[f] = (idx_t)f;
  }
  for (uint32_t v = tid; v < U; v += NT) {
    L.vflag[v] = (uint8_t)(VF_ALIVE | (A.vbound[L.vbase + v] ? VF_BOUND : 0u));
    if (!SM) vlist[v] = (idx_t)v;  // the shared-memory class scans its vertices directly (no list: 2 B / vertex saved)
  }
  if (tid == 0) {
    sh.alive = T;
    sh.slow = 0;
    sh.stop = 0;
  }
  __syncthreads();
  uint32_t nF = T, nV = U;

  int r = 0;
  for (; r < A.max_rounds; r++) {
    if (sh.alive <= L.target) break;  // reached the target before this round
    // per-round salt: equal-cost edges get a fresh pseudo-random priority every round (a fixed
    // one lets the same validation failures win again and again: 8738 instead of 454 faces on the
    // reference's box volume)
    const uint32_t salt = (uint32_t)r * 0x9E3779B9u;
    // ---- P1
    for (uint32_t i = tid; i < nV; i += NT) {
      const uint32_t v = SM ? i : (uint32_t)vlist[i];
      L.key1[v] = (key_t)S_KEYMAX;
      L.vlose[v] = 0;
      const uint8_t b = L.vflag[v];
      if (b & VF_DONE) L.vflag[v] = (uint8_t)(b & ~VF_DONE);
    }
    if (tid == 0) {
      sh.progress = 0;
      sh.ncol = 0;
    }
    __syncthreads();
    SL_MARK(0);
    // ---- P2: keys of the canonical half-edges.  A warp takes 32 alive faces per iteration and
    // posts the cached keys; faces with half-edges whose memoised state was dropped collect in
    // a per-warp queue that is evaluated (double precision cost) on dense lanes.
    {
      uint32_t* wq = L.wq + warp * SL_EQ;
      uint32_t qn = 0;  // faces in the warp's queue (warp uniform)
      // software pipeline: the face id and the three cached costs of the NEXT iteration are
      // requested (global loads, L2 latency) before the current face is processed
      const float* ecb = A.ecost + 3 * (uint64_t)L.tbase;
      uint32_t f_n = 0;
      float ec_n[3] = {0.f, 0.f, 0.f};
      if (warp * 32 + lane < nF) {
        f_n = flist[warp * 32 + lane];
        ec_n[0] = ecb[3 * (uint64_t)f_n]; ec_n[1] = ecb[3 * (uint64_t)f_n + 1]; ec_n[2] = ecb[3 * (uint64_t)f_n + 2];
      }
      for (uint32_t base = warp * 32; base < nF; base += NT) {
        const uint32_t i = base + lane;
        const uint32_t f = f_n;
        const float ec[3] = {ec_n[0], ec_n[1], ec_n[2]};
        if (i + NT < nF) {
          f_n = flist[i + NT];
          ec_n[0] = ecb[3 * (uint64_t)f_n]; ec_n[1] = ecb[3 * (uint64_t)f_n + 1]; ec_n[2] = ecb[3 * (uint64_t)f_n + 2];
        }
        uint32_t st = 0, a[3] = {0, 0, 0}, fl[3] = {0, 0, 0};
        if (i < nF) st = L.fstate[f];
        bool act = (st & 0x80u) != 0;
        if (act) {
          a[0] = sl_fget<SM>(L, f, 0); a[1] = sl_fget<SM>(L, f, 1); a[2] = sl_fget<SM>(L, f, 2);
          fl[0] = L.vflag[a[0]]; fl[1] = L.vflag[a[1]]; fl[2] = L.vflag[a[2]];
        }
        uint32_t pend = 0, nst = st;
        if (act) {
#pragma unroll
          for (int c = 0; c < 3; c++) {
            const uint32_t u = a[c], v = a[(c + 1) % 3];
            const uint32_t fe = fl[c] | fl[(c + 1) % 3];
            if (!(u < v)) continue;  // one key per edge
            // memo: 0 unknown, 1 parked (won a round, failed validation), 2 cost cached in
            // ecost, 3 known to exceed max_error.  2 / 3 are dropped when an endpoint moved
            // (CDIRTY), 1 when an endpoint's ring changed (RDIRTY).
            uint32_t es = (st >> (2 * c)) & 3u;
            if (es >= 2 && (fe & VF_CDIRTY)) es = 0;
            else if (es == 1 && (fe & VF_RDIRTY)) es = 0;
            if (es == 0) {
              pend |= 1u << c;
            } else if (es == 2) {
              sl_post(L.key1, u, v, sl_key<SM>(L, ec[c], 3u * f + (uint32_t)c, salt));
            }
            nst = (nst & ~(3u << (2 * c))) | (es << (2 * c));
          }
        }
        if (act && nst != st) L.fstate[f] = (uint8_t)nst;  // pending corners hold memo 0 until they are evaluated
        // faces with pending corners accumulate in the warp's queue over the iterations; the
        // queue is evaluated when the next iteration might not fit (>= 3 dense passes) and at the end
        const uint32_t has = pend ? 1u : 0u;
        const uint32_t bal = __ballot_sync(FULL, has);
        if (has) wq[qn + __popc(bal & ((1u << lane) - 1u))] = (f << 3) | pend;
        qn += __popc(bal);
        const bool last = base + NT >= nF;
        if (qn > (uint32_t)SL_EQ - 32 || (last && qn)) {
          __syncwarp();
          for (uint32_t j = lane; j < qn; j += 32) {
            const uint32_t e = wq[j], ef = e >> 3, ep = e & 7u;
            uint32_t est = L.fstate[ef];
#pragma unroll
            for (int c = 0; c < 3; c++) {
              if (!((ep >> c) & 1u)) continue;
              const uint32_t u = sl_fget<SM>(L, ef, c), v = sl_fget<SM>(L, ef, (c + 1) % 3);
              SEval ev;
              sl_cost<SM>(A, L, u, v, &ev);
              uint32_t es = 3;  // exceeds max_error
              if (ev.valid) {
                const float cf = __double2float_rn(ev.cost);
                A.ecost[3 * (uint64_t)(L.tbase + ef) + c] = cf;
                es = 2;
                sl_post(L.key1, u, v, sl_key<SM>(L, cf, 3u * ef + (uint32_t)c, salt));
              }
              est = (est & ~(3u << (2 * c))) | (es << (2 * c));
            }
            L.fstate[ef] = (uint8_t)est;  // the queue holds a face once: single writer
          }
          __syncwarp();
          qn = 0;
        }
      }
    }
    __syncthreads();
    SL_MARK(1);
    // ---- P3: dirty flags consumed; LOSE = a face neighbour holds a smaller key
    for (uint32_t i = tid; i < nV; i += NT) {
      const uint32_t v = SM ? i : (uint32_t)vlist[i];
      if (L.vflag[v] & (VF_CDIRTY | VF_RDIRTY)) sl_vclear<SM>(L.vflag, v, VF_CDIRTY | VF_RDIRTY);
    }
    // two faces per thread and iteration, the loads of both issued before anything depends on them
    for (uint32_t i = tid; i < nF; i += 2 * NT) {
      const uint32_t i2 = i + NT;
      const bool two = i2 < nF;
      const uint32_t fa = flist[i], fb = two ? (uint32_t)flist[i2] : fa;
      const bool la = (L.fstate[fa] & 0x80u) != 0, lb = two && (L.fstate[fb] & 0x80u) != 0;
      uint32_t a0 = 0, a1 = 0, a2 = 0, b0 = 0, b1 = 0, b2 = 0;
      if (la) { a0 = sl_fget<SM>(L, fa, 0); a1 = sl_fget<SM>(L, fa, 1); a2 = sl_fget<SM>(L, fa, 2); }
      if (lb) { b0 = sl_fget<SM>(L, fb, 0); b1 = sl_fget<SM>(L, fb, 1); b2 = sl_fget<SM>(L, fb, 2); }
      key_t ka0 = 0, ka1 = 0, ka2 = 0, kb0 = 0, kb1 = 0, kb2 = 0;
      if (la) { ka0 = L.key1[a0]; ka1 = L.key1[a1]; ka2 = L.key1[a2]; }
      if (lb) { kb0 = L.key1[b0]; kb1 = L.key1[b1]; kb2 = L.key1[b2]; }
      if (la) {
        key_t m = ka0 < ka1 ? ka0 : ka1;
        m = ka2 < m ? ka2 : m;
        if (ka0 > m) L.vlose[a0] = 1;
        if (ka1 > m) L.vlose[a1] = 1;
        if (ka2 > m) L.vlose[a2] = 1;
      }
      if (lb) {
        key_t m = kb0 < kb1 ? kb0 : kb1;
        m = kb2 < m ? kb2 : m;
        if (kb0 > m) L.vlose[b0] = 1;
        if (kb1 > m) L.vlose[b1] = 1;
        if (kb2 > m) L.vlose[b2] = 1;
      }
    }
    __syncthreads();
    SL_MARK(2);
    // ---- P4 + E: the round's winners (marked DONE on both endpoints), SL_WCAP per pass
    for (;;) {
      if (tid == 0) { sh.nwin = 0; sh.nbig = 0; }
      __syncthreads();
      for (uint32_t i = tid; i < nV; i += NT) {
        const uint32_t a = SM ? i : (uint32_t)vlist[i];
        const uint32_t fl = L.vflag[a];
        if (!(fl & VF_ALIVE) || (fl & VF_DONE) || L.vlose[a]) continue;
        const key_t key = L.key1[a];
        if (key == (key_t)S_KEYMAX) continue;
        const uint32_t hl = sl_key_edge<SM>(L, key, salt);
        const uint32_t f = hl / 3, c = hl - 3 * f;
        if (sl_fget<SM>(L, f, (int)c) != a) continue;
        const uint32_t v = sl_fget<SM>(L, f, (int)((c + 1) % 3));
        if (L.key1[v] != key || (L.vflag[v] & VF_DONE) || L.vlose[v]) continue;
        const uint32_t slot = atomicAdd(&sh.nwin, 1u);
        if (slot < (uint32_t)SL_WCAP) {
          sh.win[slot].u = a;
          sh.win[slot].v = v;
          sh.win[slot].h = hl;
          sh.win[slot].cnt[0] = 0;
          sh.win[slot].cnt[1] = 0;
          sh.win[slot].flags = 0;
          sl_vor<SM>(L.vflag, a, VF_DONE | VF_END);
          sl_vor<SM>(L.vflag, v, VF_DONE | VF_END);
        }
      }
      __syncthreads();
      SL_MARK(3);
      const uint32_t total = sh.nwin;
      const uint32_t nb = total < (uint32_t)SL_WCAP ? total : (uint32_t)SL_WCAP;
      if (nb == 0) break;
      if (A.trace != nullptr && tid == 0) sh.wins += nb;
      // key1 is dead until the next P1: the winners' entries now name their ring lists
      for (uint32_t i = tid; i < nb; i += NT) {
        L.key1[sh.win[i].u] = (key_t)(2u * i);
        L.key1[sh.win[i].v] = (key_t)(2u * i + 1u);
      }
      __syncthreads();
      SL_MARK(4);
      // ---- E1 + E2a in one barrier interval (they do not depend on each other): the first warps
      // compute placement and cost of the winners (one thread each, double precision, L2 latency)
      // while the others build the ring lists with one pass over the alive faces.
      {
        const uint32_t nbt = (nb + 31u) & ~31u;
        const bool split = NT - nbt >= NT / 2;
        if (tid < nb) {
          const uint32_t i = tid;
          SEval e;
          sl_cost<SM>(A, L, sh.win[i].u, sh.win[i].v, &e);
          sh.win[i].keep = e.valid ? e.keep : sh.win[i].u;
          sh.win[i].flags = e.valid ? 0u : WF_BAD;
          if (e.valid) {
            sh.wbest[3 * i + 0] = e.p[0]; sh.wbest[3 * i + 1] = e.p[1]; sh.wbest[3 * i + 2] = e.p[2];
          }
        }
        if (!split || tid >= nbt) {
          const uint32_t first = split ? tid - nbt : tid, step = split ? NT - nbt : NT;
          for (uint32_t i = first; i < nF; i += 2 * step) {
            const uint32_t i2 = i + step;
            const bool two = i2 < nF;
            const uint32_t fa = flist[i], fb = two ? (uint32_t)flist[i2] : fa;
            const bool la = (L.fstate[fa] & 0x80u) != 0, lb = two && (L.fstate[fb] & 0x80u) != 0;
            uint32_t x[6] = {0, 0, 0, 0, 0, 0}, fl[6] = {0, 0, 0, 0, 0, 0};
            if (la) { x[0] = sl_fget<SM>(L, fa, 0); x[1] = sl_fget<SM>(L, fa, 1); x[2] = sl_fget<SM>(L, fa, 2); }
            if (lb) { x[3] = sl_fget<SM>(L, fb, 0); x[4] = sl_fget<SM>(L, fb, 1); x[5] = sl_fget<SM>(L, fb, 2); }
            if (la) { fl[0] = L.vflag[x[0]]; fl[1] = L.vflag[x[1]]; fl[2] = L.vflag[x[2]]; }
            if (lb) { fl[3] = L.vflag[x[3]]; fl[4] = L.vflag[x[4]]; fl[5] = L.vflag[x[5]]; }
#pragma unroll
            for (int c = 0; c < 6; c++) {
              if (!(fl[c] & VF_END)) continue;
              const uint32_t sl = (uint32_t)L.key1[x[c]];
              const uint32_t p = atomicAdd(&sh.win[sl >> 1].cnt[sl & 1u], 1u);
              if (p < (uint32_t)S_MAXV) L.ring[sl * S_MAXV + p] = (idx_t)(c < 3 ? fa : fb);
            }
          }
        }
      }
      __syncthreads();
      SL_MARK(5);
      SL_MARK(6);
      // E2b: one flip test per (winner, side, ring entry)
      for (uint32_t item = tid; item < nb * 64; item += NT) {
        const uint32_t i = item >> 6, side = (item >> 5) & 1u, j = item & 31u;
        if (sh.win[i].flags & WF_BAD) continue;
        if (sh.win[i].cnt[0] > (uint32_t)S_MAXV || sh.win[i].cnt[1] > (uint32_t)S_MAXV) continue;  // fails in E2c
        if (j >= sh.win[i].cnt[side]) continue;
        const uint32_t w = side ? sh.win[i].v : sh.win[i].u, other = side ? sh.win[i].u : sh.win[i].v;
        const uint32_t f = L.ring[(2 * i + side) * S_MAXV + j];
        const uint32_t a[3] = {sl_fget<SM>(L, f, 0), sl_fget<SM>(L, f, 1), sl_fget<SM>(L, f, 2)};
        if (a[0] == other || a[1] == other || a[2] == other) continue;  // dies with the edge
        const double best[3] = {sh.wbest[3 * i], sh.wbest[3 * i + 1], sh.wbest[3 * i + 2]};
        if (sl_flips<SM>(A, L, a, w, best)) atomicOr(&sh.win[i].flags, WF_BAD);
      }
      __syncthreads();
      SL_MARK(7);
      // E2c: link condition by ballots / shuffles over the ring lists (a lane holds one ring face of
      // each endpoint), then the collapse itself.  Winners whose rings have at most 16 faces (almost
      // all) are handled by HALF warps, two winners per warp at a time: the pass is a chain of
      // dependent shared-memory accesses per winner, so its duration is the number of winners a warp
      // handles one after the other.  The few winners with larger rings take a second pass with
      // whole warps.
      sl_collapse_pass<SM, 16>(A, L, sh, nb);
      __syncthreads();
      if (sh.nbig) {
        sl_collapse_pass<SM, 32>(A, L, sh, nb);
      }
      __syncthreads();
      SL_MARK(8);
      if (total <= (uint32_t)SL_WCAP) break;
    }
    // ---- stop rules of the label
    if (tid == 0 && A.trace != nullptr && sh.work == 0 && r < 400) {
      A.trace[4 * r + 0] = sh.progress;
      A.trace[4 * r + 1] = sh.ncol;
      A.trace[4 * r + 2] = sh.alive;
      A.trace[4 * r + 3] = nF;
    }
    if (A.trace != nullptr && tid == 0) sh.visits += nF;
    if (tid == 0) {
      uint32_t stop = 0;
      if (!sh.progress) {
        stop = 1;  // nothing collapsed or parked: fixed point
      } else {
        // four consecutive rounds that each remove fewer than 0.2% of the remaining faces
        if ((uint64_t)sh.ncol * 1000 < (uint64_t)sh.alive) sh.slow++;
        else sh.slow = 0;
        if (sh.slow >= 4) stop = 1;
      }
      sh.stop = stop;
    }
    __syncthreads();
    SL_MARK(9);
    if (sh.stop) {
      r++;
      break;
    }
    // ---- dead entries leave the lists every second round
    if (r & 1) {
      nF = sl_compact<SM>(flist, flist2, nF, &sh.counter, [&](uint32_t f) { return (L.fstate[f] & 0x80u) != 0; });
      if (!SM) nV = sl_compact<SM>(vlist, vlist2, nV, &sh.counter, [&](uint32_t v) { return (L.vflag[v] & VF_ALIVE) != 0; });
    }
  }
  // ---- write the label back to the whole-task arrays
  for (uint32_t f = tid; f < T; f += NT) {
    const bool al = L.fstate[f] & 0x80u;
    A.falive[L.tbase + f] = al ? 1 : 0;
    if (SM && al) {
      uint32_t* g = A.face + 3 * (uint64_t)(L.tbase + f);
      g[0] = sl_fget<SM>(L, f, 0) + L.vbase;
      g[1] = sl_fget<SM>(L, f, 1) + L.vbase;
      g[2] = sl_fget<SM>(L, f, 2) + L.vbase;
    }
  }
  for (uint32_t v = tid; v < U; v += NT) A.valive[L.vbase + v] = (L.vflag[v] & VF_ALIVE) ? 1 : 0;
  if (tid == 0 && A.trace != nullptr) {
    for (int q = 0; q < 10; q++) atomicAdd((unsigned long long*)(A.trace + 1600) + q, sh.ph[q]);
    uint32_t* rec = A.lrec + 6 * (size_t)sh.work;
    rec[0] = T;
    rec[1] = (uint32_t)r;
    rec[2] = (uint32_t)((clock64() - sh.t_label) >> 10);
    rec[3] = (uint32_t)(sh.visits > 0xFFFFFFFFull ? 0xFFFFFFFFull : sh.visits);
    rec[4] = (uint32_t)sh.wins;
    rec[5] = SM ? 1u : ((const void*)L.key1 == (const void*)(A.key1 + L.vbase) ? 3u : 2u);
  }
  if (tid == 0) {
    atomicMax(&A.counters[1], (uint32_t)r);
    atomicAdd(&A.counters[SM ? 2 : 3], 1u);
  }
}

extern __shared__ __align__(16) unsigned char sl_smem[];

// One label per CTA (the launch has one CTA per label; a CTA takes the next label of the size-sorted
// order from a counter, so big labels start first whatever order the hardware dispatches CTAs in).
// CTAs that end after one label keep returning their SM to the block scheduler: kernels of
// other streams -- the CCL passes of the volume pipeline run on a higher-priority stream while
// MeshTasks are in flight -- get SMs within a label's run time instead of a whole task's.
__global__ void __launch_bounds__(SL_THREADS, 1) k_simp_labels(SlArgs A) {
  __shared__ SlShared sh;
  do {
    __syncthreads();  // (persistent mode) the previous label is completely written back; sh.work may be reused
    if (threadIdx.x == 0) sh.work = atomicAdd(&A.counters[0], 1u);
    __syncthreads();
    const uint32_t wi = sh.work;
    if (wi >= A.K) break;
    const uint32_t l = A.order[wi];
    const uint32_t tbase = A.tri_off[l], T = A.tri_off[l + 1] - tbase;
    const uint32_t vbase = A.vert_off[l], U = A.vert_off[l + 1] - vbase;
    const uint32_t target = A.target[l];
    if (T == 0 || T <= target) continue;  // init left every face / vertex alive
    // shared-memory layout: cost queues | ring lists | key1 | faces SoA | face list | face state | vertex flags
    const size_t wq_bytes = (size_t)(SL_THREADS / 32) * SL_EQ * 4;
    const size_t ring_sm = (size_t)SL_WCAP * 2 * S_MAXV * 2, ring_gl = (size_t)SL_WCAP * 2 * S_MAXV * 4;
    const size_t o_key = wq_bytes + ring_sm;   // shared-memory class: 16-bit face ids
    const size_t o_keyg = wq_bytes + ring_gl;  // other classes: 32-bit
    const size_t o_f0 = o_key + 4 * (size_t)U;  // 32-bit keys
    const size_t o_fl = o_f0 + 6 * (size_t)T;
    const size_t o_fs = o_fl + 2 * (size_t)T;
    const size_t o_vf = (o_fs + T + 3) & ~(size_t)3;
    const size_t o_vl = (o_vf + U + 3) & ~(size_t)3;
    const size_t need = o_vl + U + 4;
    const uint32_t cap = (uint32_t)SL_LIST_PER * blockDim.x;
    const bool fmt16 = 3ull * T <= 65536ull;
    if (need <= A.smem_bytes && T <= cap && U <= cap && fmt16) {
      SlLab<true> L;
      L.T = T; L.U = U; L.tbase = tbase; L.vbase = vbase; L.target = target;
      L.wq = (uint32_t*)sl_smem;
      L.ring = (uint16_t*)(sl_smem + wq_bytes);
      L.key1 = (uint32_t*)(sl_smem + o_key);
      L.fmt16 = true;
      L.fc0 = (uint16_t*)(sl_smem + o_f0);
      L.fc1 = L.fc0 + T;
      L.fc2 = L.fc1 + T;
      L.flist = (uint16_t*)(sl_smem + o_fl);
      L.vlist = nullptr;
      L.flist2 = L.vlist2 = nullptr;
      L.gface = nullptr;
      L.fstate = sl_smem + o_fs;
      L.vflag = sl_smem + o_vf;
      L.vlose = sl_smem + o_vl;
      sl_run<true>(A, L, sh);
    } else {
      SlLab<false> L;
      L.T = T; L.U = U; L.tbase = tbase; L.vbase = vbase; L.target = target;
      L.wq = (uint32_t*)sl_smem;  // the cost queues and the ring lists always fit
      L.ring = (uint32_t*)(sl_smem + wq_bytes);
      L.fc0 = L.fc1 = L.fc2 = nullptr;
      L.flist = A.flist + tbase; L.flist2 = A.flist2 + tbase;
      L.vlist = A.vlist + vbase; L.vlist2 = A.vlist2 + vbase;
      L.gface = A.face + 3 * (uint64_t)tbase;
      L.fmt16 = fmt16;
      // the arrays that take the atomics (keys, vertex flags) and the face states stay in shared
      // memory whenever they fit; only the faces and the alive lists are read from global memory
      const size_t h_fs = o_keyg + 8 * (size_t)U;
      const size_t h_vf = (h_fs + T + 3) & ~(size_t)3;
      const size_t h_vl = (h_vf + U + 3) & ~(size_t)3;
      if (h_vl + U + 4 <= A.smem_bytes) {
        L.key1 = (unsigned long long*)(sl_smem + o_keyg);
        L.fstate = sl_smem + h_fs;
        L.vflag = sl_smem + h_vf;
        L.vlose = sl_smem + h_vl;
      } else {
        L.key1 = A.key1 + vbase;
        L.fstate = A.fstate + tbase;
        L.vflag = A.vflag + vbase;
        L.vlose = A.vlose + vbase;
      }
      sl_run<false>(A, L, sh);
    }
  } while (A.persist);
}

__global__ void __launch_bounds__(256)
    k_simp_flags_u32(const uint8_t* __restrict__ a, uint64_t n, uint32_t* __restrict__ out) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i];
}

__global__ void __launch_bounds__(256)
    k_simp_new_offsets(const uint32_t* __restrict__ old_off, const uint32_t* __restrict__ scan,
                       uint32_t K2, uint64_t n, uint32_t total, uint32_t* __restrict__ new_off) {
  const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l < K2) new_off[l] = (old_off[l] < n) ? scan[old_off[l]] : total;
}

__global__ void __launch_bounds__(256)
    k_simp_compact_verts(Simp s, const uint32_t* __restrict__ vscan, float* __restrict__ pos_f) {
  const uint64_t v = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (v >= s.U || !s.valive[v]) return;
  const uint32_t n = vscan[v];
  pos_f[3 * (uint64_t)n + 0] = __double2float_rn(s.pos[3 * v + 0]);
  pos_f[3 * (uint64_t)n + 1] = __double2float_rn(s.pos[3 * v + 1]);
  pos_f[3 * (uint64_t)n + 2] = __double2float_rn(s.pos[3 * v + 2]);
}

__global__ void __launch_bounds__(256)
    k_simp_compact_faces(Simp s, const uint32_t* __restrict__ vscan, const uint32_t* __restrict__ fscan,
                         const uint32_t* __restrict__ new_vert_off, uint32_t* __restrict__ faces_out) {
  const uint64_t f = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (f >= s.T || !s.falive[f]) return;
  const uint32_t n = fscan[f];
  const uint32_t base = new_vert_off[s.flabel[f]];
  for (int k = 0; k < 3; k++) faces_out[3 * (uint64_t)n + k] = vscan[s.face[3 * f + k]] - base;
}

__global__ void __launch_bounds__(256)
    k_simp_export(const float* __restrict__ pos_f, uint64_t first, uint64_t count, float sx, float sy,
                  float sz, float* __restrict__ out) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= count) return;
  out[3 * i + 0] = __fadd_rn(pos_f[3 * (first + i) + 0], sx);
  out[3 * i + 1] = __fadd_rn(pos_f[3 * (first + i) + 1], sy);
  out[3 * i + 2] = __fadd_rn(pos_f[3 * (first + i) + 2], sz);
}

// exposed to mesh.cu for export of simplified positions
int simp_export_positions(ign_ctx* ctx, const float* pos_f, uint64_t first, uint64_t count,
                          const float shift[3], float* d_out) {
  if (count == 0) return IGN_OK;
  IGN_LAUNCH(ctx, k_simp_export, blocks_for(count, 256), 256, 0, pos_f, first, count, shift[0], shift[1],
             shift[2], d_out);
  return IGN_OK;
}

}  // namespace ign

using namespace ign;

extern "C" int ign_mesh_simplify(ign_mesher* m, const float resolution[3], int reduction_factor,
                                 float max_error) {
  IGN_REQUIRE(m && resolution, IGN_ERR_INVALID, "null argument");
  ign_ctx* ctx = m->ctx;
  IGN_TRY(activate(ctx));
  IGN_REQUIRE(!m->simplified, IGN_ERR_INVALID, "mesher is already simplified; call mesh() again");
  IGN_REQUIRE(reduction_factor >= 1, IGN_ERR_INVALID, "reduction_factor must be >= 1");
  m->res[0] = resolution[0];
  m->res[1] = resolution[1];
  m->res[2] = resolution[2];
  m->simp_factor = reduction_factor;
  m->simp_max_error = max_error;
  m->simp_rounds = 0;
  const uint64_t U = m->U, T = m->T, K = m->K;
  if (T == 0 || U == 0) {
    m->simplified = true;
    m->d_pos_f = nullptr;
    return IGN_OK;
  }
  Scratch sc(ctx);
  IGN_REQUIRE(sc.owner(), IGN_ERR_INVALID, "ign_mesh_simplify must own the scratch arena");

  size_t sortb = 0, scanb = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sortb, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                  (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)(3 * T));
  cub::DeviceScan::ExclusiveSum(nullptr, scanb, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                (int)(3 * T));
  const size_t tmpb = (sortb > scanb ? sortb : scanb) + 256;
  const size_t need = align_up(U * 24, 256) + align_up(U * 80, 256) + 3 * align_up(3 * T * 4, 256) +
                      align_up(U * S_VCAP * 4, 256) + align_up(T * 4, 256) + 2 * align_up(T, 256) +
                      4 * align_up(U, 256) + 3 * align_up(U * 4, 256) + align_up(U * 8, 256) +
                      6 * align_up((K + 2) * 4, 256) + align_up(3 * T * 4, 256) +
                      2 * align_up(3 * T * 4, 256) + 2 * align_up(T * 4, 256) + 2 * align_up(U * 4, 256) + tmpb +
                      align_up((size_t)ctx->sm_count * 4 * SL_WCAP * 2 * S_MAXV * 4, 256) +
                      align_up((size_t)ctx->sm_count * 4 * SL_WCAP * 3 * 8, 256) + (1 << 20);
  IGN_TRY(sc.reserve(need));
  Simp s;
  s.U = U;
  s.T = T;
  s.pos = sc.take<double>(U * 3);
  s.Q = sc.take<double>(U * 10);
  s.face = sc.take<uint32_t>(3 * T);
  s.vf = sc.take<uint32_t>(U * S_VCAP);
  uint32_t* node_v = sc.take<uint32_t>(3 * T);   // reused as face scan later
  uint32_t* node_h = sc.take<uint32_t>(3 * T);
  s.flabel = sc.take<uint32_t>(T);
  s.falive = sc.take<uint8_t>(T);
  uint8_t* fstate = sc.take<uint8_t>(T);
  s.valive = sc.take<uint8_t>(U);
  s.vbound = sc.take<uint8_t>(U);
  uint8_t* vflag = sc.take<uint8_t>(U);
  uint8_t* vlose = sc.take<uint8_t>(U);
  s.vn = sc.take<uint32_t>(U);
  uint32_t* vscan = sc.take<uint32_t>(U);
  uint32_t* vflag32 = sc.take<uint32_t>(U);
  unsigned long long* key1 = sc.take<unsigned long long>(U);
  uint32_t* d_target = sc.take<uint32_t>(K + 2);
  uint32_t* d_tri_off = sc.take<uint32_t>(K + 2);
  uint32_t* d_vert_off = sc.take<uint32_t>(K + 2);
  uint32_t* d_new_tri_off = sc.take<uint32_t>(K + 2);
  uint32_t* d_new_vert_off = sc.take<uint32_t>(K + 2);
  uint32_t* d_order = sc.take<uint32_t>(K + 2);
  uint32_t* flags = sc.take<uint32_t>(64);
  float* ecost = sc.take<float>(3 * T);
  // alive lists of the global-memory class (ping-pong); the init scratch is free by then
  uint32_t* gl_f[2] = {sc.take<uint32_t>(T), sc.take<uint32_t>(T)};
  uint32_t* gl_v[2] = {sc.take<uint32_t>(U), sc.take<uint32_t>(U)};
  void* tmp = sc.take(tmpb);
  uint32_t* sorted_v = sc.take<uint32_t>(3 * T);
  uint32_t* sorted_h = sc.take<uint32_t>(3 * T);
  IGN_REQUIRE(sc.ok(), IGN_ERR_NOMEM, "scratch arena too small (simplify: %llu faces)", (unsigned long long)T);
  s.tri_off = d_tri_off;

  std::vector<uint32_t> target(K + 2, 0);
  for (uint64_t l = 1; l <= K; l++)
    target[l] = (m->tri_off[l + 1] - m->tri_off[l]) / (uint32_t)reduction_factor;
  // work order of the label kernel: largest labels first (the tail is made of small ones)
  std::vector<uint32_t> order(K);
  for (uint64_t l = 0; l < K; l++) order[l] = (uint32_t)(l + 1);
  std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
    const uint32_t ta = m->tri_off[a + 1] - m->tri_off[a], tb = m->tri_off[b + 1] - m->tri_off[b];
    return ta != tb ? ta > tb : a < b;
  });
  IGN_TRY(small_h2d(ctx, d_target, target.data(), (K + 2) * 4));
  IGN_TRY(small_h2d(ctx, d_tri_off, m->tri_off.data(), (K + 2) * 4));
  IGN_TRY(small_h2d(ctx, d_vert_off, m->vert_off.data(), (K + 2) * 4));
  IGN_TRY(small_h2d(ctx, d_order, order.data(), K * 4));
  IGN_LAUNCH(ctx, k_simp_init_verts, blocks_for(U, 256), 256, 0, m->d_uniq_vkeys, U, (double)resolution[0],
           (double)resolution[1], (double)resolution[2], s.pos, s.valive, s.vbound, s.vn);
  IGN_LAUNCH(ctx, k_simp_init_faces, blocks_for(T, 256), 256, 0, m->d_faces, d_tri_off, d_vert_off, (uint32_t)K, T,
           s.face, s.flabel, s.falive, node_v, node_h);
  {
    int bits = 1;
    while (bits < 32 && (1ull << bits) < U) bits++;
    size_t tb = tmpb;
    IGN_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, node_v, sorted_v, node_h, sorted_h, (int)(3 * T), 0, bits,
                                           ctx->stream));
    ctx->launches += 3;
  }
  IGN_CUDA(cudaMemsetAsync(flags, 0, 64, ctx->stream));
  IGN_LAUNCH(ctx, k_simp_link, blocks_for(3 * T, 256), 256, 0, sorted_v, sorted_h, (uint64_t)(3 * T), s.vf, s.vn,
           flags + 12);
  IGN_LAUNCH(ctx, k_simp_quadrics, blocks_for(U, 128), 128, 0, s);
  IGN_LAUNCH(ctx, k_simp_boundary, blocks_for(3 * T, 256), 256, 0, s);

  // ---- all rounds of every label: persistent CTAs pull labels off the order list.  The kernel is
  // latency bound (barriers, dependent loads), so several CTAs per SM overlap each other's
  // stalls; the shared-memory budget of a label is the SM's divided by the CTAs per SM
  // (IGN_SIMP_THREADS / IGN_SIMP_CTAS override the default for experiments).
  int sl_threads = 1024, sl_ctas = 1;  // measured on B200: 1024x1 76 ms, 512x2 94 ms, 256x4 91 ms per 257^3 task
  if (const char* e = getenv("IGN_SIMP_THREADS")) sl_threads = atoi(e);
  if (const char* e = getenv("IGN_SIMP_CTAS")) sl_ctas = atoi(e);
  if (sl_threads != 256 && sl_threads != 512 && sl_threads != 1024) sl_threads = 1024;
  if (sl_ctas < 1 || sl_ctas * sl_threads > 1024) sl_ctas = 1024 / sl_threads;
  const size_t sl_static = ((sizeof(SlShared) + 255) / 256) * 256 + 1024;
  const size_t sl_dyn = ((232448 / (size_t)sl_ctas) > sl_static + 16384 ? (232448 / (size_t)sl_ctas) - sl_static : 16384) & ~(size_t)255;
  IGN_CUDA(cudaFuncSetAttribute(k_simp_labels, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sl_dyn));
  SlArgs A;
  A.pos = s.pos; A.Q = s.Q; A.face = s.face; A.falive = s.falive; A.valive = s.valive; A.vbound = s.vbound;
  A.ecost = ecost; A.key1 = key1; A.fstate = fstate; A.vflag = vflag; A.vlose = vlose;
  A.flist = gl_f[0]; A.flist2 = gl_f[1]; A.vlist = gl_v[0]; A.vlist2 = gl_v[1];
  A.tri_off = d_tri_off; A.vert_off = d_vert_off; A.target = d_target; A.order = d_order;
  A.K = (uint32_t)K; A.counters = flags;
  A.max_err2 = (double)max_error * (double)max_error;
  A.max_rounds = 400;
  // IGN_SIMP_GMEM=1 (test knob): run every label on the global-memory arrays, the path of
  // labels that do not fit shared memory (only the winners' ring lists stay in smem)
  A.trace = nullptr;
  A.lrec = nullptr;
  if (getenv("IGN_SIMP_TRACE") != nullptr) {
    A.trace = sc.take<uint32_t>(400 * 4 + 64);
    A.lrec = sc.take<uint32_t>((size_t)K * 6 + 16);
    if (!A.lrec) A.trace = nullptr;
    if (A.trace) IGN_CUDA(cudaMemsetAsync(A.trace, 0, 400 * 16 + 256, ctx->stream));
    if (A.trace) IGN_CUDA(cudaMemsetAsync(A.lrec, 0, (size_t)K * 24 + 64, ctx->stream));
  }
  const char* force_gmem = getenv("IGN_SIMP_GMEM");
  const uint32_t sl_fixed = (uint32_t)((SL_THREADS / 32) * SL_EQ * 4 + SL_WCAP * 2 * S_MAXV * 4);  // queues + ring lists
  A.smem_bytes = (force_gmem && force_gmem[0] == '1') ? sl_fixed : (uint32_t)sl_dyn;
  {
    const int slot = prof_begin(ctx, IGN_PROF_SIMP);
    // default: one CTA per label (SMs are handed back to the block scheduler after every label, so
    // higher-priority streams get them quickly); IGN_SIMP_PERSIST=1: one CTA per SM slot loops over labels
    const char* pe = getenv("IGN_SIMP_PERSIST");
    A.persist = (pe && pe[0] == '1') ? 1 : 0;
    const uint64_t slots = (uint64_t)ctx->sm_count * sl_ctas;
    const unsigned grid = A.persist ? (unsigned)(K < slots ? K : slots) : (unsigned)K;
    k_simp_labels<<<grid, sl_threads, sl_dyn, ctx->stream>>>(A);
    ctx->launches++;
    prof_end(ctx, slot);
    IGN_CUDA(cudaGetLastError());
  }

  // ---- compaction
  uint32_t* fscan = node_v;   // 3T u32 >= T
  uint32_t* fflag = node_h;
  size_t tb = tmpb;
  IGN_LAUNCH(ctx, k_simp_flags_u32, blocks_for(U, 256), 256, 0, s.valive, U, vflag32);
  IGN_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, vflag32, vscan, (int)U, ctx->stream));
  IGN_LAUNCH(ctx, k_simp_flags_u32, blocks_for(T, 256), 256, 0, s.falive, T, fflag);
  tb = tmpb;
  IGN_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, fflag, fscan, (int)T, ctx->stream));
  ctx->launches += 4;
  uint32_t last[4], hflags[16];
  IGN_TRY(small_d2h(ctx, &last[0], vscan + (U - 1), 4));
  IGN_TRY(small_d2h(ctx, &last[1], vflag32 + (U - 1), 4));
  IGN_TRY(small_d2h(ctx, &last[2], fscan + (T - 1), 4));
  IGN_TRY(small_d2h(ctx, &last[3], fflag + (T - 1), 4));
  IGN_TRY(small_d2h(ctx, hflags, flags, 64));
  IGN_TRY(small_sync(ctx));
  if (hflags[12] != 0) {
    set_error("simplify: a vertex has more than %d incident faces", S_VCAP);
    return IGN_ERR_UNSUPPORTED;
  }
  if (A.trace) {
    std::vector<uint32_t> tr(1600);
    IGN_CUDA(cudaMemcpy(tr.data(), A.trace, 1600 * 4, cudaMemcpyDeviceToHost));
    unsigned long long phs[10];
    IGN_CUDA(cudaMemcpy(phs, A.trace + 1600, 80, cudaMemcpyDeviceToHost));
    static const char* names[10] = {"P1", "P2 keys", "P3 lose", "P4 select", "setup", "E1 rings", "E2a cost", "E2b flips", "E2c link+collapse", "stop+compact"};
    unsigned long long tot = 0;
    for (int q = 0; q < 10; q++) tot += phs[q];
    for (int q = 0; q < 10; q++)
      fprintf(stderr, "phase %-18s %6.2f %%  %10.3f Mcycles\n", names[q], 100.0 * phs[q] / (tot ? tot : 1), phs[q] / 1e6);
    {
      // per-label records: where do the cycles go -- per round (fixed latency) or per face visit?
      std::vector<uint32_t> rec(6 * (size_t)K);
      IGN_CUDA(cudaMemcpy(rec.data(), A.lrec, rec.size() * 4, cudaMemcpyDeviceToHost));
      static const uint32_t edges[] = {0, 500, 1000, 2000, 4000, 8000, 16000, 32000, 64000, 0xFFFFFFFFu};
      fprintf(stderr, "%12s %7s %8s %10s %10s %9s %9s  class(sm/hy/gl)\n", "faces<", "labels", "rounds", "Mcycles", "Mvisits", "kwins", "cyc/round");
      double sr = 0, sv = 0, sc = 0, srr = 0, svv = 0, srv = 0, src = 0, svc = 0;
      for (int b = 0; b + 1 < 10; b++) {
        uint64_t n = 0, rounds = 0, kc = 0, vis = 0, wins = 0, cls[4] = {0, 0, 0, 0};
        for (uint64_t i = 0; i < K; i++) {
          const uint32_t* q = &rec[6 * i];
          if (q[1] == 0 || q[0] < edges[b] || q[0] >= edges[b + 1]) continue;
          n++; rounds += q[1]; kc += q[2]; vis += q[3]; wins += q[4]; cls[q[5] & 3]++;
          const double R = q[1], V = q[3], C = q[2] * 1024.0;
          sr += R; sv += V; sc += C; srr += R * R; svv += V * V; srv += R * V; src += R * C; svc += V * C;
        }
        if (n) fprintf(stderr, "%12u %7llu %8.1f %10.2f %10.3f %9.1f %9.0f  %llu/%llu/%llu\n", edges[b + 1], (unsigned long long)n, (double)rounds / n,
                       kc * 1024.0 / 1e6, vis / 1e6, wins / 1e3, rounds ? kc * 1024.0 / rounds : 0.0,
                       (unsigned long long)cls[1], (unsigned long long)cls[2], (unsigned long long)cls[3]);
      }
      // least squares cycles = a * rounds + b * visits (no intercept)
      const double det = srr * svv - srv * srv;
      if (det != 0) fprintf(stderr, "fit: cycles ~= %.0f * rounds + %.2f * face visits   (totals: %.0f rounds, %.3g visits, %.3g cycles)\n",
                            (src * svv - svc * srv) / det, (svc * srr - src * srv) / det, sr, sv, sc);
    }
    for (int r = 0; r < 400 && getenv("IGN_SIMP_TRACE_ROUNDS") && (tr[4 * r + 2] || tr[4 * r + 3]); r++)
      fprintf(stderr, "gpu round %d progress %u collapses %u alive %u list %u\n", r, tr[4 * r], tr[4 * r + 1], tr[4 * r + 2], tr[4 * r + 3]);
  }
  m->simp_rounds = (int)hflags[1];
  m->simp_labels_smem = hflags[2];
  m->simp_labels_gmem = hflags[3];
  const uint32_t U2 = last[0] + last[1], T2 = last[2] + last[3];
  IGN_LAUNCH(ctx, k_simp_new_offsets, blocks_for(K + 2, 256), 256, 0, d_vert_off, vscan, (uint32_t)(K + 2), U, U2,
           d_new_vert_off);
  IGN_LAUNCH(ctx, k_simp_new_offsets, blocks_for(K + 2, 256), 256, 0, d_tri_off, fscan, (uint32_t)(K + 2), T, T2,
           d_new_tri_off);
  // results overwrite the mesher's buffers (inputs were copied into the arena; the vertex buffer holds 12 B / vertex)
  float* pos_f = (float*)m->d_uniq_vkeys;
  IGN_LAUNCH(ctx, k_simp_compact_verts, blocks_for(U, 256), 256, 0, s, vscan, pos_f);
  IGN_LAUNCH(ctx, k_simp_compact_faces, blocks_for(T, 256), 256, 0, s, vscan, fscan, d_new_vert_off, m->d_faces);
  IGN_TRY(small_d2h(ctx, m->tri_off.data(), d_new_tri_off, (K + 2) * 4));
  IGN_TRY(small_d2h(ctx, m->vert_off.data(), d_new_vert_off, (K + 2) * 4));
  IGN_TRY(small_sync(ctx));
  m->U = U2;
  m->T = T2;
  m->d_pos_f = pos_f;
  m->simplified = true;
  m->present.clear();
  for (uint64_t l = 1; l <= K; l++)
    if (m->tri_off[l + 1] > m->tri_off[l]) m->present.push_back(m->ids[l - 1]);
  return IGN_OK;
}
